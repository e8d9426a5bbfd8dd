"""Time and peak device memory of the canonical (model_size 'small') featurisation: the canonical output kinds of the
profile kernel against the composition they replace, which this script keeps as its own reference.

Per shape (seeded random ACGT sequences of one length, k = 6):
  - augment_device(reduce=True) (t_norm rows -> scaler -> every slot standardised in one call) and the old composition
    (+1 counts [V, N, 4096] -> revcomp_fold -> normalize_counts -> Scaler.fit -> transform32): the median wall time of
    calls that end in a device synchronise, torch.cuda.max_memory_allocated over each call, and whether both give the same
    bits (the old one may not fit the card: then its out-of-memory error is recorded);
  - one regenerated B = 512 batch of PairBatchLoader: reduce=True (canonical rows) against reduce=False (4096 columns),
    CUDA events around batches of random pair ids, median over the repetitions.
The card's name and power limit are read in the same run.

    python tools/canonical_probe.py --shapes 100000x10000x50,1000000x2000x3 --out profiles/canonical_probe.json
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def card():
    import torch
    out = {"name": torch.cuda.get_device_name(0)}
    try:
        out["nvidia_smi"] = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                                           capture_output=True, text=True, timeout=60).stdout.strip().splitlines()[0]
    except (OSError, IndexError, subprocess.SubprocessError) as e:
        out["nvidia_smi"] = "unavailable: %s" % e
    return out


def random_seqset(n, L, seed):
    import torch
    from idelucs_b200.seqset import SeqSet
    g = torch.Generator(device="cuda").manual_seed(seed)
    a = torch.randint(0, 4, (n * L,), dtype=torch.uint8, device="cuda", generator=g)
    ascii_u8 = 65 + 2 * a + 2 * (a == 2).to(torch.uint8) + 13 * (a == 3).to(torch.uint8)   # 0 1 2 3 -> A C G T
    del a
    ss = SeqSet.from_ascii(ascii_u8, np.arange(n + 1, dtype=np.int64) * L, validate=False)
    ss._d_ascii = None   # the packed codes are all the kernels read
    return ss


def old_composition(ss, n_mimics, k, seed):
    """augment_device(reduce=True) as it was: full-width int32 counts, then the fold, the division and the scaler"""
    from idelucs_b200 import featurise as ft
    variants = ft.mimic_schedule(n_mimics)
    c = ft.profiles(ss, k, variants, out_kind=ft.OUT_COUNTS_I32, seed=seed, pseudocount=1)
    x32 = ft.normalize_counts(ft.revcomp_fold(c, k), want64=False, want32=True)
    del c
    sc = ft.Scaler.fit(x32[0], group=None)
    V, n, R = x32.shape
    return sc.transform32(x32.reshape(V * n, R)).reshape(V, n, R)


def new_path(ss, n_mimics, k, seed):
    from idelucs_b200 import utils as U
    return U.augment_device(ss, n_mimics, k=k, seed=seed, reduce=True)[0]


def measure(fn, reps):
    """(median seconds, peak bytes over one call, result of the last call) or an out-of-memory record"""
    import torch
    times, peak, out = [], 0, None
    for _ in range(reps):
        out = None
        torch.cuda.empty_cache()
        torch.cuda.synchronize()
        base = torch.cuda.memory_allocated()
        torch.cuda.reset_peak_memory_stats()
        t0 = time.perf_counter()
        try:
            out = fn()
            torch.cuda.synchronize()
        except torch.cuda.OutOfMemoryError as e:
            torch.cuda.empty_cache()
            return {"out_of_memory": str(e).splitlines()[0]}, None
        times.append(time.perf_counter() - t0)
        peak = max(peak, torch.cuda.max_memory_allocated() - base)
    return {"median_s": statistics.median(times), "times_s": times, "peak_bytes": peak, "peak_GB": peak / 1e9}, out


def batch_time(ss, n_mimics, k, reduce, reps, iters, seed):
    import torch
    from idelucs_b200 import utils as U
    loader = U.PairBatchLoader(ss, n_mimics, k=k, seed=seed, reduce=reduce, materialize_bytes=0)
    rng = np.random.default_rng(5)
    ids = [torch.from_numpy(rng.integers(0, loader.n_pairs, size=512)).cuda() for _ in range(iters)]
    for i in ids[:10]:
        loader.batch(i)
    res = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        for i in ids:
            loader.batch(i)
        e1.record()
        torch.cuda.synchronize()
        res.append(e0.elapsed_time(e1) * 1e3 / iters)
    return {"median_us": statistics.median(res), "per_rep_us": res, "columns": int(loader.batch(ids[0])["true"].shape[1])}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--shapes", default="100000x10000x50,1000000x2000x3", help="N x length x n_mimics, comma separated")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--batch-iters", type=int, default=200)
    ap.add_argument("--out", default="profiles/canonical_probe.json")
    a = ap.parse_args()
    import torch
    rep = {"card": card(), "k": 6, "shapes": []}
    for shape in a.shapes.split(","):
        n, L, n_mimics = (int(v) for v in shape.split("x"))
        ss = random_seqset(n, L, seed=n + L)
        seed = 1234
        rec = {"n": n, "length": L, "n_mimics": n_mimics, "V": max(n_mimics, 2) + 1}
        rec["new_augment_device"], new = measure(lambda: new_path(ss, n_mimics, 6, seed), a.reps)
        if new is not None:
            rec["new_out_bytes"] = new.numel() * 4
        del new
        rec["old_composition"], old = measure(lambda: old_composition(ss, n_mimics, 6, seed), a.reps)
        if old is not None:
            chk = new_path(ss, n_mimics, 6, seed)
            rec["old_equals_new"] = bool(torch.equal(chk, old))
            del chk
        del old
        torch.cuda.empty_cache()
        rec["batch_reduce_true"] = batch_time(ss, n_mimics, 6, True, a.reps, a.batch_iters, seed)
        rec["batch_reduce_false"] = batch_time(ss, n_mimics, 6, False, a.reps, a.batch_iters, seed)
        rep["shapes"].append(rec)
        print(json.dumps(rec), flush=True)
        del ss
        torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as fh:
        json.dump(rep, fh, indent=1)
    print(json.dumps(rep["card"]))


if __name__ == "__main__":
    main()
