"""Timing of the HDBSCAN and silhouette all-pairs passes split over several devices (``devices=[...]``).

Input: seeded 64-d blobs around 200 centres, float32, min_cluster_size = min_samples = N // 100 + 1 (the CLI's parameters);
the silhouette is taken of the blob labels (200 clusters), as tools/metrics_probe.py does.  Per (N, device list) it reports
the core distances, the MST, the host tail (sort, single-linkage tree, labels) and the silhouette separately, each timed on
the host clock around work that ends in a synchronise of every device used, and whether every output equals the one-device
output bit for bit.

  - N = --n-small at 1, 2, 4 and 8 distinct devices (as many as the box has) and N = --n-large at the largest count;
  - on a box with one GPU: the cost of splitting, devices=[0] * 8 against [0] at N = --n-small, alternated --reps times;
    multi-GPU speed-ups are then "not measured";
  - with --baseline-tree (a checkout of another commit, its library built): the one-device path (devices=None) of both
    trees at N = 16 000 and --n-small, in child processes alternated --reps times, with a digest of the outputs of each.

The name and power limit of every card are read in the same run.

    python tools/allpairs_devices_probe.py --baseline-tree ../parent --out profiles/allpairs_devices_probe.json
"""
import argparse
import hashlib
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

HERE = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def blobs(n, d=64, centers=200, seed=0):
    """(x float32 [n, d], the centre of every row)"""
    rng = np.random.default_rng(seed)
    c = rng.normal(0.0, 10.0, size=(centers, d))
    lab = rng.integers(0, centers, size=n)
    return (c[lab] + rng.normal(0.0, 1.0, size=(n, d))).astype(np.float32), lab


def cards():
    import torch
    out = {"names": [torch.cuda.get_device_name(i) for i in range(torch.cuda.device_count())]}
    try:
        out["nvidia_smi"] = subprocess.run(["nvidia-smi", "--query-gpu=index,name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                                           capture_output=True, text=True, timeout=60).stdout.strip().splitlines()
    except (OSError, subprocess.SubprocessError) as e:
        out["nvidia_smi"] = "unavailable: %s" % e
    return out


def sync_all():
    import torch
    for i in range(torch.cuda.device_count()):
        torch.cuda.synchronize(i)


def split_run(x, lab, devices):
    """one --n_clusters 0 tail on the given device list (None: one device, the unsplit call) -> (phase seconds, outputs)"""
    import torch
    from idelucs_b200.hdbscan import _core_parts, _mst_parts, _parts, _replicas, _workspace, labels_from_mst
    from idelucs_b200.metrics import silhouette_samples_device
    n = x.shape[0]
    m = n // 100 + 1
    sync_all()
    t0 = time.perf_counter()
    parts = _parts(x, devices)
    xs = _replicas(x, parts)
    wss = [_workspace(xs[d]) for d, _, _ in parts]
    cores = _core_parts(xs, parts, m, wss)
    sync_all()
    t1 = time.perf_counter()
    src, dst, w = _mst_parts(xs, cores, parts, wss)
    sync_all()
    t2 = time.perf_counter()
    src, dst, w = src.cpu().numpy(), dst.cpu().numpy(), w.cpu().numpy()
    labels, probs = labels_from_mst(src, dst, w, m)
    t3 = time.perf_counter()
    sil = silhouette_samples_device(x, lab, devices=devices)
    sync_all()
    t4 = time.perf_counter()
    out = dict(core=cores[x.device].cpu().numpy(), src=src, dst=dst, w=w, labels=labels, probs=probs, sil=sil)
    del xs, wss, cores
    torch.cuda.empty_cache()
    return dict(core_s=t1 - t0, mst_s=t2 - t1, host_tail_s=t3 - t2, silhouette_s=t4 - t3, total_s=t4 - t0), out


def same(a, b):
    return all(np.array_equal(a[k], b[k]) for k in a)


def digest(out):
    h = hashlib.sha256()
    for k in sorted(out):
        h.update(np.ascontiguousarray(out[k]).tobytes())
    return h.hexdigest()[:16]


def child(tree, sizes):
    """the one-device path of the package in `tree` (the calls every version of it has): per N the median of 3 timed runs"""
    sys.path.insert(0, tree)
    import torch
    from idelucs_b200.hdbscan import _workspace, core_distances, labels_from_mst, mreach_mst
    from idelucs_b200.metrics import silhouette_samples_device
    res = {}
    for n in [2000] + sizes:   # the first size loads the module and warms up
        xh, lab = blobs(n, seed=n)
        x = torch.from_numpy(xh).cuda()
        m = n // 100 + 1
        t = {"core_s": [], "mst_s": [], "silhouette_s": []}
        for _ in range(3):
            ws = _workspace(x)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            core = core_distances(x, m, ws)
            torch.cuda.synchronize()
            t1 = time.perf_counter()
            src, dst, w = mreach_mst(x, core, ws)
            torch.cuda.synchronize()
            t2 = time.perf_counter()
            labels, probs = labels_from_mst(src.cpu().numpy(), dst.cpu().numpy(), w.cpu().numpy(), m)
            torch.cuda.synchronize()
            t3 = time.perf_counter()
            sil = silhouette_samples_device(x, lab)
            torch.cuda.synchronize()
            t4 = time.perf_counter()
            t["core_s"].append(t1 - t0)
            t["mst_s"].append(t2 - t1)
            t["silhouette_s"].append(t4 - t3)
        out = dict(core=core.cpu().numpy(), src=src.cpu().numpy(), dst=dst.cpu().numpy(), w=w.cpu().numpy(), labels=labels, probs=probs, sil=sil)
        res[n] = dict({k: statistics.median(v) for k, v in t.items()}, digest=digest(out))
    print(json.dumps(res))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n-small", type=int, default=100000)
    ap.add_argument("--n-large", type=int, default=1000000)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--baseline-tree", default=None, help="checkout of the commit to compare the one-device path with (library built)")
    ap.add_argument("--child", default=None, help=argparse.SUPPRESS)
    ap.add_argument("--child-sizes", default="16000,100000", help=argparse.SUPPRESS)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if a.child:
        return child(a.child, [int(s) for s in a.child_sizes.split(",")])
    sys.path.insert(0, HERE)
    import torch
    n_gpus = torch.cuda.device_count()
    res = {"cards": cards(), "gpus": n_gpus,
           "input": "64-d blobs, 200 centres, seed = N, float32; min_cluster_size = min_samples = N // 100 + 1; silhouette of the blob labels",
           "timing": "host clock around each phase, every device synchronised at its end; one run per row after a warm-up",
           "split": [], "regression": None}
    xh, lab = blobs(4000, seed=1)
    split_run(torch.from_numpy(xh).cuda(), lab, list(range(n_gpus)))   # module load, first launches on every device
    counts = [c for c in (1, 2, 4, 8) if c <= n_gpus]
    for n, cs in ((a.n_small, counts), (a.n_large, counts[-1:])):
        xh, lab = blobs(n, seed=n)
        x = torch.from_numpy(xh).cuda()
        ref = None
        for c in cs:
            t, out = split_run(x, lab, list(range(c)))
            ref = ref or out
            r = dict(n=n, devices=list(range(c)), equal_to_one_device=same(out, ref) if c > 1 else None, **t)
            res["split"].append(r)
            print(json.dumps(r), flush=True)
    if n_gpus == 1:
        res["multi_gpu_speedup"] = "not measured: the box has one GPU"
        xh, lab = blobs(a.n_small, seed=a.n_small)
        x = torch.from_numpy(xh).cuda()
        rows = {"[0]": [], "[0]*8": []}
        outs = {}
        for _ in range(a.reps):
            for key, devs in (("[0]", [0]), ("[0]*8", [0] * 8)):
                t, outs[key] = split_run(x, lab, devs)
                rows[key].append(t)
        res["split_cost"] = dict(n=a.n_small, reps=a.reps, equal=same(outs["[0]*8"], outs["[0]"]),
                                 **{key: {k: statistics.median(t[k] for t in v) for k in v[0]} for key, v in rows.items()},
                                 runs=rows)
        print(json.dumps(res["split_cost"]), flush=True)
    if a.baseline_tree:
        runs = {"baseline": [], "this": []}
        for _ in range(a.reps):
            for key, tree in (("baseline", os.path.abspath(a.baseline_tree)), ("this", HERE)):
                p = subprocess.run([sys.executable, os.path.abspath(__file__), "--child", tree, "--child-sizes", "16000,%d" % a.n_small],
                                   capture_output=True, text=True, timeout=1800)
                if p.returncode != 0:
                    raise RuntimeError(p.stderr)
                runs[key].append(json.loads(p.stdout.strip().splitlines()[-1]))
        summary = {}
        for n in runs["this"][0]:
            summary[n] = {key: {k: [r[n][k] for r in v] for k in ("core_s", "mst_s", "silhouette_s")} for key, v in runs.items()}
            summary[n]["same_outputs"] = len({r[n]["digest"] for v in runs.values() for r in v}) == 1
        res["regression"] = dict(note="one-device path (devices=None), this tree against --baseline-tree, child processes alternated; "
                                      "per child the median of 3 runs", per_n=summary)
        print(json.dumps(res["regression"]), flush=True)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            json.dump(res, fh, indent=1)


if __name__ == "__main__":
    main()
