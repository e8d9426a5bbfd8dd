"""Timing of the silhouette pass (idl_silhouette_samples) against sklearn.metrics.silhouette_score.

Input: seeded 64-d blobs, float32, with K clusters of equal size (K = 2, 200 and N / 4; the last puts a cluster boundary
every 4 columns, so it shows what the per-row finalisation costs).  Per run it reports the host part of the call (labels to
the host, stable counting sort, order and offsets back: the time until the call returns), the kernel time (CUDA events
around a call that ends in a stream synchronise, less the host part), fp64 operations 3 D N^2 over the kernel time, and,
where --sklearn-max allows, sklearn's silhouette_score on this machine's host with the largest difference from the device
values.  The card's name and power limit are read in the same run.

    python tools/metrics_probe.py --sizes 16000,100000,1000000 --sklearn-max 16000 --out profiles/metrics_probe.json
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


def blobs(n, k, d=64, seed=0):
    """k clusters of n // k or n // k + 1 points around seeded centres, labels in random order"""
    rng = np.random.default_rng(seed)
    c = rng.normal(0.0, 10.0, size=(k, d))
    lab = rng.permutation(np.arange(n) % k)
    return (c[lab] + rng.normal(0.0, 1.0, size=(n, d))).astype(np.float32), lab


def card():
    import torch
    out = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=60).stdout.strip().splitlines()[0]
        out["nvidia_smi"] = q
    except (OSError, IndexError, subprocess.SubprocessError) as e:
        out["nvidia_smi"] = "unavailable: %s" % e
    return out


def device_run(x, lab, reps):
    """(median host part s, median call s on the device, samples)"""
    import torch
    from idelucs_b200 import _lib
    lib = _lib.load()
    n, D = x.shape
    k = int(lab.max()) + 1
    xd = torch.from_numpy(x).cuda()
    ld = torch.from_numpy(lab.astype(np.int32)).cuda()
    ws = torch.empty(lib.idl_silhouette_workspace_bytes(n, k), dtype=torch.uint8, device="cuda")
    out = torch.empty(n, dtype=torch.float64, device="cuda")
    host, call = [], []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        t0 = time.perf_counter()
        _lib.check(lib.idl_silhouette_samples(_lib.ptr(xd), _lib.ptr(ld), n, D, k, _lib.ptr(out), _lib.ptr(ws), ws.numel(), _lib.stream_ptr()))
        host.append(time.perf_counter() - t0)
        e1.record()
        torch.cuda.synchronize()
        call.append(e0.elapsed_time(e1) / 1e3)
    return statistics.median(host), statistics.median(call), out.cpu().numpy()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", default="16000,100000,1000000")
    ap.add_argument("--sklearn-max", type=int, default=16000, help="run sklearn for N up to this")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    from sklearn.metrics import silhouette_samples, silhouette_score
    device_run(*blobs(2000, 20, seed=1), reps=2)   # module load, first launches
    res = {"card": card(), "input": "64-d blobs, K equal clusters around seeded centres (seed = N + K), float32; D = 64",
           "kernel_s": "median of the device time of the call (CUDA events, ends in a synchronise) less the host part",
           "runs": []}
    for n in [int(s) for s in a.sizes.split(",")]:
        for k in (2, 200, n // 4):
            x, lab = blobs(n, k, seed=n + k)
            reps = 5 if n <= 100000 else 1
            host, call, samples = device_run(x, lab, reps)
            kern = call - host
            r = dict(n=n, clusters=k, reps=reps, host_grouping_s=host, call_s=call, kernel_s=kern,
                     fp64_ops=3 * 64 * n * n, fp64_tops=3 * 64 * n * n / kern / 1e12, device_score=float(np.mean(samples)))
            if n <= a.sklearn_max:
                x64 = x.astype(np.float64)
                t0 = time.perf_counter()
                sk = silhouette_score(x64, lab)
                r["sklearn_s"] = time.perf_counter() - t0
                r["sklearn_score"] = float(sk)
                r["score_abs_diff"] = abs(r["device_score"] - float(sk))
                r["samples_max_abs_diff"] = float(np.max(np.abs(samples - silhouette_samples(x64, lab))))
            res["runs"].append(r)
            print(json.dumps(r), flush=True)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            json.dump(res, fh, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
