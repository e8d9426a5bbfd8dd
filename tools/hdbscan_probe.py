"""Timing of the --n_clusters 0 clustering step (hdbscan_device) against sklearn.cluster.HDBSCAN.

Input: seeded 64-d blobs around 200 centres, float32, min_cluster_size = min_samples = N // 100 + 1 (the CLI's parameters).
Per N it reports the device time of idl_core_distances and of idl_mreach_mst (CUDA events around a call that ends in a
stream synchronise), the host tail (sort, single-linkage tree, labels), sklearn's fit time where --sklearn-max allows, and
whether labels and probabilities are equal.  The card's name and power limit are read in the same run.

    python tools/hdbscan_probe.py --sizes 4000,16000,100000,1000000 --sklearn-max 16000 --out profiles/hdbscan_probe.json
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def blobs(n, d=64, centers=200, seed=0):
    rng = np.random.default_rng(seed)
    c = rng.normal(0.0, 10.0, size=(centers, d))
    return (c[rng.integers(0, centers, size=n)] + rng.normal(0.0, 1.0, size=(n, d))).astype(np.float32)


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


def device_run(x):
    import torch
    from idelucs_b200.hdbscan import _workspace, core_distances, labels_from_mst, mreach_mst
    n = x.shape[0]
    m = n // 100 + 1
    xd = torch.from_numpy(x).cuda()
    ws = _workspace(xd)
    e = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
    torch.cuda.synchronize()
    e[0].record()
    core = core_distances(xd, m, ws)
    e[1].record()
    src, dst, w = mreach_mst(xd, core, ws)
    e[2].record()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    labels, probs = labels_from_mst(src.cpu().numpy(), dst.cpu().numpy(), w.cpu().numpy(), m)
    tail = time.perf_counter() - t0
    w = w.cpu().numpy()
    return dict(core_s=e[0].elapsed_time(e[1]) / 1e3, mst_s=e[1].elapsed_time(e[2]) / 1e3, host_tail_s=tail,
                tied_mst_weights=int(len(w) - len(np.unique(w)))), labels, probs


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", default="4000,16000,100000,1000000")
    ap.add_argument("--sklearn-max", type=int, default=16000, help="run sklearn for N up to this")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    from sklearn.cluster import HDBSCAN
    device_run(blobs(2000, seed=1))   # module load, first launches
    res = {"card": card(), "input": "64-d blobs, 200 centres, seed = N, min_cluster_size = min_samples = N // 100 + 1", "runs": []}
    for n in [int(s) for s in a.sizes.split(",")]:
        x = blobs(n, seed=n)
        r, labels, probs = device_run(x)
        r = dict(n=n, min_cluster_size=n // 100 + 1, device_total_s=r["core_s"] + r["mst_s"] + r["host_tail_s"], **r)
        if n <= a.sklearn_max:
            t0 = time.perf_counter()
            sk = HDBSCAN(min_cluster_size=n // 100 + 1, copy=True).fit(x.astype(np.float64))
            r["sklearn_s"] = time.perf_counter() - t0
            r["labels_equal"] = bool(np.array_equal(labels, sk.labels_))
            r["probabilities_equal"] = bool(np.array_equal(probs, sk.probabilities_))
        r["n_clusters"] = int(labels.max()) + 1
        res["runs"].append(r)
        print(json.dumps(r), flush=True)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            json.dump(res, fh, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
