"""Training throughput of ``python -m idelucs_b200`` at --gpus 1, 2 and 8 on seeded synthetic sets (10^5 x 10 kb and
10^6 x 2 kb, 5 clusters of random sequences, CLI defaults otherwise: --n_mimics 3 --batch_sz 256, RMSprop).

Each configuration runs the CLI twice in a fresh process with one voter: with --n_epochs E and with --n_epochs 0.  The second run
does everything the first does except the optimiser steps (FASTA parse, packing, scaler, graph capture, inference, vote, metrics),
so the difference of the two wall times is the training phase of E epochs, and pairs/s = E x n_pairs / that difference.  The card
name and power limit are read in the same call.  Writes profiles/cli_gpus_probe.json (or the path given as the first argument).

    python tools/cli_gpus_probe.py [out.json] [--epochs E] [--gpus 1,2,8] [--sets 100000x10000,1000000x2000]"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def write_fasta(path, n, length, seed=0, chunk=20000):
    """n random ACGT sequences of `length` bases, written in chunks (the 2 GB set never sits in memory twice)"""
    rng = np.random.default_rng(seed)
    alph = np.frombuffer(b"ACGT", dtype=np.uint8)
    with open(path, "wb") as fh:
        for c0 in range(0, n, chunk):
            m = min(chunk, n - c0)
            seqs = alph[rng.integers(0, 4, size=(m, length), dtype=np.uint8)]
            nl = np.full((m, 1), ord("\n"), dtype=np.uint8)
            body = np.concatenate([seqs, nl], axis=1)
            for i in range(m):
                fh.write(b">s%d\n" % (c0 + i))
                fh.write(body[i].tobytes())


def cli_wall(fasta, gpus, epochs, workdir):
    cmd = [sys.executable, "-m", "idelucs_b200", "--sequence_file", fasta, "--n_clusters", "5", "--n_voters", "1", "--n_epochs", str(epochs)]
    if gpus > 1:
        cmd += ["--gpus", str(gpus)]
    env = dict(os.environ, PYTHONPATH=ROOT + os.pathsep + os.environ.get("PYTHONPATH", ""))
    t0 = time.time()
    res = subprocess.run(cmd, cwd=workdir, env=env, capture_output=True, text=True)
    wall = time.time() - t0
    if res.returncode != 0:
        raise RuntimeError("%s failed:\n%s" % (" ".join(cmd), res.stderr[-3000:]))
    return wall


def card():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout
    return [line.strip() for line in out.strip().splitlines()]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("out", nargs="?", default=os.path.join(ROOT, "profiles", "cli_gpus_probe.json"))
    ap.add_argument("--epochs", type=int, default=1)
    ap.add_argument("--gpus", default="1,2,8")
    ap.add_argument("--sets", default="100000x10000,1000000x2000")
    a = ap.parse_args()
    import torch
    visible = torch.cuda.device_count()
    if visible == 0:
        raise SystemExit("no CUDA device: nothing to measure")
    result = {"cards": card(), "epochs": a.epochs, "n_mimics": 3, "batch_sz": 256, "optimizer": "RMSprop", "runs": []}
    with tempfile.TemporaryDirectory() as tmp:
        for spec in a.sets.split(","):
            n, length = (int(x) for x in spec.split("x"))
            fasta = os.path.join(tmp, "synthetic_%dx%d.fas" % (n, length))
            write_fasta(fasta, n, length)
            n_pairs = 3 * n
            for g in (int(x) for x in a.gpus.split(",")):
                if g > visible:
                    result["runs"].append({"set": spec, "gpus": g, "skipped": "only %d GPUs visible" % visible})
                    continue
                full = cli_wall(fasta, g, a.epochs, tmp)
                base = cli_wall(fasta, g, 0, tmp)
                train = full - base
                row = {"set": spec, "gpus": g, "wall_s": round(full, 2), "wall_without_training_s": round(base, 2), "training_s": round(train, 2),
                       "steps_per_epoch": -(-n_pairs // 256), "pairs_per_s": round(a.epochs * n_pairs / train, 1)}
                print(json.dumps(row), flush=True)
                result["runs"].append(row)
            os.remove(fasta)
    result["cards_after"] = card()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as fh:
        json.dump(result, fh, indent=1)
    print(json.dumps(result))


if __name__ == "__main__":
    main()
