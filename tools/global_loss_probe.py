"""Cost of ShardedTrainer(global_batch_loss=True): graph-replayed step time with and without the global-batch loss, timed with CUDA
events, at 2 and 8 GPUs (those the machine has), b = 32 / 64 / 512 pairs per rank (32 = the CLI default batch 256 at 8 GPUs),
C = 5 and 200; then one torch.profiler run per world size (b = 32, C = 5) that splits the kernel time the global loss adds into
barriers, pulls (the kernels that read peer memory) and GEMMs.  Writes JSON (default profiles/global_loss_probe.json) with the card
name and power limit read in the same run.

    python tools/global_loss_probe.py [--out PATH] [--steps 200]"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
PULLS = ("nce_gather_rows", "nce_normalize_backward_global", "iid_global_small", "iid_s2_sum", "iid_s2_kernel", "nce_rows_kernel")


def _kind(name):
    n = name.lower()
    if "barrier" in n:
        return "barrier"
    if any(p in name for p in PULLS):
        return "pull"
    if "gemm" in n or "sgemm" in n or "cutlass" in n or "xmma" in n:
        return "gemm"
    return "other"


def _worker(rank, world, port, steps, ret):
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world)
    from idelucs_b200.seqset import SeqSet
    from idelucs_b200.train import ShardedTrainer
    rng = np.random.default_rng(rank)
    alph = np.frombuffer(b"ACGT", dtype=np.uint8)
    ss = SeqSet.from_sequences([alph[rng.integers(0, 4, size=2000)].tobytes() for _ in range(3000)], device=torch.device("cuda", rank))
    rows = []
    for b in (32, 64, 512):
        for C in (5, 200):
            row = dict(world=world, pairs_per_rank=b, C=C)
            for g in (False, True):
                tr = ShardedTrainer(ss, k=6, n_clusters=C, n_mimics=3, batch_sz=b, seed=1, seq_id0=rank * 3000, world=world, global_batch_loss=g)
                assert tr.enable_cuda_graph(), getattr(tr, "_graph_error", "")
                for _ in range(20):
                    tr.step()
                torch.cuda.synchronize()
                dist.barrier()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(steps):
                    tr.step()
                e1.record()
                torch.cuda.synchronize()
                t = torch.tensor([e0.elapsed_time(e1) / steps], device="cuda")
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
                row["global_ms" if g else "per_rank_ms"] = round(float(t), 4)
                row["mode"] = tr._mode
                if g and b == 32 and C == 5:
                    from torch.profiler import ProfilerActivity, profile
                    split = {}
                    for gg, trp in ((False, None), (True, tr)):
                        if trp is None:
                            trp = ShardedTrainer(ss, k=6, n_clusters=C, n_mimics=3, batch_sz=b, seed=1, seq_id0=rank * 3000, world=world)
                            trp.enable_cuda_graph()
                        torch.cuda.synchronize()
                        with profile(activities=[ProfilerActivity.CUDA]) as prof:
                            for _ in range(50):
                                trp.step()
                            torch.cuda.synchronize()
                        tot = {}
                        for ev in prof.key_averages():
                            k = _kind(ev.key)
                            tot[k] = tot.get(k, 0.0) + ev.device_time_total / 50.0
                        split["global" if gg else "per_rank"] = {k: round(v, 2) for k, v in tot.items()}
                    row["kernel_us_per_step"] = split
                del tr
            rows.append(row)
    if rank == 0:
        ret.extend(rows)
    dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "global_loss_probe.json"))
    ap.add_argument("--steps", type=int, default=200)
    a = ap.parse_args()
    import torch.multiprocessing as mp
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    n = torch.cuda.device_count()
    out = dict(gpu=gpu.splitlines()[0] if gpu else None, devices=n, steps=a.steps, rows=[],
               note="per_rank_ms / global_ms: one graph-replayed ShardedTrainer step (k = 6, RMSprop), max over the ranks of the "
                    "CUDA-event mean; kernel_us_per_step: torch.profiler device time per step by kind")
    for world in (2, 8):
        if world > n:
            out.setdefault("not_measured", []).append("world %d: %d devices visible" % (world, n))
            continue
        ret = mp.Manager().list()
        mp.spawn(_worker, args=(world, 29600 + world, a.steps, ret), nprocs=world, join=True)
        out["rows"] += list(ret)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as fh:
        json.dump(out, fh, indent=1)
    print(json.dumps(out, indent=1))


if __name__ == "__main__":
    main()
