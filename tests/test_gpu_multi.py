"""Two-rank NCCL test of the sharded path (needs >= 2 GPUs; skipped otherwise): scaler
statistics merged over ranks == single-GPU statistics, sharded mimics identical to the
unsharded ones (global sequence ids in the RNG), data-parallel training step (eager and CUDA-graphed, flat-gradient
all-reduce), all-gathered predictions.  Every training step's optimiser update is checked bit for bit: this rank's slice of the new
parameters and its RMSprop state == idl_rmsprop_step on the rank-order sum of every rank's gradient (symmetric memory: peer loads
or NVLS multimem; with two ranks the sum has one rounding, so its order cannot matter) or on the NCCL-averaged gradient."""
import os
import sys

import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _checked_step(tr, world):
    """one training step; returns (loss, whether the optimiser's update of this rank's slice equals the reference update)"""
    import torch.distributed as dist
    from idelucs_b200 import _lib
    lib = _lib.load()
    P0, sq0 = tr._flat_param.clone(), tr._sq.clone()
    loss = float(tr.step().item())
    torch.cuda.synchronize()
    if tr._mode == "symm":   # the kernel reads every rank's gradient and leaves it untouched
        gs = [torch.empty_like(P0) for _ in range(world)]
        dist.all_gather(gs, tr._flat_grad.clone())
        total = torch.zeros_like(P0)
        for g in gs:
            total += g
        lo, hi = tr.rank * tr._shard, (tr.rank + 1) * tr._shard
        P, g, scale = P0[lo:hi].clone(), total[lo:hi].clone(), float(np.float32(1) / np.float32(world))
    else:                    # NCCL: the flat gradient was averaged in place
        lo, hi = 0, P0.numel()
        P, g, scale = P0.clone(), tr._flat_grad.clone(), 1.0
    sq = sq0.clone()
    _lib.check(lib.idl_rmsprop_step(_lib.ptr(P), _lib.ptr(g), _lib.ptr(sq), hi - lo, tr.lr, tr.alpha, tr.eps, tr.weight_decay, scale,
                                    _lib.stream_ptr()))
    return loss, torch.equal(tr._flat_param[lo:hi], P) and torch.equal(tr._sq, sq)


def _worker(rank, world, port, ret):
    sys.path.insert(0, ROOT)
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world), LOCAL_RANK=str(rank))
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world)
    from idelucs_b200 import featurise as ft
    from idelucs_b200 import parallel
    from idelucs_b200.seqset import SeqSet
    from idelucs_b200.train import ShardedTrainer
    from idelucs_b200.utils import augment_device
    dev = torch.device("cuda", rank)
    rng = np.random.default_rng(0)
    n, k = 600, 5
    lengths = rng.integers(300, 3000, size=n)
    alph = np.frombuffer(b"ACGT", dtype=np.uint8)
    seqs = [alph[rng.integers(0, 4, size=int(L))].tobytes() for L in lengths]
    ranges = parallel.shard_ranges(lengths, world)
    lo, hi = ranges[rank]
    ss = SeqSet.from_sequences(seqs[lo:hi], device=dev)
    prof, sc, _ = augment_device(ss, 6, k=k, seed=42, group=dist.group.WORLD, seq_id0=lo)
    ok = True
    if rank == 0:  # the unsharded computation on one GPU
        full = SeqSet.from_sequences(seqs, device=dev)
        pf, scf, _ = augment_device(full, 6, k=k, seed=42)
        ok = ok and torch.allclose(sc.mean64, scf.mean64, rtol=1e-13, atol=0) and torch.allclose(sc.scale64, scf.scale64, rtol=1e-10)
        ok = ok and torch.allclose(prof, pf[:, lo:hi], rtol=1e-5, atol=1e-5)
        ok = ok and bool((prof == pf[:, lo:hi]).float().mean() > 0.99)
    tr = ShardedTrainer(ss, k=k, n_clusters=4, n_mimics=6, batch_sz=64, seed=3, seq_id0=lo, world=world)
    graphed = tr.enable_cuda_graph()                            # step + flat-gradient all-reduce in one CUDA graph
    steps = [_checked_step(tr, world) for _ in range(4)]
    ok = ok and all(np.isfinite(l) for l, _ in steps)
    opt_ok = [o for _, o in steps]
    w = next(tr.net.parameters()).detach().clone()
    ws = [torch.empty_like(w) for _ in range(world)]
    dist.all_gather(ws, w)
    ok = ok and all(torch.equal(ws[0], x) for x in ws)          # replicas stay identical (averaged gradients)
    if rank == 0:
        ret["graph"] = bool(graphed)
        ret["graph_error"] = getattr(tr, "_graph_error", "")
        ret["path"] = tr._mode + ("/multimem" if tr._mode == "symm" and tr._mc[0] else "/peer loads" if tr._mode == "symm" else "")
    tr._graph = None                                            # the same step eagerly
    steps = [_checked_step(tr, world) for _ in range(3)]
    ok = ok and all(np.isfinite(l) for l, _ in steps)
    opt_ok += [o for _, o in steps]
    w = next(tr.net.parameters()).detach().clone()
    dist.all_gather(ws, w)
    ok = ok and all(torch.equal(ws[0], x) for x in ws)
    preds, probs, lat = tr.predict(ss, k=k)      # inference tail: all three row blocks all-gathered in rank order
    ok = ok and preds.shape[0] == n and probs.shape[0] == n and tuple(lat.shape) == (n, 64)
    if rank == 0:   # ... and equal to scoring the unsharded set with the same (replicated) network
        x = ft.Scaler.fit(ft.profiles(full, k, [ft.VariantSpec(ft.KIND_CLEAN)], out_kind=ft.OUT_FREQ_F64)[0])
        f64 = ft.profiles(full, k, [ft.VariantSpec(ft.KIND_CLEAN)], out_kind=ft.OUT_FREQ_F64)[0]
        xs = x.transform64(f64, want32=True)
        tr.net.eval()
        with torch.no_grad():
            out, lat_full = tr.net(xs)
        tr.net.train()
        ok = ok and torch.allclose(lat_full, lat, rtol=1e-4, atol=1e-4) and bool((out.argmax(1) == preds).float().mean() > 0.99)
    # the same checks on the NCCL path (all-reduce + idl_rmsprop_step), graphed and eager
    trn = ShardedTrainer(ss, k=k, n_clusters=4, n_mimics=6, batch_sz=64, seed=3, seq_id0=lo, world=world, use_symmetric_memory=False)
    graphed_nccl = trn.enable_cuda_graph()
    opt_nccl = [_checked_step(trn, world)[1] for _ in range(2)]
    trn._graph = None
    opt_nccl += [_checked_step(trn, world)[1] for _ in range(2)]
    t = torch.tensor([1.0 if ok else 0.0, 1.0 if all(opt_ok) else 0.0, 1.0 if all(opt_nccl) and graphed_nccl and trn._mode == "nccl" else 0.0],
                     device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MIN)
    if rank == 0:
        ret["ok"] = bool(t[0].item() == 1.0)
        ret["optimizer"] = (opt_ok, bool(t[1].item() == 1.0))
        ret["optimizer_nccl"] = (opt_nccl, bool(t[2].item() == 1.0))
    dist.destroy_process_group()


@pytest.mark.timeout(240)
def test_two_gpu_sharding():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import torch.multiprocessing as mp
    mgr = mp.Manager()
    ret = mgr.dict()
    mp.spawn(_worker, args=(2, 29700 + os.getpid() % 200, ret), nprocs=2, join=True)
    print("optimiser path:", ret["path"])
    assert ret["ok"]
    assert ret["graph"], ret["graph_error"]
    assert ret["optimizer"][1], (ret["path"], ret["optimizer"][0])       # per step on rank 0: eager after the four graphed ones
    assert ret["optimizer_nccl"][1], ret["optimizer_nccl"][0]
