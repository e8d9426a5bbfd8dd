"""SGD and Adam on the training step and the CLI's --gpus path (-m gpu):

  1. idl_sgd_step / idl_adam_step against torch.optim.SGD(momentum=0.9, weight_decay=0.01) / torch.optim.Adam over 12 steps from
     the same state (the first step and later ones);
  2. idl_{rmsprop,sgd,adam}_allreduce_step with W pseudo-ranks on one GPU (the kernel only dereferences the addresses it is given)
     == the single-rank kernel on the rank-order gradient sum scaled by 1 / W, bit for bit;
  3. ShardedTrainer(optimizer=...) at world 1, graphed: every step's update == the single-rank kernel on the gradient the step
     wrote; reinit keeps the optimiser state and the graph, and draws the weights again; the epoch loss accumulated on the device;
  4. two GPUs (skipped with fewer): SGD and Adam updates over symmetric memory bit for bit, and ``main([..., "--gpus", "2"])`` end
     to end with --n_clusters 5 and 0;
  5. two GPUs: the clustering accuracy of the data-parallel training against the live reference's distribution, with the
     protocol of test_gpu_e2e_stats.py."""
import ctypes
import glob
import json
import os
import sys

import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

LR, MOMENTUM, WD, BETAS, EPS = 1e-3, 0.9, 0.01, (0.9, 0.999), 1e-8


def _single_step(lib, opt, p, g, state, n, step, gscale, wd):
    """the single-rank kernel of `opt` on flat buffers (state: list of its state tensors)"""
    from idelucs_b200 import _lib
    st = [_lib.ptr(s) for s in state]
    if opt == "RMSprop":
        return lib.idl_rmsprop_step(_lib.ptr(p), _lib.ptr(g), *st, n, LR, 0.99, EPS, wd, gscale, _lib.stream_ptr())
    if opt == "SGD":
        return lib.idl_sgd_step(_lib.ptr(p), _lib.ptr(g), *st, n, LR, MOMENTUM, wd, _lib.ptr(step), gscale, _lib.stream_ptr())
    return lib.idl_adam_step(_lib.ptr(p), _lib.ptr(g), *st, n, LR, *BETAS, EPS, wd, _lib.ptr(step), gscale, _lib.stream_ptr())


# ---------------------------------------------------------------------------------------------------------------------------------
# 1. against torch.optim
# ---------------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("opt,wd,gscale", [("SGD", WD, 1.0), ("SGD", WD, 0.5), ("Adam", 0.0, 1.0), ("Adam", WD, 0.25)])
def test_single_rank_steps_match_torch_optim(opt, wd, gscale):
    from idelucs_b200 import _lib
    lib = _lib.load()
    gen = torch.Generator(device="cuda").manual_seed(5)
    n = 100003   # (not a multiple of 4: the kernels are elementwise)
    p0 = torch.randn(n, device="cuda", generator=gen)
    p_ref = p0.clone().requires_grad_(True)
    ref = (torch.optim.SGD([p_ref], lr=LR, momentum=MOMENTUM, weight_decay=wd) if opt == "SGD"
           else torch.optim.Adam([p_ref], lr=LR, betas=BETAS, eps=EPS, weight_decay=wd))
    p = p0.clone()
    state = [torch.zeros(n, device="cuda") for _ in range(1 if opt == "SGD" else 2)]
    step = torch.zeros((), dtype=torch.int64, device="cuda")
    for t in range(12):
        g = torch.randn(n, device="cuda", generator=gen) * 10.0 ** (t % 3 - 1)
        p_ref.grad = g * gscale
        ref.step()
        step.add_(1)
        _lib.check(_single_step(lib, opt, p, g, state, n, step, gscale, wd))
        torch.cuda.synchronize()
        want = p_ref.detach()
        # norm-wise relative error (max |error| / max |p|): a parameter that momentum carries across zero has no useful
        # element-wise relative error, since a last-bit difference in the buffer becomes a large share of a tiny value
        err = float((p - want).abs().max())
        assert err <= 2e-6 * float(want.abs().max()), (opt, t, err)
        ts = ref.state[p_ref]
        wants = [ts["momentum_buffer"]] if opt == "SGD" else [ts["exp_avg"], ts["exp_avg_sq"]]
        for s, w in zip(state, wants):   # (relative to the largest entry: momentum + gradient cancels near zero)
            assert float((s - w).abs().max()) <= 2e-6 * float(w.abs().max()), (opt, t, float((s - w).abs().max()))


# ---------------------------------------------------------------------------------------------------------------------------------
# 2. the all-reduce steps, W pseudo-ranks on one GPU
# ---------------------------------------------------------------------------------------------------------------------------------
def _allreduce(lib, opt, gp, pp, state, n_total, r, W, step):
    from idelucs_b200 import _lib
    st = [_lib.ptr(s) for s in state]
    if opt == "RMSprop":
        return lib.idl_rmsprop_allreduce_step(gp, pp, 0, 0, *st, n_total, r, W, LR, 0.99, EPS, WD, _lib.stream_ptr())
    if opt == "SGD":
        return lib.idl_sgd_allreduce_step(gp, pp, 0, 0, *st, n_total, r, W, LR, MOMENTUM, WD, _lib.ptr(step), _lib.stream_ptr())
    return lib.idl_adam_allreduce_step(gp, pp, 0, 0, *st, n_total, r, W, LR, *BETAS, EPS, WD, _lib.ptr(step), _lib.stream_ptr())


@pytest.mark.parametrize("opt", ["RMSprop", "SGD", "Adam"])
@pytest.mark.parametrize("W", [2, 3, 8])
def test_allreduce_pseudo_ranks_equal_single_rank_step(opt, W):
    from idelucs_b200 import _lib
    lib = _lib.load()
    gen = torch.Generator(device="cuda").manual_seed(W)
    n_states = 2 if opt == "Adam" else 1
    for n_total in (4 * W, W * (606208 + 4 * 1001)):   # smallest allowed; a shard whose grid-stride loop iterates
        shard = n_total // W
        p0 = torch.randn(n_total, device="cuda", generator=gen)
        params = [p0.clone() for _ in range(W)]
        grads = [torch.zeros(n_total, device="cuda") for _ in range(W)]
        states = [[torch.zeros(shard, device="cuda") for _ in range(n_states)] for _ in range(W)]
        p_ref, st_ref = p0.clone(), [torch.zeros(n_total, device="cuda") for _ in range(n_states)]
        gp = (ctypes.c_uint64 * W)(*[g.data_ptr() for g in grads])
        pp = (ctypes.c_uint64 * W)(*[p.data_ptr() for p in params])
        step = torch.zeros((), dtype=torch.int64, device="cuda")
        for t in range(3):   # the state and the step number carry over
            total = torch.zeros(n_total, device="cuda")
            for r in range(W):
                grads[r].copy_(torch.randn(n_total, device="cuda", generator=gen) * 10.0 ** (t - 1))
                total += grads[r]                                   # float32, rank order, from zero: the kernel's sum
            step.add_(1)
            for r in range(W):
                _lib.check(_allreduce(lib, opt, gp, pp, states[r], n_total, r, W, step))
            _lib.check(_single_step(lib, opt, p_ref, total, st_ref, n_total, step, float(np.float32(1) / np.float32(W)), WD))
            torch.cuda.synchronize()
            case = (opt, W, n_total, t)
            for r in range(W):
                assert torch.equal(params[r], p_ref), (case, r, int((params[r] != p_ref).sum()))
                for s, sr in zip(states[r], st_ref):
                    assert torch.equal(s, sr[r * shard:(r + 1) * shard]), (case, r)


# ---------------------------------------------------------------------------------------------------------------------------------
# 3. ShardedTrainer(optimizer=...) at world 1
# ---------------------------------------------------------------------------------------------------------------------------------
def _random_seqset(n, seed):
    from idelucs_b200.seqset import SeqSet
    rng = np.random.default_rng(seed)
    alph = np.frombuffer(b"ACGT", dtype=np.uint8)
    return SeqSet.from_sequences([alph[rng.integers(0, 4, size=int(L))].tobytes() for L in rng.integers(500, 3000, size=n)])


def _checked_replay(tr, lib):
    """one graph replay; True when the new parameters and state == the single-rank kernel on the state before it and the
    gradient the replay wrote"""
    P0, S0 = tr._flat_param.clone(), [s.clone() for s in tr._state]
    tr.step()
    torch.cuda.synchronize()
    P, S = P0.clone(), [s.clone() for s in S0]
    from idelucs_b200 import _lib
    _lib.check(_single_step(lib, tr.optimizer, P, tr._flat_grad, S, P.numel(), tr._step_no, 1.0, tr.weight_decay))
    torch.cuda.synchronize()
    return torch.equal(tr._flat_param, P) and all(torch.equal(a, b) for a, b in zip(tr._state, S))


@pytest.mark.parametrize("opt", ["RMSprop", "SGD", "Adam"])
def test_sharded_trainer_optimizers_and_reinit(opt):
    from idelucs_b200 import _lib
    from idelucs_b200.train import ShardedTrainer
    lib = _lib.load()
    tr = ShardedTrainer(_random_seqset(300, 3), k=5, n_clusters=5, n_mimics=3, batch_sz=128, seed=3, optimizer=opt)
    assert tr.weight_decay == (0.0 if opt == "Adam" else 0.01)
    assert tr.enable_cuda_graph(), getattr(tr, "_graph_error", "")
    tr.reset_optimizer()
    assert int(tr._step_no.item()) == 0 and all(float(s.abs().sum()) == 0 for s in tr._state)
    assert all(_checked_replay(tr, lib) for _ in range(4))   # the first step (SGD: buffer = gradient; Adam: t = 1) and later ones
    # reinit: fresh Kaiming-normal weights and zero biases, the optimiser state and the step counter untouched
    state, t = [s.clone() for s in tr._state], int(tr._step_no.item())
    tr.reinit(11)
    P1 = tr._flat_param.clone()
    assert all(torch.equal(a, b) for a, b in zip(tr._state, state)) and int(tr._step_no.item()) == t
    for m in tr.net.modules():
        if isinstance(m, torch.nn.Linear):
            assert float(m.bias.abs().max()) == 0.0
            assert abs(float(m.weight.std()) / (2.0 / m.weight.shape[1]) ** 0.5 - 1.0) < 0.1
    losses = []
    for _ in range(5):   # the captured graph still replays, on the new weights
        assert _checked_replay(tr, lib)
        losses.append(float(tr._loss.item()))
    assert int(tr._step_no.item()) == t + 5
    tr.epoch_loss(1)   # (restart the accumulator: it also holds the steps before reinit)
    for _ in range(6):
        tr.step()
        losses.append(float(tr._loss.item()))
    assert abs(tr.epoch_loss(6) - sum(losses[-6:]) / 5) <= 1e-5 * abs(sum(losses[-6:]) / 5)   # contrastive_training_epoch's division
    tr.reinit(11)
    assert torch.equal(tr._flat_param, P1)   # the same seed draws the same weights


# ---------------------------------------------------------------------------------------------------------------------------------
# 4. two GPUs: symmetric-memory SGD / Adam updates, and the CLI
# ---------------------------------------------------------------------------------------------------------------------------------
def _checked_step_multi(tr, world):
    """one data-parallel step; True when this rank's slice of the new parameters and its state == the single-rank kernel on the
    rank-order sum of every rank's gradient (symmetric memory) or on the NCCL-averaged gradient"""
    import torch.distributed as dist
    from idelucs_b200 import _lib
    lib = _lib.load()
    P0, S0 = tr._flat_param.clone(), [s.clone() for s in tr._state]
    tr.step()
    torch.cuda.synchronize()
    if tr._mode == "symm":
        gs = [torch.empty_like(P0) for _ in range(world)]
        dist.all_gather(gs, tr._flat_grad.clone())
        total = torch.zeros_like(P0)
        for g in gs:
            total += g
        lo, hi = tr.rank * tr._shard, (tr.rank + 1) * tr._shard
        P, g, scale = P0[lo:hi].clone(), total[lo:hi].clone(), float(np.float32(1) / np.float32(world))
    else:
        lo, hi = 0, P0.numel()
        P, g, scale = P0.clone(), tr._flat_grad.clone(), 1.0
    S = [s.clone() for s in S0]
    _lib.check(_single_step(lib, tr.optimizer, P, g, S, hi - lo, tr._step_no, scale, tr.weight_decay))
    torch.cuda.synchronize()
    return torch.equal(tr._flat_param[lo:hi], P) and all(torch.equal(a, b) for a, b in zip(tr._state, S))


def _init(rank, world, port):
    sys.path.insert(0, ROOT)
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world)


def _optim_worker(rank, world, port, ret):
    import torch.distributed as dist
    _init(rank, world, port)
    from idelucs_b200 import parallel
    from idelucs_b200.seqset import SeqSet
    from idelucs_b200.train import ShardedTrainer
    rng = np.random.default_rng(0)
    lengths = rng.integers(300, 3000, size=600)
    alph = np.frombuffer(b"ACGT", dtype=np.uint8)
    seqs = [alph[rng.integers(0, 4, size=int(L))].tobytes() for L in lengths]
    lo, hi = parallel.shard_ranges(lengths, world)[rank]
    ss = SeqSet.from_sequences(seqs[lo:hi], device=torch.device("cuda", rank))
    res = {}
    for opt in ("SGD", "Adam"):
        for symm in (True, False):
            tr = ShardedTrainer(ss, k=5, n_clusters=4, n_mimics=6, batch_sz=64, seed=3, seq_id0=lo, world=world, optimizer=opt,
                                use_symmetric_memory=symm)
            graphed = tr.enable_cuda_graph()
            tr.reset_optimizer()
            ok = [_checked_step_multi(tr, world) for _ in range(3)]
            tr.reinit(5)
            ok += [_checked_step_multi(tr, world) for _ in range(2)]
            ws = [torch.empty_like(tr._flat_param) for _ in range(world)]
            dist.all_gather(ws, tr._flat_param.clone())
            t = torch.tensor([1.0 if all(ok) and graphed and all(torch.equal(ws[0], w) for w in ws) else 0.0], device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MIN)
            res["%s/%s" % (opt, tr._mode)] = (bool(t.item() == 1.0), ok)
            del tr
    if rank == 0:
        ret.update(res)
    dist.destroy_process_group()


def _two_gpus():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")


@pytest.mark.timeout(300)
def test_two_gpu_sgd_adam_updates_bit_exact():
    _two_gpus()
    import torch.multiprocessing as mp
    ret = mp.Manager().dict()
    mp.spawn(_optim_worker, args=(2, 29500 + os.getpid() % 200, ret), nprocs=2, join=True)
    res = dict(ret)
    assert set(res) == {"SGD/symm", "SGD/nccl", "Adam/symm", "Adam/nccl"}, res
    for k, (ok, steps) in res.items():
        assert ok, (k, steps)


@pytest.mark.timeout(900)
@pytest.mark.parametrize("n_clusters", [5, 0])
def test_cli_two_gpus(fasta_files, golden_dir, tmp_path, monkeypatch, n_clusters):
    _two_gpus()
    import multiprocessing
    from idelucs_b200 import __main__ as cli
    monkeypatch.chdir(tmp_path)
    fasta = fasta_files["Influenza-A"]
    cli.main(["--sequence_file", fasta, "--GT_file", os.path.join(golden_dir, "Influenza-A_GT.tsv"), "--n_clusters", str(n_clusters),
              "--n_epochs", "3", "--n_voters", "2", "--batch_sz", "512", "--gpus", "2", "--optimizer", "Adam"])
    assert multiprocessing.active_children() == []
    n = sum(1 for line in open(fasta) if line.startswith(">"))
    found = {f: glob.glob(os.path.join(str(tmp_path), "Results", "*", "*", f)) for f in ("assignments.tsv", "metrics.tsv")}
    assert all(len(v) == 1 for v in found.values()), found
    rows = open(found["assignments.tsv"][0]).read().splitlines()
    assert rows[0] == "sequence_id\tassignment\tconfidence_score" and len(rows) == n + 1
    head, vals = open(found["metrics.tsv"][0]).read().splitlines()
    assert "ACC" in head.split("\t") and len(vals.split("\t")) == len(head.split("\t"))


# ---------------------------------------------------------------------------------------------------------------------------------
# 5. two GPUs: statistical parity with the live reference
# ---------------------------------------------------------------------------------------------------------------------------------
N_SEEDS, N_EPOCHS = 20, 35


def _stats_worker(rank, world, port, fastas, golden_dir, ret):
    import torch.distributed as dist
    _init(rank, world, port)
    from sklearn.metrics import adjusted_rand_score
    from idelucs_b200 import featurise as ft
    from idelucs_b200 import parallel
    from idelucs_b200.seqset import SeqSet, read_fasta_native
    from idelucs_b200.train import ShardedTrainer
    from idelucs_b200.utils import SummaryFasta, cluster_acc
    with open(os.path.join(golden_dir, "e2e_reference.json")) as fh:
        ref = json.load(fh)["datasets"]
    out = {}
    for stem, fasta in fastas.items():
        C, GB = ref[stem]["n_clusters"], ref[stem]["batch_sz"]
        _, _, byte_off = read_fasta_native(fasta, pinned=False)
        n = byte_off.size - 1
        lo, hi = parallel.shard_ranges(np.diff(byte_off), world)[rank]
        ss = SeqSet.from_fasta(fasta, device=torch.device("cuda", rank), rows=(lo, hi))
        steps = -(-(len(ft.mimic_schedule(3)) - 1) * n // GB)
        if rank == 0:
            _, _, GT, _ = SummaryFasta(fasta, os.path.join(golden_dir, stem + "_GT.tsv"))
            labels = {c: i for i, c in enumerate(sorted(set(GT)))}
            y_true = np.array([labels[c] for c in GT])
        accs, aris = [], []
        for s in range(N_SEEDS):   # what the CLI's rank loop does for one voter
            tr = ShardedTrainer(ss, k=6, n_clusters=C, n_mimics=3, batch_sz=GB // world, lamb=2.8, weight=0.25, lr=1e-3, seed=1000 + s,
                                seq_id0=lo, world=world)
            tr.enable_cuda_graph()
            tr.reset_optimizer()
            tr.reinit(1000 + s)
            for _ in range(N_EPOCHS):
                for _ in range(steps):
                    tr.step()
                tr.epoch_loss(steps)
            y_pred, _, _ = tr.predict(ss, k=6)
            if rank == 0:
                y_pred = y_pred.cpu().numpy()
                accs.append(cluster_acc(y_true, y_pred)[1])
                aris.append(adjusted_rand_score(y_true, y_pred))
            del tr
        out[stem] = (accs, aris)
    if rank == 0:
        ret.update(out)
    dist.destroy_process_group()


@pytest.mark.timeout(1800)
def test_two_gpu_accuracy_distribution_matches_reference(fasta_files, golden_dir):
    _two_gpus()
    import torch.multiprocessing as mp
    from scipy.stats import mannwhitneyu
    ret = mp.Manager().dict()
    mp.spawn(_stats_worker, args=(2, 29900 + os.getpid() % 80, dict(fasta_files), golden_dir, ret), nprocs=2, join=True)
    with open(os.path.join(golden_dir, "e2e_reference.json")) as fh:
        ref = json.load(fh)["datasets"]
    fails = []
    for stem in ("Influenza-A", "Actinopterygii"):
        accs, aris = (np.array(x) for x in ret[stem])
        r_acc, r_ari = np.array(ref[stem]["acc"]), np.array(ref[stem]["ari"])
        p_acc = mannwhitneyu(accs, r_acc, alternative="two-sided").pvalue
        p_ari = mannwhitneyu(aris, r_ari, alternative="two-sided").pvalue
        hi, r_hi = float((accs > 0.97).mean()), float((r_acc > 0.97).mean())
        print("\n%s, 2 GPUs: ACC %.3f +- %.3f (reference %.3f +- %.3f), share > 0.97: %.2f (reference %.2f), Mann-Whitney p: ACC %.3f ARI %.3f"
              % (stem, accs.mean(), accs.std(), r_acc.mean(), r_acc.std(), hi, r_hi, p_acc, p_ari))
        print("sorted ACC:", np.round(np.sort(accs), 3).tolist())
        if not (p_acc > 0.05 and p_ari > 0.05 and abs(hi - r_hi) <= 0.3 and abs(accs.mean() - r_acc.mean()) < 0.06):
            fails.append((stem, p_acc, p_ari, hi, r_hi, float(accs.mean()), float(r_acc.mean())))
    assert not fails, fails
