"""The global-batch loss of the data-parallel step (LossFunctions.GlobalBatchLoss, ShardedTrainer(global_batch_loss=True)):

  1. W pseudo-ranks on one GPU (the kernels only dereference the peer addresses they are given): every rank's loss is the same bits,
     and the ranks' dz, dh (over W) and the loss equal a float64 restatement of (1 - w) InfoNCE + w IIC on the global batch and
     the one-GPU train_losses_and_grads on the stacked global batch;
  2. at world 1 the flag changes nothing, bit for bit;
  3. two GPUs (skipped with fewer), symmetric memory and NCCL, eager and replayed from the CUDA graph: every step's gradient is
     that of the float64 global-batch step rebuilt from each rank's batch and dropout masks, the update is the optimiser's on it,
     both modes give the same bits, the replicas stay identical and epoch_loss is the same on both ranks;
  4. two GPUs: ``main([..., "--gpus", "2", "--global_batch_loss"])`` end to end with --n_clusters 5 and 0;
  5. two GPUs: clustering accuracy with the global loss against the live reference's distribution."""
import glob
import json
import os
import sys

import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LAMB, WEIGHT, TEMP, D = 2.8, 0.25, 0.85, 64


def _inputs(B, C, seed):
    """global stacked z [2B, C] (softmax rows) and h [2B, D] (the modified view correlated with the true one)"""
    g = torch.Generator(device="cuda").manual_seed(seed)
    z = torch.softmax(torch.randn(2 * B, C, device="cuda", generator=g) * 2.0, 1)
    a = torch.randn(B, D, device="cuda", generator=g)
    h = torch.cat((a, 0.3 * a + torch.randn(B, D, device="cuda", generator=g)), 0)
    return z.contiguous(), h.contiguous()


def _rows(r, b, B):
    """global rows of rank r's stacked local batch"""
    return torch.cat((torch.arange(r * b, (r + 1) * b), torch.arange(B + r * b, B + (r + 1) * b))).cuda()


def _want64(z, h):
    """(loss, dz, dh) of the global batch in float64 (the reference's formulations)"""
    from test_gpu_parity import _ref_iid64, _ref_style_info_nce
    B = z.shape[0] // 2
    zd = z.double().requires_grad_(True)
    hd = h.double().requires_grad_(True)
    loss = (1 - WEIGHT) * _ref_style_info_nce(hd[:B], hd[B:], TEMP) + WEIGHT * _ref_iid64(zd[:B], zd[B:], LAMB)
    gz, gh = torch.autograd.grad(loss, (zd, hd))
    return float(loss.detach()), gz, gh


def _pseudo_ranks(z, h, W, b, C):
    """GlobalBatchLoss of W pseudo-ranks on one GPU, stage by stage: [(loss, dz, dh)] in rank order"""
    from idelucs_b200.LossFunctions import GlobalBatchLoss
    B = W * b
    ranks = [GlobalBatchLoss(r, W, b, C, D, z.device, LAMB, WEIGHT, TEMP) for r in range(W)]
    for gl in ranks:
        gl.set_peers([g.send1.data_ptr() for g in ranks], [g.send2.data_ptr() for g in ranks])
    for r, gl in enumerate(ranks):
        idx = _rows(r, b, B)
        gl.stage1(z[idx], h[idx])
    for gl in ranks:
        gl.stage2()
    out = [gl.stage3() for gl in ranks]
    torch.cuda.synchronize()
    return out


def _close(got, want, tag):
    err = float((got.double() - want).abs().max())
    assert err <= 1e-4 * float(want.abs().max()), (tag, err, float(want.abs().max()))


@pytest.mark.parametrize("C", [3, 5, 8, 16, 17, 200])
@pytest.mark.parametrize("W", [2, 3, 8])
def test_pseudo_ranks_equal_global_batch(W, C):
    from idelucs_b200.LossFunctions import train_losses_and_grads
    for b in (37, 64):
        B = W * b
        z, h = _inputs(B, C, 100 * W + C + b)
        out = _pseudo_ranks(z, h, W, b, C)
        tag = (W, C, b)
        losses = [o[0] for o in out]
        assert all(torch.equal(losses[0], l) for l in losses), (tag, [float(l) for l in losses])
        dz = torch.empty_like(z)
        dh = torch.empty_like(h)
        for r, (_, dzr, dhr) in enumerate(out):
            idx = _rows(r, b, B)
            dz[idx] = dzr / W
            dh[idx] = dhr / W
        lw, gz, gh = _want64(z, h)
        assert abs(float(losses[0]) - lw) < 1e-5, (tag, float(losses[0]), lw)
        _close(dz, gz, tag + ("dz",))
        _close(dh, gh, tag + ("dh",))
        l1, dz1, dh1 = train_losses_and_grads(z, h, LAMB, WEIGHT, TEMP)   # one GPU on the stacked global batch
        assert abs(float(l1) - float(losses[0])) < 1e-5, tag
        _close(dz, dz1.double(), tag + ("dz one GPU",))
        _close(dh, dh1.double(), tag + ("dh one GPU",))


def _random_seqset(n, seed):
    from idelucs_b200.seqset import SeqSet
    rng = np.random.default_rng(seed)
    alph = np.frombuffer(b"ACGT", dtype=np.uint8)
    return SeqSet.from_sequences([alph[rng.integers(0, 4, size=int(L))].tobytes() for L in rng.integers(500, 3000, size=n)])


def test_world_one_flag_changes_nothing():
    from idelucs_b200.train import ShardedTrainer
    ss = _random_seqset(300, 4)
    trs = [ShardedTrainer(ss, k=5, n_clusters=5, n_mimics=3, batch_sz=96, seed=4, global_batch_loss=g) for g in (False, True)]
    assert trs[1]._gloss is None
    losses = [[], []]
    for i, tr in enumerate(trs):
        for _ in range(3):
            losses[i].append(tr.step().clone())
        assert tr.enable_cuda_graph(), getattr(tr, "_graph_error", "")
        for _ in range(3):
            losses[i].append(tr.step().clone())
    torch.cuda.synchronize()
    assert all(torch.equal(a, b) for a, b in zip(*losses))
    assert torch.equal(trs[0]._flat_param, trs[1]._flat_param) and torch.equal(trs[0]._sq, trs[1]._sq)


# ---------------------------------------------------------------------------------------------------------------------------------
# 3. two GPUs
# ---------------------------------------------------------------------------------------------------------------------------------
def _init(rank, world, port):
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world)


def _views(tr, flat):
    out, o = [], 0
    for p in tr.net.parameters():
        out.append(flat[o:o + p.numel()].view_as(p))
        o += p.numel()
    return out


def _gather(t, world):
    import torch.distributed as dist
    ts = [torch.empty_like(t) for _ in range(world)]
    dist.all_gather(ts, t.contiguous())
    return ts


def _check_global_step(tr, world, P0, S0, x, rec1, rec2, loss):
    """one global-loss step: the loss and the mean of the ranks' gradients against the float64 global-batch step (each rank's
    batch and its ReLU - Dropout factors 2 [out > 0]), and the update against the single-rank RMSprop kernel on the rank-order
    gradient sum (NCCL: on the averaged gradient the step left in the flat buffer).  Returns (failures, mean of the ranks' gradients)."""
    from idelucs_b200 import _lib
    from test_gpu_parity import _ref_iid64, _ref_style_info_nce
    fails = []
    xs, r1s, r2s = _gather(x, world), _gather(rec1, world), _gather(rec2, world)
    grads = _gather(tr._flat_grad.clone(), world)
    W1, b1, W2, b2, W3, b3 = params = [v.detach().double().requires_grad_(True) for v in _views(tr, P0)]
    b = x.shape[0] // 2
    zs, hs = [], []
    for xr, q1, q2 in zip(xs, r1s, r2s):
        d1 = (xr.double() @ W1.t() + b1) * (2.0 * (q1 > 0).double())
        h = d1 @ W2.t() + b2
        z = torch.softmax((h * (2.0 * (q2 > 0).double())) @ W3.t() + b3, 1)
        zs.append(z); hs.append(h)
    zg = torch.cat([z[:b] for z in zs] + [z[b:] for z in zs])
    hg = torch.cat([h[:b] for h in hs] + [h[b:] for h in hs])
    B = world * b
    want = (1 - tr.weight) * _ref_style_info_nce(hg[:B], hg[B:], 0.85) + tr.weight * _ref_iid64(zg[:B], zg[B:], tr.lamb)
    gwant = torch.autograd.grad(want, params)
    if abs(float(loss) - float(want)) >= 1e-5:
        fails.append(("loss", float(loss), float(want)))
    mean = sum(g.double() for g in grads) / world
    for g, gw in zip(_views(tr, mean), gwant):
        if float((g - gw).abs().max()) > 1e-4 * float(gw.abs().max()):
            fails.append(("grad", tuple(gw.shape), float((g - gw).abs().max()), float(gw.abs().max())))
    total = torch.zeros_like(grads[0])
    for g in grads:
        total += g
    lib = _lib.load()
    if tr._mode == "symm":
        lo, hi = tr.rank * tr._shard, (tr.rank + 1) * tr._shard
        P, g, scale = P0[lo:hi].clone(), total[lo:hi].clone(), float(np.float32(1) / np.float32(world))
    else:
        lo, hi = 0, P0.numel()
        P, g, scale = P0.clone(), tr._flat_grad.clone(), 1.0
    S = S0.clone()
    _lib.check(lib.idl_rmsprop_step(_lib.ptr(P), _lib.ptr(g), _lib.ptr(S), hi - lo, tr.lr, tr.alpha, tr.eps, tr.weight_decay, scale, _lib.stream_ptr()))
    torch.cuda.synchronize()
    if not (torch.equal(tr._flat_param[lo:hi], P) and torch.equal(tr._sq, S)):
        fails.append(("update", int((tr._flat_param[lo:hi] != P).sum())))
    return fails, total / world


def _train_worker(rank, world, port, ret):
    import torch.distributed as dist
    _init(rank, world, port)
    from idelucs_b200 import parallel, train
    from idelucs_b200.seqset import SeqSet
    rng = np.random.default_rng(0)
    lengths = rng.integers(300, 3000, size=600)
    alph = np.frombuffer(b"ACGT", dtype=np.uint8)
    seqs = [alph[rng.integers(0, 4, size=int(L))].tobytes() for L in lengths]
    lo, hi = parallel.shard_ranges(lengths, world)[rank]
    ss = SeqSet.from_sequences(seqs[lo:hi], device=torch.device("cuda", rank))
    recs = []
    fwd = train._relu_dropout_fwd

    def recording_fwd(*a):
        out = fwd(*a)
        recs.append(out.clone())   # (under capture the clone is part of the graph: every replay refreshes it)
        return out
    train._relu_dropout_fwd = recording_fwd
    res, firsts = {}, {}
    for symm in (True, False):
        tr = train.ShardedTrainer(ss, k=5, n_clusters=5, n_mimics=6, batch_sz=48, seed=3, seq_id0=lo, world=world, use_symmetric_memory=symm,
                                  global_batch_loss=True)
        fails = []
        tr._batch = tr._featurise(tr._next_ids()).clone()
        for i in range(6):
            graphed = i >= 3
            if i == 3:
                if not tr.enable_cuda_graph():
                    fails.append(("graph", getattr(tr, "_graph_error", "")))
                    break
                cap = recs[-2], recs[-1]
            P0, S0, x = tr._flat_param.clone(), tr._sq.clone(), tr._batch.clone()
            loss = tr.step()
            torch.cuda.synchronize()
            r1, r2 = cap if graphed else (recs[-2], recs[-1])
            f, mean = _check_global_step(tr, world, P0, S0, x, r1, r2, float(loss))
            fails += [(i, e) for e in f]
            if i == 0:   # (same start, same batches and masks: the two exchanges must give the same bits)
                firsts[tr._mode] = (float(loss), mean)
            ls = _gather(loss.reshape(1).clone(), world)
            if not torch.equal(ls[0], ls[1]):
                fails.append((i, "loss differs between the ranks"))
        ws = _gather(tr._flat_param.clone(), world)
        if not all(torch.equal(ws[0], w) for w in ws):
            fails.append("replicas differ")
        el = _gather(torch.tensor([tr.epoch_loss(6)], device="cuda"), world)
        if not torch.equal(el[0], el[1]):
            fails.append("epoch_loss differs")
        res[tr._mode] = fails
        del tr
    same = len(firsts) == 2 and firsts["symm"][0] == firsts["nccl"][0] and torch.equal(firsts["symm"][1], firsts["nccl"][1])
    if rank == 0:
        ret.update(res)
        ret["modes_agree"] = same
    dist.destroy_process_group()


def _two_gpus():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")


@pytest.mark.timeout(600)
def test_two_gpu_global_steps_equal_float64_reference():
    _two_gpus()
    import torch.multiprocessing as mp
    ret = mp.Manager().dict()
    mp.spawn(_train_worker, args=(2, 29700 + os.getpid() % 100, ret), nprocs=2, join=True)
    res = dict(ret)
    assert set(res) == {"symm", "nccl", "modes_agree"}, res
    assert res["symm"] == [] and res["nccl"] == [], res
    assert res["modes_agree"]


@pytest.mark.timeout(900)
@pytest.mark.parametrize("n_clusters", [5, 0])
def test_cli_two_gpus_global_batch_loss(fasta_files, golden_dir, tmp_path, monkeypatch, n_clusters):
    _two_gpus()
    import multiprocessing
    from idelucs_b200 import __main__ as cli
    monkeypatch.chdir(tmp_path)
    fasta = fasta_files["Influenza-A"]
    cli.main(["--sequence_file", fasta, "--GT_file", os.path.join(golden_dir, "Influenza-A_GT.tsv"), "--n_clusters", str(n_clusters),
              "--n_epochs", "3", "--n_voters", "2", "--batch_sz", "512", "--gpus", "2", "--global_batch_loss"])
    assert multiprocessing.active_children() == []
    n = sum(1 for line in open(fasta) if line.startswith(">"))
    found = {f: glob.glob(os.path.join(str(tmp_path), "Results", "*", "*", f)) for f in ("assignments.tsv", "metrics.tsv")}
    assert all(len(v) == 1 for v in found.values()), found
    rows = open(found["assignments.tsv"][0]).read().splitlines()
    assert rows[0] == "sequence_id\tassignment\tconfidence_score" and len(rows) == n + 1
    head, vals = open(found["metrics.tsv"][0]).read().splitlines()
    assert "ACC" in head.split("\t") and len(vals.split("\t")) == len(head.split("\t"))


# ---------------------------------------------------------------------------------------------------------------------------------
# 5. two GPUs: statistical parity with the live reference (the protocol of test_gpu_cli_gpus.py's accuracy test)
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
        for s in range(N_SEEDS):
            tr = ShardedTrainer(ss, k=6, n_clusters=C, n_mimics=3, batch_sz=GB // world, lamb=2.8, weight=0.25, lr=1e-3, seed=1000 + s,
                                seq_id0=lo, world=world, global_batch_loss=True)
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
def test_two_gpu_global_loss_accuracy_matches_reference(fasta_files, golden_dir):
    _two_gpus()
    import torch.multiprocessing as mp
    from scipy.stats import mannwhitneyu
    ret = mp.Manager().dict()
    mp.spawn(_stats_worker, args=(2, 29800 + os.getpid() % 80, dict(fasta_files), golden_dir, ret), nprocs=2, join=True)
    with open(os.path.join(golden_dir, "e2e_reference.json")) as fh:
        ref = json.load(fh)["datasets"]
    fails = []
    for stem in ("Influenza-A", "Actinopterygii"):
        accs, aris = (np.array(x) for x in ret[stem])
        r_acc, r_ari = np.array(ref[stem]["acc"]), np.array(ref[stem]["ari"])
        p_acc = mannwhitneyu(accs, r_acc, alternative="two-sided").pvalue
        p_ari = mannwhitneyu(aris, r_ari, alternative="two-sided").pvalue
        hi, r_hi = float((accs > 0.97).mean()), float((r_acc > 0.97).mean())
        print("\n%s, 2 GPUs, global loss: ACC %.3f +- %.3f (reference %.3f +- %.3f), share > 0.97: %.2f (reference %.2f), Mann-Whitney p: "
              "ACC %.3f ARI %.3f" % (stem, accs.mean(), accs.std(), r_acc.mean(), r_acc.std(), hi, r_hi, p_acc, p_ari))
        if not (p_acc > 0.05 and p_ari > 0.05 and abs(hi - r_hi) <= 0.3 and abs(accs.mean() - r_acc.mean()) < 0.06):
            fails.append((stem, p_acc, p_ari, hi, r_hi, float(accs.mean()), float(r_acc.mean())))
    assert not fails, fails
