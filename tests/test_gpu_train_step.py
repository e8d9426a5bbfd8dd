"""The training step of train.ShardedTrainer against independent references:

  * the fused ReLU - Dropout kernels and idl_sum_parts_bias against a numpy float32 restatement, bit for bit, with the keep mask
    drawn from a vectorised Philox4x32-10 on the host (pinned to the oracle's scalar one);
  * idl_rmsprop_allreduce_step with W pseudo-ranks on one GPU (the kernel only dereferences the addresses it is given) against
    idl_rmsprop_step on the rank-order sum of the gradients, bit for bit;
  * whole ShardedTrainer steps, eager and replayed from the CUDA graph, against NetLinear rebuilt in float64 from the parameters
    before the step: keep masks, loss, every gradient slice, the optimiser update and the hand-over of the next batch."""
import math
import sys

import numpy as np
import pytest

import idelucs_oracle as orc

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

M32 = np.uint64(0xFFFFFFFF)


def _philox(c0, c1, c2, c3, k0, k1):
    """Philox4x32-10 over arrays of counters (uint64 arrays holding 32-bit words; the 32 x 32-bit products are exact in 64 bits)"""
    c0, c1, c2, c3 = (np.asarray(c, dtype=np.uint64) & M32 for c in (c0, c1, c2, c3))
    k0, k1 = np.uint64(int(k0) & 0xFFFFFFFF), np.uint64(int(k1) & 0xFFFFFFFF)
    for _ in range(10):
        p0 = np.uint64(0xD2511F53) * c0
        p1 = np.uint64(0xCD9E8D57) * c2
        c0, c1, c2, c3 = ((p1 >> np.uint64(32)) ^ c1 ^ k0) & M32, p1 & M32, ((p0 >> np.uint64(32)) ^ c3 ^ k1) & M32, p0 & M32
        k0, k1 = (k0 + np.uint64(0x9E3779B9)) & M32, (k1 + np.uint64(0xBB67AE85)) & M32
    return c0, c1, c2, c3


def _words(n, seed, step, tag):
    """the dropout word of elements 0..n-1 of training step `step`: counter (e div 4, step lo, step hi, tag ^ ((e div 4) >> 32)),
    key (seed lo, seed hi), word e mod 4"""
    q = np.arange((n + 3) // 4, dtype=np.uint64)
    w = _philox(q, np.full_like(q, step & 0xFFFFFFFF), np.full_like(q, step >> 32), np.uint64(tag) ^ (q >> np.uint64(32)), seed, seed >> 32)
    return np.stack(w, 1).reshape(-1)[:n]


def _thresh(p):
    """elements whose word is below floor(float64(float32 p) 2^32) are dropped"""
    return min(int(float(np.float32(p)) * 4294967296.0), 0xFFFFFFFF)


def _inv_keep(p):
    return np.float32(1) / (np.float32(1) - np.float32(p))


def test_vectorised_philox_equals_oracle():
    rng = np.random.default_rng(17)
    c = rng.integers(0, 2 ** 32, size=(300, 4), dtype=np.uint64)
    k = rng.integers(0, 2 ** 32, size=(300, 2), dtype=np.uint64)
    c[:3] = [[0, 0, 0, 0], [0xFFFFFFFF] * 4, [0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344]]
    k[:3] = [[0, 0], [0xFFFFFFFF] * 2, [0xa4093822, 0x299f31d0]]
    for i in range(300):
        got = _philox(*(c[i:i + 1, j] for j in range(4)), k[i, 0], k[i, 1])
        assert tuple(int(g[0]) for g in got) == orc.philox4x32_10(tuple(c[i]), tuple(k[i])), i
    # the same words in one call over every counter at once
    full = _philox(c[:, 0], c[:, 1], c[:, 2], c[:, 3], 0x12345678, 0x9ABCDEF0)
    for i in range(0, 300, 37):
        assert tuple(int(g[i]) for g in full) == orc.philox4x32_10(tuple(c[i]), (0x12345678, 0x9ABCDEF0))


# ---------------------------------------------------------------------------------------------------------------------------------
# a. fused ReLU - Dropout, its backward and idl_sum_parts_bias, bit for bit
# ---------------------------------------------------------------------------------------------------------------------------------
SHAPES = [(1, 4), (3, 12), (7, 20), (1024, 512), (1024, 64), (4096, 516)]   # the last one runs the grid-stride loops (M N > 1184 x 1024)
PARTS = [1, 2, 4, 8, 16]
PS = [0.0, 0.1, 0.5, 0.9, 1.0 - 2.0 ** -24]
STEPS = [None, 5, 2 ** 32 + 3]
KEYS = [((1 << 40) | 0x1234567, 1), (0xFEDCBA9876543210, 2), ((3 << 61) + 12345, 0xDEADBEEF)]


def _bits(a):
    return np.ascontiguousarray(a, dtype=np.float32).view(np.uint32)


@pytest.mark.parametrize("shape", SHAPES, ids=["%dx%d" % s for s in SHAPES])
def test_relu_dropout_and_sum_parts_bit_exact(shape):
    from idelucs_b200 import _lib
    lib = _lib.load()
    M, N = shape
    rng = np.random.default_rng(M * 1000 + N)
    words = {}
    for i, (n_parts, with_bias) in enumerate((n, b) for n in PARTS for b in (True, False)):
        p = PS[(i + M) % len(PS)]
        step = STEPS[i % 3]
        seed, tag = KEYS[(i // 3 + i) % 3]
        parts = rng.standard_normal((n_parts, M, N), dtype=np.float32)
        bias = rng.standard_normal(N, dtype=np.float32) if with_bias else None
        dy = rng.standard_normal((M, N), dtype=np.float32)
        # numpy float32: parts added in index order, then the bias
        v = parts[0].copy()
        for q in range(1, n_parts):
            v = v + parts[q]
        if bias is not None:
            v = v + bias
        t = 0 if step is None else step
        if (t, seed, tag) not in words:
            words[(t, seed, tag)] = _words(M * N, seed, t, tag).reshape(M, N)
        kept = words[(t, seed, tag)] >= np.uint64(_thresh(p))
        ik = _inv_keep(p)
        want = np.where((v > 0) & kept, v * ik, np.float32(0)).astype(np.float32)
        want_dx = np.where(want > 0, dy * ik, np.float32(0)).astype(np.float32)

        d_parts = torch.from_numpy(parts).cuda()
        d_bias = None if bias is None else torch.from_numpy(bias).cuda()
        d_step = None if step is None else torch.tensor(step, dtype=torch.int64, device="cuda")
        out = torch.full((M, N), 7.0, device="cuda")
        _lib.check(lib.idl_relu_dropout_forward(_lib.ptr(d_parts), n_parts, _lib.ptr(d_bias), M, N, p, seed, _lib.ptr(d_step), tag, _lib.ptr(out),
                                                _lib.stream_ptr()))
        got = out.cpu().numpy()
        case = (M, N, n_parts, with_bias, p, step, hex(seed), tag)
        assert np.array_equal(_bits(got), _bits(want)), (case, int((_bits(got) != _bits(want)).sum()))
        dx = torch.full((M, N), 7.0, device="cuda")
        _lib.check(lib.idl_relu_dropout_backward(_lib.ptr(out), _lib.ptr(torch.from_numpy(dy).cuda()), M * N, p, _lib.ptr(dx), _lib.stream_ptr()))
        assert np.array_equal(_bits(dx.cpu().numpy()), _bits(want_dx)), case
        s = torch.full((M, N), 7.0, device="cuda")
        _lib.check(lib.idl_sum_parts_bias(_lib.ptr(d_parts), n_parts, _lib.ptr(d_bias), M, N, _lib.ptr(s), _lib.stream_ptr()))
        assert np.array_equal(_bits(s.cpu().numpy()), _bits(v)), case
        if p == 0.5 and M * N >= 4096:   # the law: about half of the active units survive
            assert abs(float(kept.mean()) - 0.5) < 0.02, case


# ---------------------------------------------------------------------------------------------------------------------------------
# b. idl_rmsprop_allreduce_step, W pseudo-ranks on one GPU
# ---------------------------------------------------------------------------------------------------------------------------------
LR, ALPHA, EPS, WD = 1e-3, 0.99, 1e-8, 0.01
GUARD = 64            # sentinel floats on either side of every buffer (256 bytes: the buffers stay 16-byte aligned)
SENTINEL = -1234.5


def _guarded(n, fill=None):
    """[GUARD | n | GUARD] float32 on the device, sentinel-filled; returns (whole buffer, the n-float view)"""
    whole = torch.full((n + 2 * GUARD,), SENTINEL, device="cuda")
    if fill is not None:
        whole[GUARD:GUARD + n].copy_(fill)
    return whole, whole[GUARD:GUARD + n]


def _sentinels_intact(whole):
    return bool((whole[:GUARD] == SENTINEL).all()) and bool((whole[-GUARD:] == SENTINEL).all())


def _trainer_k6_size(W):
    from idelucs_b200.PytorchUtils import NetLinear
    n = sum(p.numel() for p in NetLinear(4096, 5).parameters())
    return n + (-n) % (4 * W)


@pytest.mark.parametrize("W", [1, 2, 3, 4, 8, 16])
def test_rmsprop_allreduce_pseudo_ranks_equal_rmsprop_step(W):
    import ctypes
    from idelucs_b200 import _lib
    lib = _lib.load()
    gen = torch.Generator(device="cuda").manual_seed(W)
    # smallest allowed; a shard whose grid-stride loop iterates (> 148 x 256 x 4 x 4 floats); the trainer's k = 6 buffer, padded
    for n_total in (4 * W, W * (606208 + 4 * 1001), _trainer_k6_size(W)):
        shard = n_total // W
        p0 = torch.randn(n_total, device="cuda", generator=gen)
        params = [_guarded(n_total, p0) for _ in range(W)]
        grads = [_guarded(n_total) for _ in range(W)]
        sqs = [_guarded(shard, torch.zeros(shard)) for _ in range(W)]
        p_ref, sq_ref = p0.clone(), torch.zeros(n_total, device="cuda")
        gp = (ctypes.c_uint64 * W)(*[g[1].data_ptr() for g in grads])
        pp = (ctypes.c_uint64 * W)(*[p[1].data_ptr() for p in params])
        for step in range(3):   # sq carries over
            total = torch.zeros(n_total, device="cuda")
            for r in range(W):
                grads[r][1].copy_(torch.randn(n_total, device="cuda", generator=gen) * 10.0 ** (step - 1))
                total += grads[r][1]                                  # float32, rank order, from zero: the kernel's sum
            for r in range(W):
                _lib.check(lib.idl_rmsprop_allreduce_step(gp, pp, 0, 0, _lib.ptr(sqs[r][1]), n_total, r, W, LR, ALPHA, EPS, WD, _lib.stream_ptr()))
            _lib.check(lib.idl_rmsprop_step(_lib.ptr(p_ref), _lib.ptr(total), _lib.ptr(sq_ref), n_total, LR, ALPHA, EPS, WD,
                                            float(np.float32(1) / np.float32(W)), _lib.stream_ptr()))
            torch.cuda.synchronize()
            case = (W, n_total, step)
            for r in range(W):
                assert torch.equal(sqs[r][1], sq_ref[r * shard:(r + 1) * shard]), (case, r)
                assert torch.equal(params[r][1], p_ref), (case, r, int((params[r][1] != p_ref).sum()))
            assert all(_sentinels_intact(b[0]) for b in params + grads + sqs), case


# ---------------------------------------------------------------------------------------------------------------------------------
# c. ShardedTrainer steps against a float64 reference step
# ---------------------------------------------------------------------------------------------------------------------------------
U32 = 2.0 ** -24     # unit roundoff of float32
LAMBDA = 10.0        # probabilistic bound on an fp32 inner product of n terms (Higham & Mary, SIAM J. Sci. Comput. 2019):
#                      |error| <= LAMBDA sqrt(n) u sum |x_i w_i| except with probability <= 2 n exp(-LAMBDA^2 / 2) (< 1e-17 per element)


def _delta(n):
    return LAMBDA * math.sqrt(n) * U32


def _views(tr, flat):
    """the network's parameters as views into a flat buffer laid out like the trainer's"""
    out, o = [], 0
    for p in tr.net.parameters():
        out.append(flat[o:o + p.numel()].view_as(p))
        o += p.numel()
    return out


def _keep(tr, step, tag, shape):
    w = _words(shape[0] * shape[1], tr._drop_seed, step, tag).reshape(shape)
    return torch.from_numpy(w >= np.uint64(_thresh(0.5))).cuda()


def _check_step(tr, before, after, ids, rec1, rec2, loss):
    """one step of the trainer against its float64 restatement: `before` = (P, sq, x) snapshotted before it"""
    from idelucs_b200 import _lib
    from test_gpu_parity import _ref_iid64, _ref_style_info_nce
    P, sq, x = before
    t = int(tr._step_no.item())
    tag = "step %d" % t
    # 1. the hand-over: the batch the next step consumes is the featurised pairs of the ids drawn in this one
    assert torch.equal(tr._batch, tr.loader.batch(ids)["both"]), tag
    # 2. NetLinear in float64, with the ReLU - Dropout factors 2 [out > 0] of the kernels' outputs
    W1, b1, W2, b2, W3, b3 = params = [v.detach().double().requires_grad_(True) for v in _views(tr, P)]
    xd = x.double()
    B = x.shape[0] // 2
    a1 = xd @ W1.t() + b1
    f1 = 2.0 * (rec1 > 0).double()
    d1 = a1 * f1
    h = d1 @ W2.t() + b2
    f2 = 2.0 * (rec2 > 0).double()
    z = torch.softmax((h * f2) @ W3.t() + b3, 1)
    want = (1 - tr.weight) * _ref_style_info_nce(h[:B], h[B:], 0.85) + tr.weight * _ref_iid64(z[:B], z[B:], tr.lamb)
    gwant = torch.autograd.grad(want, params)
    with torch.no_grad():
        # keep masks: the kernels' active set == [a64 > 0] and the host Philox keep bit, outside the band where fp32 rounding can
        # move a pre-activation across zero
        K1 = W1.shape[1]
        s1 = xd.abs() @ W1.abs().t() + b1.abs()
        band1 = a1.abs() <= _delta(K1 + tr.first_layer_split + 1) * s1
        act1 = (a1 > 0) & _keep(tr, t, 1, tuple(a1.shape))
        assert torch.equal((rec1 > 0)[~band1], act1[~band1]), (tag, int(((rec1 > 0) != act1)[~band1].sum()))
        assert bool(((rec1.double() - d1).abs() <= 2 * _delta(K1 + tr.first_layer_split + 1) * s1).all()), tag   # (x 2: 1 / (1 - p))
        r1 = rec1.double()
        s2 = r1.abs() @ W2.abs().t() + b2.abs()
        band2 = h.abs() <= _delta(W2.shape[1] + tr.small_gemm_split[0] + 1) * s2 + (r1 - d1).abs() @ W2.abs().t()
        act2 = (h > 0) & _keep(tr, t, 2, tuple(h.shape))
        assert torch.equal((rec2 > 0)[~band2], act2[~band2]), (tag, int(((rec2 > 0) != act2)[~band2].sum()))
        for band in (band1, band2):
            assert int(band.sum()) <= 0.005 * band.numel() + 4, (tag, int(band.sum()), band.numel())
        kept = float(((rec1 > 0) & (a1 > 0)).sum()) / float((a1 > 0).sum())
        assert abs(kept - 0.5) < 0.03, (tag, kept)
        # loss and every parameter's gradient slice
        assert abs(float(loss) - float(want)) < 2e-5, (tag, float(loss), float(want))
        for g, gw, p in zip(_views(tr, tr._flat_grad), gwant, tr.net.parameters()):
            assert float((g.double() - gw).abs().max()) <= 1e-4 * float(gw.abs().max()), (tag, tuple(p.shape))
    # 3. the optimiser: idl_rmsprop_step on copies of the state before the step and the gradients it wrote
    lib = _lib.load()
    P2, sq2 = P.clone(), sq.clone()
    _lib.check(lib.idl_rmsprop_step(_lib.ptr(P2), _lib.ptr(tr._flat_grad), _lib.ptr(sq2), P2.numel(), tr.lr, tr.alpha, tr.eps, tr.weight_decay, 1.0,
                                    _lib.stream_ptr()))
    assert torch.equal(after[0], P2) and torch.equal(after[1], sq2), tag


def _random_seqset(n, seed):
    from idelucs_b200.seqset import SeqSet
    rng = np.random.default_rng(seed)
    alph = np.frombuffer(b"ACGT", dtype=np.uint8)
    return SeqSet.from_sequences([alph[rng.integers(0, 4, size=int(L))].tobytes() for L in rng.integers(500, 3000, size=n)])


CONFIGS = [(6, 5, 512), (3, 12, 100), (4, 200, 333)]


@pytest.mark.parametrize("k,C,B", CONFIGS, ids=["k%d_C%d_B%d" % c for c in CONFIGS])
def test_sharded_trainer_steps_equal_float64_reference(monkeypatch, k, C, B):
    from idelucs_b200 import train
    tr = train.ShardedTrainer(_random_seqset(300, k), k=k, n_clusters=C, n_mimics=3, batch_sz=B, seed=k)
    recs, drawn = [], []
    fwd = train._relu_dropout_fwd

    def recording_fwd(*a):
        out = fwd(*a)
        recs.append(out.clone())   # under capture the clone is part of the graph: every replay refreshes it
        return out
    monkeypatch.setattr(train, "_relu_dropout_fwd", recording_fwd)
    nxt = tr._next_ids

    def recording_next_ids():
        ids = nxt()
        drawn.append(ids.clone())
        return ids
    tr._next_ids = recording_next_ids
    tr._batch = tr._featurise(tr._next_ids()).clone()   # (what step() does before the first step)

    def snapshot():
        return tr._flat_param.clone(), tr._sq.clone(), tr._batch.clone()

    for i in range(3):   # eager steps
        before = snapshot()
        if i == 1:       # gradients are written into the flat buffer, never accumulated
            for g in _views(tr, tr._flat_grad):
                g.fill_(1e30)
        loss = tr.step()
        torch.cuda.synchronize()
        _check_step(tr, before, (tr._flat_param, tr._sq), drawn[-1], recs[-2], recs[-1], loss.item())
    assert tr.enable_cuda_graph(), getattr(tr, "_graph_error", "")
    cap1, cap2 = recs[-2], recs[-1]
    prev_t, prev_mask = int(tr._step_no.item()), None
    for i in range(3):   # graph replays
        before = snapshot()
        tr.step()
        torch.cuda.synchronize()
        assert int(tr._step_no.item()) == prev_t + 1
        prev_t = int(tr._step_no.item())
        _check_step(tr, before, (tr._flat_param, tr._sq), drawn[-1], cap1, cap2, tr._loss.item())
        mask = cap1 > 0
        assert prev_mask is None or not torch.equal(mask, prev_mask), "a replay drew the previous mask again"
        prev_mask = mask
    # one replay == the same step run eagerly from the same state
    tr._ids.copy_(tr._next_ids())
    state = [t.clone() for t in (tr._flat_param, tr._sq, tr._step_no, tr._batch, tr._ids)]
    tr._graph.replay()
    torch.cuda.synchronize()
    replayed = [t.clone() for t in (tr._flat_param, tr._flat_grad, tr._sq, tr._loss, tr._batch)]
    for t, s in zip((tr._flat_param, tr._sq, tr._step_no, tr._batch, tr._ids), state):
        t.copy_(s)
    loss = tr._step_from_ids()
    torch.cuda.synchronize()
    for name, a, b in zip(("parameters", "gradients", "sq", "loss", "next batch"), replayed, (tr._flat_param, tr._flat_grad, tr._sq, loss, tr._batch)):
        assert torch.equal(a, b), (name, int((a != b).sum()))
