"""The k = 6 two-call path (idl_profiles_prepare + idl_profiles_prepared) through its C ABI, beyond what the Python
wrappers use: item lists (d_sidx), stale prepared buffers, output layouts, the capacity limits of the producer/consumer
kernel, the status / statistics contracts and the IEEE arithmetic of the standardised rows.

Three yardsticks for every call:
  * the generic kernel (plain idl_profiles on the same request) must match bit for bit;
  * the oracle (mutate-and-recount, float32((c + pc) / sum), then (x - mean32) / scale32 in numpy float32) on sampled
    (item, slot) pairs, always on the first, last and edge-length items;
  * the route.  The results are identical whichever kernel produced them, so each call also reports
      - how many kernels it launched: the fast route launches profiles_pc_kernel ahead of the generic kernel's
        deferred-item pass, one launch more than the fallback (idl_launch_count);
      - the deferred-item counter work_counter[1] (a uint64 at byte 8 of the profile workspace): fill_params zeroes it,
        prep_kernel and profiles_pc_kernel add one per item they hand to the generic kernel.
    A call on the fast route with a matching buffer defers exactly the items the prepare pass flagged; with a stale
    buffer it defers every item; the fallback route defers none."""
import ctypes

import numpy as np
import pytest

import idelucs_oracle as orc

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

F = 4096
MAX_LEN = 20480          # longest item the fast kernels stage in shared memory (SSEQ_CHUNKS x 64 bases)
ALPH = np.frombuffer(b"ACGTACGTACGTACGTACGTACGTN", dtype=np.uint8)
ACGT = np.frombuffer(b"ACGT", dtype=np.uint8)


class Abi(object):
    """ctypes calls of the two entry points; every call checks that d_status is all zero afterwards"""

    def __init__(self):
        from idelucs_b200 import _lib, featurise
        from idelucs_b200.seqset import SeqSet
        self.L, self.ft, self.SeqSet = _lib, featurise, SeqSet
        self.lib = _lib.load()
        self.dev = torch.device("cuda", torch.cuda.current_device())
        self.sm = torch.cuda.get_device_properties(self.dev).multi_processor_count
        self.STD, self.FREQ = featurise.OUT_STD_F32, featurise.OUT_FREQ_F32

    def deferred(self):
        """work_counter[1] of the last call on the current stream (kernels.cu fill_params: uint64 at byte 8)"""
        torch.cuda.synchronize()
        ws = self.ft._workspace(self.dev, self.lib.idl_profiles_workspace_bytes(), "prof")
        return int(ws[8:16].cpu().numpy().view(np.uint64)[0])

    def prepare(self, ss, variants, n=None, sidx=None, seed=0, seq_id0=0, pc=1, stats=True):
        n = (ss.n if sidx is None else int(sidx.numel())) if n is None else n
        buf = torch.empty(self.lib.idl_prepare_bytes(n), dtype=torch.uint8, device=self.dev)
        parts, part_n = self.ft._stats_buffers(F, self.dev) if stats else (None, None)
        n_parts = ctypes.c_int(0)
        status = torch.zeros(n, dtype=torch.int32, device=self.dev)
        self.L.check(self.lib.idl_profiles_prepare(
            *self.ft._seqset_args(ss), self.L.ptr(sidx), n, seq_id0, 6, self.ft._variant_array(variants), len(variants), self.ft._seed(seed),
            pc, self.L.ptr(buf), buf.numel(), self.L.ptr(parts), self.L.ptr(part_n), self.ft.MAX_PARTS, ctypes.byref(n_parts),
            self.L.ptr(status), *self.ft._workspace_args(self.lib, self.dev)))
        flagged = self.deferred()
        assert int(status.count_nonzero()) == 0, "d_status not zero after idl_profiles_prepare"
        # PrepMeta.flags (prep.cuh: 64-byte header, then 32 bytes per item, flags at byte 12): the items left to the generic kernel
        flags = buf[64:64 + 32 * n].view(torch.int32).reshape(n, 8)[:, 3].cpu().numpy()
        assert int((flags != 0).sum()) == flagged, "deferred-item counter disagrees with the prepared buffer's flags"
        scaler = self.ft.Scaler.from_partials(parts[:n_parts.value], part_n[:n_parts.value]) if stats else None
        return Prep(buf, flagged, flags != 0, scaler)

    def prepared(self, ss, variants, prep, out_kind, n=None, sidx=None, seed=0, seq_id0=0, pc=1, mean=None, scale=None,
                 out=None, out_off=None, out_stride=F):
        """-> (out, took_fast_route, deferred items)"""
        n = (ss.n if sidx is None else int(sidx.numel())) if n is None else n
        S = len(variants)
        if out is None:
            out = torch.full((S, n, F), float("nan"), dtype=torch.float32, device=self.dev)
            out_off = [s * n * F for s in range(S)]
        status = torch.zeros(n, dtype=torch.int32, device=self.dev)
        offs = (ctypes.c_int64 * S)(*[int(o) for o in out_off])
        torch.cuda.synchronize()
        l0 = self.lib.idl_launch_count()
        self.L.check(self.lib.idl_profiles_prepared(
            *self.ft._seqset_args(ss), self.L.ptr(sidx), n, seq_id0, 6, self.ft._variant_array(variants), S, self.ft._seed(seed), out_kind,
            self.L.ptr(out), offs, out_stride, pc, self.L.ptr(mean), self.L.ptr(scale), self.L.ptr(status), self.L.ptr(prep.buf),
            prep.buf.numel(), *self.ft._workspace_args(self.lib, self.dev)))
        launches = self.lib.idl_launch_count() - l0
        deferred = self.deferred()
        assert int(status.count_nonzero()) == 0, "d_status not zero after idl_profiles_prepared"
        base = 2 if out_kind == self.STD else 1     # (rscale_kernel) + the generic kernel
        assert launches in (base, base + 1), launches
        return out, launches == base + 1, deferred

    def generic(self, ss, variants, out_kind, sidx=None, seed=0, seq_id0=0, pc=1, mean=None, scale=None):
        return self.ft.profiles(ss, 6, variants, out_kind=out_kind, seed=seed, sidx=sidx, seq_id0=seq_id0, pseudocount=pc,
                                mean=mean, scale=scale, chunked=False)

    def route(self, what, ss, variants, prep, out_kind, fast, deferred=None, want=None, **kw):
        """idl_profiles_prepared == ``want`` (default: the generic kernel on the same request), then its route"""
        got, took_fast, n_def = self.prepared(ss, variants, prep, out_kind, **kw)
        if want is None:
            want = self.generic(ss, variants, out_kind, **{k: v for k, v in kw.items() if k not in ("n",)})
        same(got, want, what)
        assert took_fast == fast, "%s: %s route taken, expected the %s route" % (what, "fast" if took_fast else "fallback", "fast" if fast else "fallback")
        want_def = (prep.flagged if deferred is None else deferred) if fast else 0
        assert n_def == want_def, "%s: %d items deferred to the generic kernel, expected %d" % (what, n_def, want_def)
        return got


class Prep(object):
    def __init__(self, buf, flagged, flag_mask, scaler):
        self.buf, self.flagged, self.flag_mask, self.scaler = buf, flagged, flag_mask, scaler


def same(got, want, what):
    """bit-for-bit equality with a report of where the first rows differ"""
    assert got.shape == want.shape, (what, tuple(got.shape), tuple(want.shape))
    g, w = got.contiguous().view(torch.int32), want.contiguous().view(torch.int32)
    if torch.equal(g, w):
        return
    bad = (g != w).reshape(-1, got.shape[-1]).any(dim=1).nonzero().flatten()[:5].tolist()
    rows = [divmod(r, got.shape[-2]) if got.dim() == 3 else r for r in bad]
    n_bad = int((g != w).reshape(-1, got.shape[-1]).any(dim=1).sum())
    raise AssertionError("%s: %d rows differ from the yardstick, first (slot, item): %s" % (what, n_bad, rows))


def oracle_row(seq, seq_id, spec, seed, pc, mean=None, scale=None):
    """float32 profile of one (sequence, variant): the oracle's mutations, recounted from scratch"""
    edits = orc.rng_variant_edits(seed, seq_id, spec.rng_id, spec.kind, orc.codes_of_seq(seq), len(seq), spec.p1, spec.p2, spec.n_bp)
    mut = bytearray(seq)
    for pos, val in edits:
        mut[pos] = b"ACGTN"[val]
    cnt = np.zeros(F, np.int64)
    orc.kmer_counts(mut, 6, cnt)
    c = cnt + pc
    x = (c / c.sum()).astype(np.float32)
    if mean is not None:
        x = (x - mean) / scale
    return x


def check_oracle(got, seqs, variants, items, slots, seed, seq_id0=0, sidx=None, pc=1, scaler=None, mean=None, scale=None):
    if scaler is not None:
        mean, scale = scaler.mean32, scaler.scale32
    m = None if mean is None else mean.cpu().numpy()
    s = None if scale is None else scale.cpu().numpy()
    sx = None if sidx is None else sidx.cpu().numpy()
    for w in sorted(set(int(i) for i in items)):
        q = w if sx is None else int(sx[w])
        row = got[:, w].cpu().numpy()
        for v in sorted(set(slots)):
            want = oracle_row(seqs[q], seq_id0 + q, variants[v], seed, pc, m, s)
            assert np.array_equal(row[v].view(np.int32), want.view(np.int32)), \
                "oracle: item %d (sequence %d, length %d) slot %d: %d bins differ" % (w, q, len(seqs[q]), v, int((row[v] != want).sum()))


def V(ft, kind, p1=0.0, p2=0.0, n_bp=0, rng_id=0):
    return ft.VariantSpec(kind, p1, p2, n_bp, rng_id=rng_id)


def schedule(ft, n_randn=4, n_bp=20):
    """the reference schedule (three Bernoulli slots first) with a clean slot at the end"""
    v = [V(ft, ft.KIND_BOTH, 1e-2, 0.5e-2, rng_id=0), V(ft, ft.KIND_TRANSITION, p1=1e-2, rng_id=1), V(ft, ft.KIND_TRANSVERSION, p2=0.5e-2, rng_id=2)]
    v += [V(ft, ft.KIND_RANDOM_N, n_bp=n_bp, rng_id=3 + i) for i in range(n_randn)]
    return v + [V(ft, ft.KIND_CLEAN, rng_id=3 + n_randn)]


def bern_slots(ft, variants):
    return [i for i, v in enumerate(variants) if v.kind in (ft.KIND_TRANSITION, ft.KIND_TRANSVERSION, ft.KIND_BOTH)]


def random_seqs(rng, lens, alph=ALPH):
    return [alph[rng.integers(0, alph.size, size=int(L))].tobytes() for L in lens]


@pytest.fixture(scope="module")
def abi():
    return Abi()


@pytest.fixture(scope="module")
def base(abi):
    """700 sequences: ragged lengths, a few the prepare pass must flag (longer than 20 480 bases, or so many mutations that
    the on-chip delta list overflows)"""
    rng = np.random.default_rng(7)
    lens = rng.integers(40, 6000, size=700)
    lens[[3, 100, 401, 650]] = [MAX_LEN + 1, 30000, 17000, 15500]
    seqs = random_seqs(rng, lens)
    return seqs, abi.SeqSet.from_sequences(seqs)


def sample_items(n, rng, extra=()):
    return [0, n - 1] + rng.integers(0, n, size=3).tolist() + list(extra)


# ---------------------------------------------------------------- item selection
@pytest.mark.parametrize("kind", ["permutation", "repeated", "strided"])
def test_sidx_through_both_calls(abi, base, kind):
    """the same d_sidx for prepare and prepared: the RNG id of item w is seq_id0 + sidx[w]; statistics equal
    idl_profile_stats over the same items"""
    ft = abi.ft
    seqs, ss = base
    rng = np.random.default_rng(["permutation", "repeated", "strided"].index(kind))
    if kind == "permutation":
        idx = rng.permutation(ss.n)[:500]
        idx[[10, 200]] = [3, 100]                                  # flagged items at two places
    elif kind == "repeated":
        idx = rng.integers(0, 40, size=400)
        idx[[0, 1, 399]] = [401, 401, 3]
    else:
        idx = np.arange(3, ss.n, 2)
    sidx = torch.from_numpy(idx.astype(np.int32)).to(abi.dev)
    n = sidx.numel()
    variants = schedule(ft)
    seed, seq_id0 = 0x5EED0001, 1000
    prep = abi.prepare(ss, variants, sidx=sidx, seed=seed, seq_id0=seq_id0)
    long_items = np.nonzero(ss.lengths[idx] > MAX_LEN)[0]
    assert prep.flag_mask[long_items].all() and prep.flagged >= max(1, long_items.size)
    # statistics: idl_profile_stats over the same items
    parts, part_n = ft._stats_buffers(F, abi.dev)
    n_parts = ctypes.c_int(0)
    abi.L.check(abi.lib.idl_profile_stats(*ft._seqset_args(ss), abi.L.ptr(sidx), n, seq_id0, 6, ft._variant_array(variants[:1]), ft._seed(seed),
                                          None, None, 1, abi.L.ptr(parts), abi.L.ptr(part_n), ft.MAX_PARTS, ctypes.byref(n_parts), None,
                                          *ft._workspace_args(abi.lib, abi.dev)))
    g = ft.Scaler.from_partials(parts[:n_parts.value], part_n[:n_parts.value])
    a = prep.scaler
    assert torch.allclose(g.mean64, a.mean64, rtol=1e-13, atol=0) and torch.allclose(g.scale64, a.scale64, rtol=1e-9, atol=0)
    assert float(((g.mean32 - a.mean32).abs() / g.mean32.abs()).max()) < 2e-7
    kw = dict(sidx=sidx, seed=seed, seq_id0=seq_id0)
    f = abi.route("FREQ, sidx " + kind, ss, variants, prep, abi.FREQ, True, **kw)
    s = abi.route("STD, sidx " + kind, ss, variants, prep, abi.STD, True, mean=a.mean32, scale=a.scale32, **kw)
    if kind == "repeated":                                         # repeated items: identical rows in every slot
        first = {}
        for w, q in enumerate(idx.tolist()):
            first.setdefault(q, w)
        pairs = [(first[q], w) for w, q in enumerate(idx.tolist()) if first[q] != w]
        assert pairs
        for w0, w1 in pairs[:50]:
            assert torch.equal(f[:, w0], f[:, w1]) and torch.equal(s[:, w0], s[:, w1]), (w0, w1)
    items = sample_items(n, rng, [int(np.nonzero(prep.flag_mask)[0][0])])
    slots = [0, 1, 2, 3, len(variants) - 1]
    check_oracle(f, seqs, variants, items, slots, seed, seq_id0, sidx)
    check_oracle(s, seqs, variants, items[:3], slots, seed, seq_id0, sidx, scaler=a)


# ---------------------------------------------------------------- stale buffers
STALE = ["seed", "seq_id0", "pseudocount", "slot0_kind", "bern_rate", "bern_rng_id", "added_bern", "n_items", "seqset", "sidx"]


@pytest.mark.parametrize("field", STALE)
def test_stale_buffer_defers_every_item(abi, base, field):
    """a buffer prepared for call A, used for a call B that differs in one stamped field: the fast kernel notices (every
    item deferred) and B's rows are the generic kernel's"""
    ft = abi.ft
    seqs, ss_full = base
    ss = abi.SeqSet.from_sequences(seqs[:400])
    rng = np.random.default_rng(11)
    perm_a = torch.from_numpy(rng.permutation(400).astype(np.int32)).to(abi.dev)
    va = [V(ft, ft.KIND_BOTH, 1e-2, 0.5e-2, rng_id=0), V(ft, ft.KIND_TRANSITION, p1=1e-2, rng_id=1),
          V(ft, ft.KIND_RANDOM_N, n_bp=20, rng_id=3), V(ft, ft.KIND_RANDOM_N, n_bp=20, rng_id=4), V(ft, ft.KIND_CLEAN, rng_id=5)]
    A = dict(ss=ss, variants=va, seed=9, seq_id0=0, pc=1, n=400, sidx=None)
    B = dict(A)
    if field == "seed":
        B["seed"] = 10
    elif field == "seq_id0":
        B["seq_id0"] = 1
    elif field == "pseudocount":
        B["pc"] = 2
    elif field == "slot0_kind":
        B["variants"] = [V(ft, ft.KIND_TRANSITION, 1e-2, 0.5e-2, rng_id=0)] + va[1:]
    elif field == "bern_rate":
        B["variants"] = va[:1] + [V(ft, ft.KIND_TRANSITION, p1=2e-2, rng_id=1)] + va[2:]
    elif field == "bern_rng_id":
        B["variants"] = va[:1] + [V(ft, ft.KIND_TRANSITION, p1=1e-2, rng_id=7)] + va[2:]
    elif field == "added_bern":                                    # a third Bernoulli slot, ahead of the second one
        B["variants"] = va[:1] + [V(ft, ft.KIND_TRANSVERSION, p2=0.5e-2, rng_id=2)] + va[1:]
    elif field == "n_items":
        B["n"] = 399
    elif field == "seqset":                                        # same lengths, other bases; A's set stays alive
        B["ss"] = abi.SeqSet.from_sequences(random_seqs(rng, [len(s) for s in seqs[:400]]))
    elif field == "sidx":
        A["sidx"] = perm_a
        B["sidx"] = torch.flip(perm_a, [0]).contiguous()
    prep = abi.prepare(A["ss"], A["variants"], n=A["n"], sidx=A["sidx"], seed=A["seed"], seq_id0=A["seq_id0"], pc=A["pc"])

    def gen(c):
        x = abi.generic(c["ss"], c["variants"], abi.FREQ, sidx=c["sidx"], seed=c["seed"], seq_id0=c["seq_id0"], pc=c["pc"])
        return x[:, :c["n"]]

    ga, gb = gen(A), gen(B)
    if field != "n_items":
        # the check is not vacuous: the rows A's buffer describes are not B's (for n_items, A's rows are B's, but the delta
        # section of the buffer starts at an offset that depends on n_items)
        rows = bern_slots(ft, B["variants"])
        assert not torch.equal(ga[rows].view(torch.int32), gb[rows].view(torch.int32)), field
    abi.route("stale " + field, B["ss"], B["variants"], prep, abi.FREQ, True, deferred=B["n"], want=gb, n=B["n"], sidx=B["sidx"],
              seed=B["seed"], seq_id0=B["seq_id0"], pc=B["pc"])


@pytest.mark.parametrize("change", ["randn_nbp", "randn_rng_id", "slot_positions", "freq_then_std", "other_statistics"])
def test_changes_outside_the_stamp_keep_the_fast_route(abi, base, change):
    """what the prepared buffer does not depend on may change between prepare and prepared: still the fast route, still exact"""
    ft = abi.ft
    seqs, ss = base
    va = schedule(ft, n_randn=3)
    seed, seq_id0 = 77, 5
    prep = abi.prepare(ss, va, seed=seed, seq_id0=seq_id0)
    kw = dict(seed=seed, seq_id0=seq_id0)
    sc = prep.scaler
    rng = np.random.default_rng(3)
    items = sample_items(ss.n, rng)
    if change in ("randn_nbp", "randn_rng_id", "slot_positions"):
        vb = list(va)
        if change == "randn_nbp":
            vb[4] = V(ft, ft.KIND_RANDOM_N, n_bp=7, rng_id=4)
        elif change == "randn_rng_id":
            vb[4] = V(ft, ft.KIND_RANDOM_N, n_bp=20, rng_id=40)
        else:                                                      # Bernoulli slots keep their order, the others move around them
            vb = [va[0], va[3], va[6], va[1], va[4], va[2], va[5]]
        got = abi.route(change, ss, vb, prep, abi.STD, True, mean=sc.mean32, scale=sc.scale32, **kw)
        check_oracle(got, seqs, vb, items, range(len(vb)), seed, seq_id0, scaler=sc)
    elif change == "freq_then_std":
        f = abi.route("FREQ", ss, va, prep, abi.FREQ, True, **kw)
        abi.route("STD after FREQ", ss, va, prep, abi.STD, True, mean=sc.mean32, scale=sc.scale32, **kw)
        check_oracle(f, seqs, va, items, range(len(va)), seed, seq_id0)
    else:
        m2 = (torch.rand(F, device=abi.dev) * 1e-3).float()
        s2 = (torch.rand(F, device=abi.dev) * 1e-3 + 1e-5).float()
        abi.route("STD, prepare's statistics", ss, va, prep, abi.STD, True, mean=sc.mean32, scale=sc.scale32, **kw)
        got = abi.route("STD, other statistics", ss, va, prep, abi.STD, True, mean=m2, scale=s2, **kw)
        check_oracle(got, seqs, va, items[:3], range(len(va)), seed, seq_id0, mean=m2, scale=s2)


# ---------------------------------------------------------------- output layouts
def test_output_layouts(abi, base):
    """x_train's interleaved [pairs, 2, F] layout and a base offset by 16 bytes take the fast route and equal the [V, n, F]
    rows.  Every kernel writes these rows as 16-byte vectors, so a base offset by 4 bytes or an out_off of 2 elements is
    refused before anything is launched (the generic kernel cannot take such rows either)"""
    ft = abi.ft
    seqs, ss = base
    va = schedule(ft, n_randn=2)
    S, n = len(va), ss.n
    prep = abi.prepare(ss, va, seed=4)
    sc = prep.scaler
    kw = dict(seed=4, mean=sc.mean32, scale=sc.scale32)
    want = abi.route("[V, n, F]", ss, va, prep, abi.STD, True, **kw)
    check_oracle(want, seqs, va, sample_items(n, np.random.default_rng(1)), range(S), 4, scaler=sc)
    sentinel = -12345.0
    # x_train of AugmentFasta: pair j*n + w = (slot 0 of w, slot j + 1 of w), rows of 2F floats
    x = torch.full(((S - 1) * n, 2, F), sentinel, device=abi.dev)
    offs = [0] + [((j * n) * 2 + 1) * F for j in range(S - 1)]
    _, fast, n_def = abi.prepared(ss, va, prep, abi.STD, out=x, out_off=offs, out_stride=2 * F, **kw)
    same(x[:n, 0], want[0], "x_train slot 0")
    for j in range(S - 1):
        same(x[j * n:(j + 1) * n, 1], want[j + 1], "x_train slot %d" % (j + 1))
    assert bool((x[n:, 0] == sentinel).all()), "x_train: rows outside the layout were written"
    assert fast and n_def == prep.flagged, ("x_train layout route", fast, n_def)
    total = S * n * F
    buf = torch.full((total + 8,), sentinel, device=abi.dev)
    _, fast, n_def = abi.prepared(ss, va, prep, abi.STD, out=buf[4:], out_off=[s * n * F for s in range(S)], **kw)
    same(buf[4:4 + total].view(S, n, F), want, "base + 16 bytes")
    assert fast and n_def == prep.flagged, ("base + 16 bytes route", fast, n_def)
    assert bool((buf[:4] == sentinel).all()) and bool((buf[4 + total:] == sentinel).all()), "base + 16 bytes: rows outside the layout were written"
    for shift, off in ((1, 0), (0, 2)):                             # base offset (elements), out_off offset (elements)
        buf = torch.full((total + 8,), sentinel, device=abi.dev)
        offs = [off + s * n * F for s in range(S)]
        l0 = abi.lib.idl_launch_count()
        with pytest.raises(abi.L.IdelucsB200Error, match="d_out must be 16-byte aligned and out_off multiples of 4"):
            abi.prepared(ss, va, prep, abi.STD, out=buf[shift:], out_off=offs, **kw)
        with pytest.raises(abi.L.IdelucsB200Error, match="d_out must be 16-byte aligned and out_off multiples of 4"):
            ft.profiles(ss, 6, va, out_kind=abi.STD, seed=4, mean=sc.mean32, scale=sc.scale32, out=buf[shift:], out_off=offs, out_stride=F)
        assert abi.lib.idl_launch_count() == l0 and bool((buf == sentinel).all()), (shift, off)


# ---------------------------------------------------------------- capacity edges
def test_item_count_edge(abi):
    """the fast kernel needs n_items >= 2 x SMs"""
    ft = abi.ft
    rng = np.random.default_rng(2)
    n = 2 * abi.sm
    seqs = random_seqs(rng, rng.integers(100, 3000, size=n))
    ss = abi.SeqSet.from_sequences(seqs)
    va = schedule(ft, n_randn=2)
    for m, fast in ((n, True), (n - 1, False)):
        prep = abi.prepare(ss, va, n=m, seed=12)
        got = abi.route("n_items = %d" % m, ss, va, prep, abi.FREQ, fast, n=m, seed=12, want=abi.generic(ss, va, abi.FREQ, seed=12)[:, :m])
        check_oracle(got, seqs, va, [0, m - 1], range(len(va)), 12)


def test_slot_and_bernoulli_edges(abi, base):
    """64 slots with Bernoulli slots at 0 / 17 / 63 and 4 distinct rates (fast route); 65 slots or a fourth Bernoulli slot
    take the fallback, and idl_profiles_prepare refuses the fourth Bernoulli slot"""
    ft = abi.ft
    seqs, ss = base
    v64 = [V(ft, ft.KIND_RANDOM_N if i % 3 else ft.KIND_CLEAN, n_bp=(i % 7) * 2, rng_id=100 + i) for i in range(64)]
    v64[0] = V(ft, ft.KIND_BOTH, 1.1e-2, 0.4e-2, rng_id=0)
    v64[17] = V(ft, ft.KIND_TRANSITION, p1=2e-2, rng_id=17)
    v64[63] = V(ft, ft.KIND_TRANSVERSION, p2=0.7e-2, rng_id=63)
    assert sum(v.n_bp for v in v64) <= 981
    prep = abi.prepare(ss, v64, seed=21)
    got = abi.route("64 slots", ss, v64, prep, abi.FREQ, True, seed=21)
    check_oracle(got, seqs, v64, [0, ss.n - 1, 401], [0, 1, 2, 17, 62, 63], 21)
    v65 = v64 + [V(ft, ft.KIND_RANDOM_N, n_bp=3, rng_id=64)]
    abi.route("65 slots", ss, v65, prep, abi.FREQ, False, seed=21)
    v4b = list(v64)
    v4b[30] = V(ft, ft.KIND_TRANSITION, p1=1.1e-2, rng_id=30)
    with pytest.raises(abi.L.IdelucsB200Error, match="at most 3 Bernoulli slots"):
        abi.prepare(ss, v4b, seed=21)
    abi.route("4 Bernoulli slots", ss, v4b, prep, abi.FREQ, False, seed=21)


@pytest.mark.parametrize("limit,value,fast", [("n_bp", 21, True), ("n_bp", 22, False), ("draws", 981, True), ("draws", 982, False)])
def test_random_n_edges(abi, base, limit, value, fast):
    """a Random_N slot removes at most 21 x 6 = 126 windows on the fast route, and one sequence's draws fill at most
    PC_REM / 6 = 981 removal lists"""
    ft = abi.ft
    seqs, ss = base
    va = [V(ft, ft.KIND_CLEAN, rng_id=0), V(ft, ft.KIND_BOTH, 1e-2, 0.5e-2, rng_id=1)]
    if limit == "n_bp":
        va += [V(ft, ft.KIND_RANDOM_N, n_bp=value, rng_id=2 + i) for i in range(3)]
    else:
        va += [V(ft, ft.KIND_RANDOM_N, n_bp=21, rng_id=2 + i) for i in range(46)] + [V(ft, ft.KIND_RANDOM_N, n_bp=value - 46 * 21, rng_id=48)]
    prep = abi.prepare(ss, va, seed=31, seq_id0=2)
    sc = prep.scaler
    got = abi.route("%s = %d" % (limit, value), ss, va, prep, abi.STD, fast, seed=31, seq_id0=2, mean=sc.mean32, scale=sc.scale32)
    check_oracle(got, seqs, va, [0, ss.n - 1, 5], [0, 1, 2, len(va) - 1], 31, 2, scaler=sc)


def test_length_edges_and_shared_window_totals(abi):
    """20 480 bases (the longest item the fast kernels stage) and 20 481 (flagged), empty and shorter than k, chunk
    boundaries, all-N and N-rich items; slot 0 Random_N(0), a clean slot and another Random_N(0) share window totals"""
    ft = abi.ft
    rng = np.random.default_rng(13)
    edge = [MAX_LEN, MAX_LEN + 1, 0, 1, 2, 3, 4, 5, 63, 64, 65]
    seqs = random_seqs(rng, edge, ACGT)
    seqs += [b"N" * 500, ALPH[np.r_[rng.integers(0, 24, size=1500), np.full(1500, 24)][rng.permutation(3000)]].tobytes()]
    n_edge = len(seqs)
    seqs += random_seqs(rng, rng.integers(100, 4000, size=2 * abi.sm))
    ss = abi.SeqSet.from_sequences(seqs)
    va = [V(ft, ft.KIND_RANDOM_N, n_bp=0, rng_id=0), V(ft, ft.KIND_TRANSITION, p1=1e-2, rng_id=1), V(ft, ft.KIND_CLEAN, rng_id=2),
          V(ft, ft.KIND_RANDOM_N, n_bp=0, rng_id=3), V(ft, ft.KIND_RANDOM_N, n_bp=20, rng_id=4), V(ft, ft.KIND_TRANSVERSION, p2=0.5e-2, rng_id=5)]
    prep = abi.prepare(ss, va, seed=41, seq_id0=9)
    assert prep.flag_mask.tolist() == [len(s) > MAX_LEN for s in seqs], np.nonzero(prep.flag_mask)[0]
    sc = prep.scaler
    f = abi.route("lengths, FREQ", ss, va, prep, abi.FREQ, True, seed=41, seq_id0=9)
    s = abi.route("lengths, STD", ss, va, prep, abi.STD, True, seed=41, seq_id0=9, mean=sc.mean32, scale=sc.scale32)
    items = list(range(n_edge)) + [ss.n - 1]
    check_oracle(f, seqs, va, items, range(len(va)), 41, 9)
    check_oracle(s, seqs, va, items, range(len(va)), 41, 9, scaler=sc)


# ---------------------------------------------------------------- contracts
@pytest.mark.parametrize("pc", [0, 3])
@pytest.mark.parametrize("want_stats", [True, False])
def test_pseudocounts_and_statistics_free_prepare(abi, pc, want_stats):
    """pseudocounts 0 (colstats16_kernel<false>) and 3; prepare without statistics keeps the flagged items in the buffer
    alone (d_status is cleared): prepared must still defer exactly those.  Every item keeps valid windows in every slot,
    so no frequency is 0 / 0 under pseudocount 0."""
    ft = abi.ft
    rng = np.random.default_rng(17 + pc)
    lens = rng.integers(400, 8000, size=2 * abi.sm + 50)
    lens[[1, 200]] = [MAX_LEN + 1, 26000]
    seqs = random_seqs(rng, lens)
    ss = abi.SeqSet.from_sequences(seqs)
    va = schedule(ft, n_randn=3)
    prep = abi.prepare(ss, va, seed=51, seq_id0=4, pc=pc, stats=want_stats)
    assert prep.flag_mask[[1, 200]].all()
    g = ft.profile_stats(ss, 6, va[0], seed=51, seq_id0=4, pseudocount=pc, fast=False)
    if want_stats:
        a = prep.scaler
        assert torch.allclose(g.mean64, a.mean64, rtol=1e-13, atol=0) and torch.allclose(g.scale64, a.scale64, rtol=1e-9, atol=0)
        nz = g.mean32 != 0
        assert float(((g.mean32 - a.mean32).abs()[nz] / g.mean32.abs()[nz]).max()) < 2e-7 and torch.equal(a.mean32[~nz], g.mean32[~nz])
    assert_normal_scale(g.scale32)
    kw = dict(seed=51, seq_id0=4, pc=pc)
    f = abi.route("pseudocount %d, FREQ" % pc, ss, va, prep, abi.FREQ, True, **kw)
    s = abi.route("pseudocount %d, STD" % pc, ss, va, prep, abi.STD, True, mean=g.mean32, scale=g.scale32, **kw)
    items = [0, 1, 200, ss.n - 1]
    check_oracle(f, seqs, va, items, [0, 1, 2, 3, 6], 51, 4, pc=pc)
    check_oracle(s, seqs, va, items[:2], [0, 1, 2, 3, 6], 51, 4, pc=pc, scaler=g)


# ---------------------------------------------------------------- standardisation arithmetic
def assert_normal_scale(scale32):
    s = scale32.double()
    assert bool(torch.isfinite(s).all()) and float(s.min()) >= 2.0 ** -126, "scale32 outside the finite normal floats: %g" % float(s.min())


def test_standardisation_is_ieee_division(abi, base):
    """(x - mean32) / scale32 on both routes equals IEEE float32 arithmetic (numpy) bit for bit for hand-made statistics:
    scale 1 and powers of two, scales from 1e-30 to 1e30, mean 0, a mean above every frequency, a mean equal to a row's
    value (exact zeros), and a mean one ulp above a row's value with scale 1e30 (subnormal quotients).  The kernels require
    a finite, normal scale32."""
    ft = abi.ft
    seqs, ss = base
    va = schedule(ft, n_randn=2)
    prep = abi.prepare(ss, va, seed=61)
    x = abi.generic(ss, va, abi.FREQ, seed=61)
    check_oracle(x, seqs, va, [0, ss.n - 1], range(len(va)), 61)
    xn = x.cpu().numpy()
    rng = np.random.default_rng(8)
    col = np.arange(F) % 8
    mean = np.zeros(F, np.float32)
    scale = np.ones(F, np.float32)

    def logu(lo, hi, m):
        return (10.0 ** rng.uniform(lo, hi, size=m)).astype(np.float32)

    g = col == 1; scale[g] = np.ldexp(1.0, rng.integers(-20, 21, size=g.sum())).astype(np.float32); mean[g] = rng.uniform(0, 1e-3, g.sum())
    g = col == 2; scale[g] = logu(-30, 0, g.sum()); mean[g] = rng.uniform(0, 1e-3, g.sum())
    g = col == 3; scale[g] = logu(0, 30, g.sum()); mean[g] = 2.0                       # above every frequency
    g = col == 4; scale[g] = logu(-30, 30, g.sum()); mean[g] = -1.0
    g = col == 5; scale[g] = logu(-3, 0, g.sum()); mean[g] = xn[0, 7][g]                # row 7 of slot 0: exact zeros
    g = col == 6; scale[g] = logu(-30, -10, g.sum())
    g = col == 7; scale[g] = prep.scaler.scale32.cpu().numpy()[g]; mean[g] = prep.scaler.mean32.cpu().numpy()[g]
    g = col == 0; scale[g] = 1e30; mean[g] = np.nextafter(xn[0, 9][g], np.float32(1))   # row 9 of slot 0: subnormal quotients
    want = (xn - mean) / scale
    a = np.abs(want)
    assert np.isfinite(want).all() and (a[..., col != 0][a[..., col != 0] != 0] >= np.float32(2.0 ** -126)).all()
    assert ((a[0, 9][col == 0] < np.float32(2.0 ** -126)) & (a[0, 9][col == 0] > 0)).all()
    assert (want[0, 7][col == 5] == 0).all()
    m, s = torch.from_numpy(mean).to(abi.dev), torch.from_numpy(scale).to(abi.dev)
    want_t = torch.from_numpy(want).to(abi.dev)
    same(abi.generic(ss, va, abi.STD, seed=61, mean=m, scale=s), want_t, "generic STD vs IEEE")
    abi.route("fast STD vs IEEE", ss, va, prep, abi.STD, True, want=want_t, seed=61, mean=m, scale=s)


def test_scaler_emits_finite_normal_scales_on_pathological_columns(abi):
    """idl_scaler_finalize (sklearn's near-constant rule: scale 1) never emits a zero, subnormal or infinite scale32 for
    frequency columns: constant, near-constant, all zero (pseudocount 0), one non-zero row with the smallest frequency a
    sequence shorter than 2^31 bases can have, a single row"""
    ft = abi.ft
    n = 5000
    f0 = np.float32(1.0 / 24576)
    cols = [np.full(n, 0.25), np.r_[np.full(n - 1, 0.25), np.nextafter(np.float32(0.25), np.float32(1))], np.zeros(n),
            np.r_[np.zeros(n - 1), 1.0 / 20480], np.full(n, f0), np.r_[np.full(n - 1, f0), np.nextafter(f0, np.float32(1))],
            np.r_[np.zeros(n - 1), 1.0 / (2 ** 31 - 1)], np.random.default_rng(1).random(n) * 1e-3]
    X = np.stack(cols, axis=1).astype(np.float32)
    for m in (X, X[:1], X[:2]):
        sc = ft.Scaler.fit(torch.from_numpy(np.ascontiguousarray(m)).to(abi.dev))
        assert_normal_scale(sc.scale32)
        assert float(sc.scale32[0]) == 1.0 and float(sc.scale32[2]) == 1.0
