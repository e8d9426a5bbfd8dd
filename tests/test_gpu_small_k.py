"""GPU tests at small k (-m gpu): the k = 1, 2, 3 instantiations of the generic profile kernel (2 warps, two private
copies so a half-group holds one slot, partial granule loops) and the canonical k-mer path of --model_size small at every
k = 1..6, against the oracle's mutate-and-recount (idelucs/kmers.pyx:38-50 on the mutated bytes), its FCGR loop
(kmers.pyx:53-123), its canonical folding (idelucs/utils.py:208-221, 246-250) and sklearn's StandardScaler arithmetic
(utils.py:358-366)."""
import os

import numpy as np
import pytest

import idelucs_oracle as orc

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

SMALL_K = [1, 2, 3]
ALL_K = [1, 2, 3, 4, 5, 6]
# 20 480 = SSEQ_CHUNKS x 64 (the last length staged in shared memory); 65 535 the last length of the uint16 short path
LENGTHS = (0, 1, 63, 64, 65, 127, 128, 129, 4099, 20480, 20481, 65535, 65536, 70001)


@pytest.fixture(scope="module")
def ft():
    from idelucs_b200 import featurise
    return featurise


@pytest.fixture(scope="module")
def SeqSet():
    from idelucs_b200.seqset import SeqSet
    return SeqSet


def _rand_seq(rng, L, n_rate=0.002):
    """random ACGT bytes with scattered Ns and, from 64 bases on, N runs (scaffold gaps)"""
    a = np.frombuffer(b"ACGT", dtype=np.uint8)[rng.integers(0, 4, size=L)].copy()
    if n_rate > 0 and L > 0:
        a[rng.random(L) < n_rate] = ord("N")
        for _ in range(min(3, L // 64)):
            p = int(rng.integers(0, L))
            a[p:p + int(rng.integers(1, min(200, L // 8) + 1))] = ord("N")
    return a.tobytes()


def _oracle_counts(seqs, k, seed, variants, seq_id0=0, explicit=None):
    """[V, N, 4^k] int32: apply the variant's edits (rng mode: the oracle's specification of the counter-based RNG;
    explicit: the given lists) to a copy of the bytes and recount from scratch."""
    out = np.zeros((len(variants), len(seqs), 4 ** k), np.int32)
    for i, s in enumerate(seqs):
        codes = orc.codes_of_seq(s)
        for v, spec in enumerate(variants):
            if spec.kind == 5:
                pos, val = explicit[spec.explicit_idx][i]
                edits = list(zip(np.asarray(pos).tolist(), np.asarray(val).tolist()))
            else:
                rid = spec.rng_id if spec.rng_id is not None else v
                edits = orc.rng_variant_edits(seed, seq_id0 + i, rid, spec.kind, codes, len(s), spec.p1, spec.p2, spec.n_bp)
            mut = bytearray(s)
            for p, val in edits:
                mut[p] = b"ACGTN"[val]
            orc.kmer_counts(mut, k, out[v, i])
    return out


def _check_all_outputs(ft, ss, seqs, k, variants, seed, seq_id0, lists=None, explicit=None, **kw):
    want = _oracle_counts(seqs, k, seed, variants, seq_id0, explicit)
    got = ft.profiles(ss, k, variants, out_kind=ft.OUT_COUNTS_I32, seed=seed, seq_id0=seq_id0, edit_lists=lists, **kw).cpu().numpy()
    bad = np.argwhere((got != want).any(axis=2))
    assert bad.size == 0, ("counts differ (variant, sequence):", bad[:10].tolist(), [len(s) for s in seqs])
    w64 = (want + 1) / (want + 1).sum(axis=2, keepdims=True)           # utils.py:242-250
    f64 = ft.profiles(ss, k, variants, out_kind=ft.OUT_FREQ_F64, seed=seed, seq_id0=seq_id0, edit_lists=lists, **kw).cpu().numpy()
    assert np.array_equal(f64, w64)
    w32 = w64.astype(np.float32)                                       # utils.py:353
    f32 = ft.profiles(ss, k, variants, out_kind=ft.OUT_FREQ_F32, seed=seed, seq_id0=seq_id0, edit_lists=lists, **kw).cpu().numpy()
    assert np.array_equal(f32, w32)
    mean, var, scale = orc.standard_scaler_fit(w32[0])                 # utils.py:358-359 (sklearn arithmetic)
    m32, s32 = mean.astype(np.float32), scale.astype(np.float32)
    std = ft.profiles(ss, k, variants, out_kind=ft.OUT_STD_F32, seed=seed, seq_id0=seq_id0, edit_lists=lists,
                      mean=torch.from_numpy(m32).cuda(), scale=torch.from_numpy(s32).cuda(), **kw).cpu().numpy()
    wstd = orc.standard_scaler_transform(w32.reshape(-1, 4 ** k), mean, scale).reshape(w32.shape)   # utils.py:361-366
    assert np.array_equal(std, wstd)
    return want


def _explicit_lists(rng, seqs):
    """one explicit list per sequence: substitutions and Ns, scattered and clustered, including the first and last base"""
    lists = []
    for s in seqs:
        L = len(s)
        if L == 0:
            lists.append((np.zeros(0, np.int64), np.zeros(0, np.int64)))
            continue
        pos = np.concatenate([rng.integers(0, L, size=min(L, 200)), np.arange(0, min(L, 30), 3), [0, L - 1, L // 2, L // 2 + 1]])
        pos = np.unique(pos[pos < L])
        lists.append((pos, rng.integers(0, 5, size=pos.size)))
    return lists


def _all_kinds(ft):
    variants = [ft.VariantSpec(ft.KIND_CLEAN), ft.VariantSpec(ft.KIND_TRANSITION, p1=1e-2), ft.VariantSpec(ft.KIND_TRANSVERSION, p2=0.5e-2),
                ft.VariantSpec(ft.KIND_BOTH, 1e-2, 0.5e-2), ft.VariantSpec(ft.KIND_RANDOM_N, n_bp=20),
                ft.VariantSpec(ft.KIND_RANDOM_N, n_bp=333), ft.VariantSpec(ft.KIND_EXPLICIT, explicit_idx=0)]
    for i, v in enumerate(variants):
        v.rng_id = i
    return variants


SEED = 0x5EED00AB12


@pytest.mark.parametrize("k", SMALL_K)
def test_small_k_every_variant_and_output_kind_vs_oracle(ft, SeqSet, k):
    """every variant kind x every output kind at the lengths where the kernel changes paths: empty, shorter than a window,
    one word of packed bases either side, the shared-memory staging limit, the last uint16 short-path length and the
    int32 long path; plus a homopolymer whose single k = 1 bin holds 65 535, the ceiling of the uint16 private copies"""
    rng = np.random.default_rng(300 + k)
    lens = sorted(set(LENGTHS + (k - 1, k)))
    seqs = [_rand_seq(rng, L) for L in lens] + [b"A" * 65535, b"C" * 4099]
    ss = SeqSet.from_sequences(seqs)
    explicit = [_explicit_lists(rng, seqs)]
    lists = ft.pack_edit_lists(explicit, len(seqs), ss.device)
    want = _check_all_outputs(ft, ss, seqs, k, _all_kinds(ft), seed=SEED, seq_id0=17, lists=lists, explicit=explicit)
    hp = len(lens)
    assert want[0, hp, 0] == 65535 - (k - 1)                          # the homopolymer's bin really is at the ceiling
    assert (want[1:4, hp, 0] < want[0, hp, 0]).all()                   # and its Bernoulli mimics do mutate it


@pytest.mark.parametrize("k", SMALL_K)
def test_small_k_selection_accumulate_and_pair_layout(ft, SeqSet, k):
    """the call modes at small k: slot selection per item (sidx / sel, items on both sides of 65 535 bases) against the
    rows of the full call, accumulate into a pre-filled buffer, and the (true, mimic) pair layout through out_off /
    out_stride that AugmentFasta's rows use"""
    rng = np.random.default_rng(400 + k)
    lens = [70001, 65535, 129, 20481, 1, 3000, 65536, 64, 0, 777]
    seqs = [_rand_seq(rng, L) for L in lens]
    n = len(seqs)
    ss = SeqSet.from_sequences(seqs)
    explicit = [_explicit_lists(rng, seqs)]
    lists = ft.pack_edit_lists(explicit, n, ss.device)
    variants = _all_kinds(ft)
    V, F = len(variants), 4 ** k
    want = _oracle_counts(seqs, k, SEED, variants, 3, explicit)
    full = ft.profiles(ss, k, variants, out_kind=ft.OUT_COUNTS_I32, seed=SEED, seq_id0=3, edit_lists=lists).cpu().numpy()
    assert np.array_equal(full, want)
    # selection: item w is sequence sidx[w] with the slots sel[w]
    sidx = torch.tensor([0, 6, 1, 0, 9, 3, 8, 2, 5, 6, 4], dtype=torch.int32, device="cuda")
    sel = torch.from_numpy(np.stack([np.zeros(sidx.numel(), np.int32), rng.integers(1, V, size=sidx.numel()).astype(np.int32)], 1)).cuda()
    sel[3] = torch.tensor([6, 5], dtype=torch.int32)
    got = ft.profiles(ss, k, variants, out_kind=ft.OUT_COUNTS_I32, seed=SEED, seq_id0=3, edit_lists=lists, sidx=sidx, sel=sel).cpu().numpy()
    for w in range(sidx.numel()):
        for s in range(2):
            assert np.array_equal(got[s, w], want[int(sel[w, s]), int(sidx[w])]), (w, s)
    f32_full = ft.profiles(ss, k, variants, out_kind=ft.OUT_FREQ_F32, seed=SEED, seq_id0=3, edit_lists=lists)
    f32_sel = ft.profiles(ss, k, variants, out_kind=ft.OUT_FREQ_F32, seed=SEED, seq_id0=3, edit_lists=lists, sidx=sidx, sel=sel)
    assert torch.equal(f32_sel, f32_full[sel.long().t(), sidx.long().unsqueeze(0)])
    # accumulate: the counts are added to what the buffer holds
    pattern = torch.from_numpy(rng.integers(-1000, 1000, size=(V, n, F)).astype(np.int32)).cuda()
    acc = pattern.clone()
    ft.profiles(ss, k, variants, out_kind=ft.OUT_COUNTS_I32, seed=SEED, seq_id0=3, edit_lists=lists, out=acc,
                out_off=[v * n * F for v in range(V)], out_stride=F, accumulate=True)
    assert np.array_equal(acc.cpu().numpy(), pattern.cpu().numpy() + want)
    # pair layout: row (j*n + i) = (slot 0 of item i, slot j+1 of item i); the 'true' column of mimics j > 0 is not written
    sc = ft.Scaler.fit(f32_full[0])
    std_full = ft.profiles(ss, k, variants, out_kind=ft.OUT_STD_F32, seed=SEED, seq_id0=3, edit_lists=lists, mean=sc.mean32, scale=sc.scale32)
    x = torch.full(((V - 1) * n, 2, F), float("nan"), dtype=torch.float32, device="cuda")
    offs = [0] + [((j * n) * 2 + 1) * F for j in range(V - 1)]
    ft.profiles(ss, k, variants, out_kind=ft.OUT_STD_F32, seed=SEED, seq_id0=3, edit_lists=lists, mean=sc.mean32, scale=sc.scale32,
                out=x, out_off=offs, out_stride=2 * F)
    assert torch.equal(x[:n, 0], std_full[0])
    assert torch.equal(x[:, 1].reshape(V - 1, n, F), std_full[1:])
    assert bool(x[n:, 0].isnan().all())


@pytest.mark.parametrize("k", SMALL_K)
def test_small_k_big_plan_and_high_rates_vs_oracle(ft, SeqSet, k):
    """a plan too big for the kernel parameter (70 variants > 64 cached descriptors, 8 distinct rates > 4 cached gap
    tables), more slots than one supergroup holds (and more Random_N draws than one supergroup buffers), and rates high
    enough on 20-70 kb sequences that one tile's edits overflow the 2 048-entry on-chip list: nothing may be dropped"""
    rng = np.random.default_rng(500 + k)
    seqs = [_rand_seq(rng, L) for L in (50000, 20000, 70000, 33000)]
    ss = SeqSet.from_sequences(seqs)
    variants = [ft.VariantSpec(ft.KIND_TRANSITION, p1=0.2), ft.VariantSpec(ft.KIND_BOTH, 0.1, 0.1), ft.VariantSpec(ft.KIND_TRANSVERSION, p2=0.6),
                ft.VariantSpec(ft.KIND_BOTH, 1.0, 0.0), ft.VariantSpec(ft.KIND_CLEAN), ft.VariantSpec(ft.KIND_BOTH, 1e-2, 0.5e-2),
                ft.VariantSpec(ft.KIND_TRANSVERSION, p2=0.03), ft.VariantSpec(ft.KIND_RANDOM_N, n_bp=333)]
    variants += [ft.VariantSpec(ft.KIND_RANDOM_N, n_bp=20) for _ in range(60)]
    variants += [ft.VariantSpec(ft.KIND_RANDOM_N, n_bp=7), ft.VariantSpec(ft.KIND_TRANSITION, p1=0.01)]
    for i, v in enumerate(variants):
        v.rng_id = i
    rates = {v.p1 for v in variants if v.kind in (1, 3)} | {v.p2 for v in variants if v.kind in (2, 3)}
    assert len(variants) > 64 and len(rates) >= 6
    _check_all_outputs(ft, ss, seqs, k, variants, seed=31337, seq_id0=0)


@pytest.mark.parametrize("k", SMALL_K)
def test_small_k_in_kernel_statistics_vs_oracle(ft, SeqSet, k):
    """profile_stats (the generic kernel's statistics mode: one part per CTA of the persistent grid, merged over many
    64-part chunks by scaler_finalize_kernel) against float64 numpy statistics of the oracle's float32 frequencies"""
    rng = np.random.default_rng(600 + k)
    seqs = [_rand_seq(rng, int(L), n_rate=0.01) for L in rng.integers(k, 200, size=3000)]
    ss = SeqSet.from_sequences(seqs)
    seed = 4242
    for spec in (ft.VariantSpec(ft.KIND_CLEAN, rng_id=0), ft.VariantSpec(ft.KIND_BOTH, 1e-2, 0.5e-2, rng_id=1),
                 ft.VariantSpec(ft.KIND_RANDOM_N, n_bp=20, rng_id=2)):
        want = _oracle_counts(seqs, k, seed, [spec], seq_id0=9)[0]
        w32 = ((want + 1) / (want + 1).sum(axis=1, keepdims=True)).astype(np.float32)
        x64 = w32.astype(np.float64)
        mean, var = x64.mean(axis=0), x64.var(axis=0)
        a = ft.profile_stats(ss, k, spec, seed=seed, seq_id0=9)
        np.testing.assert_allclose(a.mean64.cpu().numpy(), mean, rtol=1e-13, atol=0)
        np.testing.assert_allclose(a.var64.cpu().numpy(), var, rtol=1e-8, atol=1e-30)
        np.testing.assert_allclose(a.scale64.cpu().numpy(), np.sqrt(var), rtol=1e-8, atol=0)
        b = ft.profile_stats(ss, k, spec, seed=seed, seq_id0=9)
        for name in ("mean64", "var64", "scale64", "mean32", "scale32"):
            assert torch.equal(getattr(a, name), getattr(b, name)), name     # static rows per CTA: reproducible
        f32 = ft.profiles(ss, k, [spec], out_kind=ft.OUT_FREQ_F32, seed=seed, seq_id0=9)[0]
        assert np.array_equal(f32.cpu().numpy(), w32)
        c = ft.Scaler.fit(f32)
        np.testing.assert_allclose(a.mean64.cpu().numpy(), c.mean64.cpu().numpy(), rtol=1e-13, atol=0)
        np.testing.assert_allclose(a.var64.cpu().numpy(), c.var64.cpu().numpy(), rtol=1e-8, atol=1e-30)
    # every column constant (3 000 copies of one sequence): variance exactly 0, scale exactly 1
    one = _rand_seq(rng, 500)
    ssc = SeqSet.from_sequences([one] * 3000)
    want = np.zeros(4 ** k, np.int32)
    orc.kmer_counts(bytearray(one), k, want)
    w32 = ((want + 1) / (want + 1).sum()).astype(np.float32)
    s = ft.profile_stats(ssc, k, ft.VariantSpec(ft.KIND_CLEAN), seed=seed)
    assert np.array_equal(s.mean64.cpu().numpy(), w32.astype(np.float64))
    assert bool((s.var64 == 0).all()) and bool((s.scale64 == 1).all()) and bool((s.scale32 == 1).all())


def _canonical(k):
    return [m for m in range(4 ** k) if m <= orc.reverse_complement(m, k)]


@pytest.mark.parametrize("k", ALL_K)
def test_index_maps_vs_oracle(ft, SeqSet, k):
    """cgr_batch (plain and accumulating) and kmers.cgr against the oracle's FCGR loop; revcomp_fold + normalize_counts
    against kmer_rev_comp's in-place int32 semantics (odd pair sums truncate) and counts / np.sum(counts);
    idl_revcomp_canonical against the oracle's canonical list"""
    import idelucs_b200.kmers as km
    from idelucs_b200 import _lib
    rng = np.random.default_rng(700 + k)
    F = 4 ** k
    seqs = [_rand_seq(rng, int(L), n_rate=0.02) for L in (0, k, 63, 64, 65, 1000, 5000)]
    ss = SeqSet.from_sequences(seqs)
    counts = ft.kmer_counts_batch(ss, k)
    want = np.zeros((len(seqs), F), np.int32)
    for i, s in enumerate(seqs):
        orc.cgr(s, k, want[i])
    assert np.array_equal(ft.cgr_batch(counts, k).cpu().numpy(), want)
    pattern = rng.integers(-50, 50, size=(len(seqs), F)).astype(np.int32)
    acc = ft.cgr_batch(counts, k, cgr=torch.from_numpy(pattern).cuda())
    assert np.array_equal(acc.cpu().numpy(), pattern + want)
    raw = bytearray(rng.integers(60, 90, size=3000, dtype=np.uint8).tobytes())   # strict alphabet: every other byte resets
    a, b = np.full(F, 3, np.int32), np.full(F, 3, np.int32)
    km.cgr(raw, k, a)
    orc.cgr(raw, k, b)
    assert np.array_equal(a, b)
    # canonical list
    canon = _canonical(k)
    assert len(canon) == [2, 10, 32, 136, 512, 2080][k - 1]
    lib = _lib.load()
    assert lib.idl_revcomp_canonical(k, None) == len(canon)
    assert ft.canonical_index(k, ss.device).cpu().numpy().tolist() == canon
    # folding + normalisation: count rows of real sequences (+1) and random rows with large and odd pair sums
    rows = np.concatenate([counts.cpu().numpy() + 1, rng.integers(0, 1 << 20, size=(20, F)).astype(np.int32),
                           rng.integers(0, 3, size=(20, F)).astype(np.int32) + 1])
    fold_want = np.stack([orc.kmer_rev_comp(r.copy(), k) for r in rows])
    rc = np.array([orc.reverse_complement(m, k) for m in canon])
    assert ((rows[:, canon] + rows[:, rc]) % 2 == 1).any()              # the int truncation matters
    fold = ft.revcomp_fold(torch.from_numpy(rows).cuda(), k)
    assert np.array_equal(fold.cpu().numpy(), fold_want)
    f64, f32 = ft.normalize_counts(fold, want64=True, want32=True)
    w64 = fold_want / np.sum(fold_want, axis=1, keepdims=True)          # utils.py:250 on the int32 vector
    assert np.array_equal(f64.cpu().numpy(), w64)
    assert np.array_equal(f32.cpu().numpy(), w64.astype(np.float32))
    assert np.array_equal(ft.normalize_counts(fold).cpu().numpy(), w64)


def _write_fasta(path, seqs):
    with open(path, "wb") as fh:
        for i, s in enumerate(seqs):
            fh.write(b">seq%d\n" % i)
            for o in range(0, len(s), 70):
                fh.write(s[o:o + 70] + b"\n")


@pytest.mark.parametrize("k", ALL_K)
def test_canonical_path_end_to_end_vs_oracle(ft, SeqSet, k, tmp_path):
    """--model_size small's featurisation (AugmentFasta / PairBatchLoader / SequenceDataset with reduce=True) at every k:
    +1-pseudocount counts of every mimic -> kmer_rev_comp -> / sum -> float32 -> StandardScaler of the t_norm slot ->
    (x - mean32) / scale32.  At k = 1 and 2 the canonical width (2, 10 columns) is not a multiple of 4."""
    from idelucs_b200 import utils as U
    rng = np.random.default_rng(800 + k)
    seqs = [_rand_seq(rng, int(L), n_rate=0.005) for L in rng.integers(max(k, 30), 3000, size=24)]
    ss = SeqSet.from_sequences(seqs)
    n_mimics, seed = 3, 99991
    variants = ft.mimic_schedule(n_mimics)
    x, sc, _ = U.augment_device(ss, n_mimics, k=k, seed=seed, seq_id0=0, reduce=True)
    c = _oracle_counts(seqs, k, seed, variants) + 1
    fold = np.stack([np.stack([orc.kmer_rev_comp(r.copy(), k) for r in cv]) for cv in c])
    x32 = (fold / fold.sum(axis=2, keepdims=True)).astype(np.float32)
    R = x32.shape[2]
    mean, var, scale = orc.standard_scaler_fit(x32[0])
    np.testing.assert_allclose(sc.mean64.cpu().numpy(), mean, rtol=1e-13, atol=0)
    np.testing.assert_allclose(sc.var64.cpu().numpy(), var, rtol=1e-8, atol=1e-30)
    want = orc.standard_scaler_transform(x32.reshape(-1, R), sc.mean64.cpu().numpy(), sc.scale64.cpu().numpy()).reshape(x32.shape)
    got = x.cpu().numpy()
    assert got.shape == (n_mimics + 1, len(seqs), R) and got.dtype == np.float32
    assert np.array_equal(got, want)
    loader = U.PairBatchLoader(ss, n_mimics, k=k, seed=seed, reduce=True)
    assert torch.equal(loader.profiles, x)
    # SequenceDataset(reduce=True): clean float64 canonical profiles + their own float64 scaler (utils.py:400-405)
    path = str(tmp_path / "small_k.fas")
    _write_fasta(path, seqs)
    ds = U.SequenceDataset(path, k=k, reduce=True)
    _, ref = orc.kmersFasta(path, k=k, reduce=True)
    m, _, s = orc.standard_scaler_fit(ref)
    np.testing.assert_allclose(ds.kmers, (ref - m) / s, rtol=1e-9, atol=1e-9)
    assert tuple(ds.kmers32.shape) == (len(seqs), R)


@pytest.mark.parametrize("model_size,k", [("small", 2), ("linear", 3)])
def test_cli_small_k(golden_dir, fasta_files, tmp_path, monkeypatch, model_size, k):
    """the CLI end to end at small k: canonical 2-mers (10 features) for model_size 'small', plain 3-mers for 'linear'"""
    from idelucs_b200 import __main__ as cli
    monkeypatch.chdir(tmp_path)
    gt = os.path.join(golden_dir, "Actinopterygii_GT.tsv")
    args = dict(sequence_file=fasta_files["Actinopterygii"], GT_file=gt, n_clusters=3, k=k, n_mimics=3, batch_sz=256, optimizer="RMSprop",
                weight=0.25, lr=1e-3, scheduler="None", plot=False, n_epochs=2, n_voters=1, model_size=model_size)
    args["lambda"] = 2.8
    torch.manual_seed(0); np.random.seed(0)
    y = cli.run(args)
    assert np.asarray(y).shape == (113,)
    out = [os.path.join(dp, f) for dp, _, fs in os.walk(str(tmp_path)) for f in fs if f == "assignments.tsv"]
    assert len(out) == 1
    with open(out[0]) as fh:
        lines = fh.read().splitlines()
    assert lines[0].split("\t") == ["sequence_id", "assignment", "confidence_score"] and len(lines) == 1 + 113
