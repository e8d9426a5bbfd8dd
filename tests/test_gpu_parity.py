"""GPU parity tests (run with -m gpu on the B200): the CUDA path, called through the C ABI
(ctypes), against the CPU oracle on the same inputs and against the golden vectors that the
live reference produced (oracle/gen_golden.py).  Integer work must be bit-exact."""
import hashlib
import json
import os

import sys

import numpy as np
import pytest

import idelucs_oracle as orc

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


@pytest.fixture(scope="module")
def ft():
    from idelucs_b200 import featurise
    return featurise


@pytest.fixture(scope="module")
def SeqSet():
    from idelucs_b200.seqset import SeqSet
    return SeqSet


def _golden(golden_dir):
    with open(os.path.join(golden_dir, "golden.json")) as fh:
        return json.load(fh)


def test_kmer_count_kats(golden_dir, ft, SeqSet):
    with open(os.path.join(golden_dir, "kmer_kats.json")) as fh:
        kats = json.load(fh)
    for k in (1, 2, 3, 4, 5, 6):
        sub = [c for c in kats if c["k"] == k]
        if not sub:
            continue
        ss = SeqSet.from_sequences([bytes.fromhex(c["seq_hex"]) for c in sub], alphabet="strict")
        got = ft.kmer_counts_batch(ss, k).cpu().numpy()
        for i, c in enumerate(sub):
            want = np.zeros(4 ** k, np.int32)
            want[c["nz_idx"]] = c["nz_val"]
            assert np.array_equal(got[i], want), (k, i)


@pytest.mark.parametrize("stem", ["Influenza-A", "Actinopterygii"])
@pytest.mark.parametrize("k", [4, 5, 6])
def test_fasta_counts_and_frequencies(golden_dir, fasta_files, ft, SeqSet, stem, k):
    g = _golden(golden_dir)["files"][stem][f"k{k}"]
    ss = SeqSet.from_fasta(fasta_files[stem])
    assert ss.n == g["n"]
    counts = ft.kmer_counts_batch(ss, k).cpu().numpy()
    assert int(counts.sum()) == g["counts_sum"]
    assert counts[0, :8].tolist() == g["counts_row0"]
    assert sha(counts) == g["counts_sha256"]            # bit-exact vs idelucs.kmers.kmer_counts
    clean = [ft.VariantSpec(ft.KIND_CLEAN)]
    f64 = ft.profiles(ss, k, clean, out_kind=ft.OUT_FREQ_F64)[0].cpu().numpy()
    assert sha(f64) == g["freq64_sha256"]               # bit-exact vs idelucs.utils.kmersFasta
    f32 = ft.profiles(ss, k, clean, out_kind=ft.OUT_FREQ_F32)[0].cpu().numpy()
    assert sha(f32) == g["freq32_sha256"]               # == kmersFasta(...).astype(float32)
    # accumulate semantics of kmers.pyx (counts are added INTO the caller's buffer)
    acc = torch.ones((ss.n, 4 ** k), dtype=torch.int32, device="cuda")
    ft.kmer_counts_batch(ss, k, counts=acc)
    assert np.array_equal(acc.cpu().numpy(), counts + 1)


def test_strict_alphabet_random_bytes(ft, SeqSet):
    rng = np.random.default_rng(3)
    seqs = [rng.integers(0, 256, size=int(rng.integers(0, 700)), dtype=np.uint8).tobytes() for _ in range(64)]
    seqs += [b"", b"A", b"ACGTA", bytes(range(256)) * 3]
    ss = SeqSet.from_sequences(seqs, alphabet="strict")
    for k in (2, 5, 6):
        got = ft.kmer_counts_batch(ss, k).cpu().numpy()
        for i, s in enumerate(seqs):
            want = np.zeros(4 ** k, np.int32)
            orc.kmer_counts(bytearray(s), k, want)
            assert np.array_equal(got[i], want), (k, i)


def test_check_sequence_semantics(ft, SeqSet):
    seqs = [b"acgtuUswkmyrbdhvnSWKMYRBDHV-ACGTN" * 5, b"AC GT\tACGTAC\nGTACGT\rACGTTTGAC", b"", b"ACGTNNNNACGTACGTAC"]
    ss = SeqSet.from_sequences(seqs, names=["a", "b", "c", "d"])
    got = ft.kmer_counts_batch(ss, 3).cpu().numpy()
    for i, s in enumerate(seqs):
        want = np.zeros(64, np.int32)
        orc.kmer_counts(orc.check_sequence("x", bytearray(s)), 3, want)
        assert np.array_equal(got[i], want), i
    with pytest.raises(ValueError, match=r"Invalid DNA byte in sequence s2: 'X'"):
        SeqSet.from_sequences([b"ACGT", b"ACGTACGTACGTACGTACGTAXGT"], names=["s1", "s2"])
    with pytest.raises(ValueError, match="Bad character in sequence header"):
        SeqSet.from_sequences([b"ACGT"], names=[">s1"])
    with pytest.raises(ValueError, match="tab included in header"):
        SeqSet.from_sequences([b"ACGT"], names=["s\t1"])


@pytest.mark.parametrize("k", [4, 5, 6])
def test_rng_mimics_bit_exact_vs_oracle(fasta_files, ft, SeqSet, k):
    """every variant kind of the AugmentFasta schedule, rng mode: integer counts equal the
    oracle's mutate-and-recount, on real sequences, random ones with Ns, and edge lengths"""
    rng = np.random.default_rng(k)
    recs = orc.read_fasta(fasta_files["Influenza-A"])[:24] + orc.read_fasta(fasta_files["Actinopterygii"])[:3]
    seqs = [bytes(s) for _, s in recs]
    alph = np.frombuffer(b"ACGTACGTACGTACGTACGTN", dtype=np.uint8)
    seqs += [alph[rng.integers(0, alph.size, size=L)].tobytes() for L in (0, 1, 5, 6, 63, 64, 65, 127, 128, 129, 300, 4099)]
    ss = SeqSet.from_sequences(seqs)
    variants = ft.mimic_schedule(6)
    seed = 0xC0FFEE1234
    got = ft.profiles(ss, k, variants, out_kind=ft.OUT_COUNTS_I32, seed=seed, seq_id0=1000).cpu().numpy()
    want = orc.rng_mimic_counts([bytearray(s) for s in seqs], k, seed, [v.kind for v in variants], seq_id0=1000)
    assert got.shape == want.shape
    bad = np.argwhere((got != want).any(axis=2))
    assert bad.size == 0, bad[:10]
    # frequencies: float32(count+1 / sum) exactly
    f32 = ft.profiles(ss, k, variants, out_kind=ft.OUT_FREQ_F32, seed=seed, seq_id0=1000).cpu().numpy()
    w32 = ((want + 1) / (want + 1).sum(axis=2, keepdims=True)).astype(np.float32)
    assert np.array_equal(f32, w32)


def test_rng_high_rates_and_many_variants(ft, SeqSet):
    rng = np.random.default_rng(9)
    alph = np.frombuffer(b"ACGTACGTACGTN", dtype=np.uint8)
    seqs = [alph[rng.integers(0, alph.size, size=L)].tobytes() for L in (900, 257, 2000, 31)]
    ss = SeqSet.from_sequences(seqs)
    variants = [ft.VariantSpec(ft.KIND_BOTH, 0.3, 0.25), ft.VariantSpec(ft.KIND_TRANSITION, p1=0.9),
                ft.VariantSpec(ft.KIND_TRANSVERSION, p2=0.6), ft.VariantSpec(ft.KIND_CLEAN)]
    variants += [ft.VariantSpec(ft.KIND_RANDOM_N, n_bp=20) for _ in range(60)]
    variants += [ft.VariantSpec(ft.KIND_RANDOM_N, n_bp=7), ft.VariantSpec(ft.KIND_RANDOM_N, n_bp=333)]
    for i, v in enumerate(variants):
        v.rng_id = i
    got = ft.profiles(ss, 5, variants, out_kind=ft.OUT_COUNTS_I32, seed=77).cpu().numpy()
    for v, spec in enumerate(variants):
        for i, s in enumerate(seqs):
            edits = orc.rng_variant_edits(77, i, v, spec.kind, orc.codes_of_seq(s), len(s), spec.p1, spec.p2, spec.n_bp)
            mut = bytearray(s)
            for pos, val in edits:
                mut[pos] = b"ACGTN"[val]
            want = np.zeros(4 ** 5, np.int32)
            orc.kmer_counts(mut, 5, want)
            assert np.array_equal(got[v, i], want), (v, i)


@pytest.mark.parametrize("k", [4, 5, 6])
def test_augment_fasta_reference_mutations_bit_exact(golden_dir, fasta_files, ft, SeqSet, k):
    """The reference's own mutations (np.random.seed(0); random.seed(0)), exported as edit
    lists, through the explicit-list path + scaler + standardise == the reference's
    AugmentFasta output, bit for bit (sha256 of x_train)."""
    g = _golden(golden_dir)["files"]["Influenza-A"]["augment_seed0_nmimics3"]
    ed = np.load(os.path.join(golden_dir, "influenza_edits_seed0.npz"))
    ss = SeqSet.from_fasta(fasta_files["Influenza-A"])
    n, offs = ss.n, ed["offsets"]
    lut = np.full(256, 4, np.int64)
    for i, ch in enumerate(b"ACGT"):
        lut[ch] = i
    explicit = [[(ed["pos"][offs[p * n + i]:offs[p * n + i + 1]], lut[ed["newbyte"][offs[p * n + i]:offs[p * n + i + 1]]])
                 for i in range(n)] for p in range(4)]
    lists = ft.pack_edit_lists(explicit, n, ss.device)
    variants = [ft.VariantSpec(ft.KIND_EXPLICIT, explicit_idx=p) for p in range(4)]
    F = 4 ** k
    t_norm = ft.profiles(ss, k, variants[:1], out_kind=ft.OUT_FREQ_F32, edit_lists=lists)[0]
    sc = ft.Scaler.fit(t_norm)
    x = torch.empty((3 * n, 2, F), dtype=torch.float32, device=ss.device)
    # row (j*n + i): column 0 = t_norm_i, column 1 = mimic_{j+1,i}   (utils.py:338-353, mimic-major)
    offs_out = [0] + [((j * n) * 2 + 1) * F for j in range(3)]
    ft.profiles(ss, k, variants, out_kind=ft.OUT_STD_F32, edit_lists=lists, mean=sc.mean32, scale=sc.scale32,
                out=x, out_off=offs_out, out_stride=2 * F)
    x[n:2 * n, 0] = x[:n, 0]
    x[2 * n:, 0] = x[:n, 0]
    xh = x.cpu().numpy()
    rows = np.load(os.path.join(golden_dir, f"influenza_xtrain_rows_k{k}.npz"))
    assert np.array_equal(xh[rows["rows"]], rows["x"])
    assert sha(xh) == g[f"k{k}"]["x_train_sha256"]


@pytest.mark.parametrize("stem", ["Influenza-A", "Actinopterygii"])
def test_inference_profiles_bit_exact(golden_dir, fasta_files, ft, SeqSet, stem):
    """SequenceDataset (utils.py:400-405): clean float64 profiles + own float64 scaler"""
    g = _golden(golden_dir)["files"][stem]["inference_k6"]
    ss = SeqSet.from_fasta(fasta_files[stem])
    f64 = ft.profiles(ss, 6, [ft.VariantSpec(ft.KIND_CLEAN)], out_kind=ft.OUT_FREQ_F64)[0]
    sc = ft.Scaler.fit(f64)
    x = sc.transform64(f64).cpu().numpy()
    rows = np.load(os.path.join(golden_dir, f"{stem}_inference_rows_k6.npz"))
    np.testing.assert_allclose(x[rows["rows"]], rows["x"], rtol=1e-9, atol=1e-9)
    # float64 statistics are merged in a different order than numpy's pairwise sum: the
    # standardised values agree to ~1e-12 relative (far inside the float32 cast of models.py:163)
    want = np.asarray(orc.inference_profiles(fasta_files[stem], 6)[1])
    np.testing.assert_allclose(x, want, rtol=1e-10, atol=1e-10)
    assert sha(f64.cpu().numpy()) == _golden(golden_dir)["files"][stem]["k6"]["freq64_sha256"]
    x32 = sc.transform64(f64, want32=True).cpu().numpy()
    np.testing.assert_allclose(x32, x.astype(np.float32), rtol=1e-6, atol=1e-6)


def test_scaler_matches_oracle(ft):
    rng = np.random.default_rng(4)
    X = (rng.random((5000, 256)) * 1e-3).astype(np.float32)
    X[:, 3] = X[0, 3]
    X[:, 5] = 0.0
    X[:, 7] = 1.0 + X[:, 7] * 1e-4
    sc = ft.Scaler.fit(torch.from_numpy(X).cuda())
    mean, var, scale = orc.standard_scaler_fit(X)
    np.testing.assert_allclose(sc.mean64.cpu().numpy(), mean, rtol=1e-13)
    np.testing.assert_allclose(sc.var64.cpu().numpy(), var, rtol=1e-9, atol=1e-30)
    assert sc.scale64[3].item() == 1.0 and sc.scale64[5].item() == 1.0
    np.testing.assert_allclose(sc.scale64.cpu().numpy(), scale, rtol=1e-9)
    got = sc.transform32(torch.from_numpy(X).cuda().clone()).cpu().numpy()
    want = orc.standard_scaler_transform(X, mean, scale)
    assert (got != want).mean() < 1e-3
    np.testing.assert_allclose(got, want, rtol=2e-6, atol=1e-6)


def test_selection_mode_equals_full_mode(ft, SeqSet):
    """pair batches (sidx/sel) regenerate exactly the rows of the full featurisation"""
    rng = np.random.default_rng(12)
    seqs = [np.frombuffer(b"ACGT", dtype=np.uint8)[rng.integers(0, 4, size=int(rng.integers(200, 3000)))].tobytes() for _ in range(40)]
    ss = SeqSet.from_sequences(seqs)
    variants = ft.mimic_schedule(8)
    full = ft.profiles(ss, 6, variants, out_kind=ft.OUT_FREQ_F32, seed=5)
    B = 64
    sidx = torch.from_numpy(rng.integers(0, 40, size=B).astype(np.int32)).cuda()
    mim = torch.from_numpy(rng.integers(1, 9, size=B).astype(np.int32)).cuda()
    sel = torch.stack([torch.zeros_like(mim), mim], dim=1).contiguous()
    out = ft.profiles(ss, 6, variants, out_kind=ft.OUT_FREQ_F32, seed=5, sidx=sidx, sel=sel)
    assert out.shape == (2, B, 4096)
    assert torch.equal(out[0], full[0][sidx.long()])
    assert torch.equal(out[1], full[mim.long(), sidx.long()])


def test_full_size_properties(ft, SeqSet):
    """BASELINE config 3 shape (10 kb sequences, k=6, n_mimics=50) on a slab: size-independent
    properties — window-count conservation, unit row sums, determinism, N-mimic bounds."""
    rng = np.random.default_rng(1)
    n, L, k, n_mimics = 512, 10000, 6, 50
    flat = np.frombuffer(b"ACGT", dtype=np.uint8)[rng.integers(0, 4, size=n * L)]
    ss = SeqSet.from_ascii(flat, np.arange(n + 1, dtype=np.int64) * L)
    variants = [ft.VariantSpec(ft.KIND_CLEAN)] + ft.mimic_schedule(n_mimics)
    for i, v in enumerate(variants):
        v.rng_id = i
    c = ft.profiles(ss, k, variants, out_kind=ft.OUT_COUNTS_I32, seed=3)
    tot = c.sum(dim=2)
    assert bool((tot[0] == L - k + 1).all())                       # clean: every window counted
    assert bool((tot[1:4] == L - k + 1).all())                     # substitutions keep every window
    assert bool((tot[4:] <= L - k + 1).all()) and bool((tot[4:] >= L - k + 1 - 20 * k).all())
    assert bool((c >= 0).all())
    assert bool(((c[4:] - c[0:1]) <= 0).all())                     # Random_N only removes windows
    c2 = ft.profiles(ss, k, variants, out_kind=ft.OUT_COUNTS_I32, seed=3)
    assert torch.equal(c, c2)                                      # counter-based RNG: deterministic
    f = ft.profiles(ss, k, variants, out_kind=ft.OUT_FREQ_F32, seed=3)
    assert float((f.double().sum(dim=2) - 1).abs().max()) < 1e-5
    c3 = ft.profiles(ss, k, variants, out_kind=ft.OUT_COUNTS_I32, seed=4)
    assert not torch.equal(c[1], c3[1])
    # each of the ~L*(1-(1-p1)(1-p2)) edits of pass 0 moves k windows from one bin to another:
    # L1 distance of the histograms ~ 2k per edit, minus remove/add collisions in the same bin
    dist_both = (c[1] - c[0]).abs().sum(dim=1).double().mean().item() / (2 * k)
    assert 0.6 * L * 0.015 < dist_both < 1.02 * L * 0.015, dist_both


def _loss_inputs(B, C, salt):
    import gen_golden
    return gen_golden.loss_inputs(B, C, salt)


def test_iid_loss_goldens(golden_dir):
    from idelucs_b200.LossFunctions import IID_loss, compute_joint
    with open(os.path.join(golden_dir, "iid_loss.json")) as fh:
        cases = json.load(fh)
    for c in cases:
        z1n, z2n = _loss_inputs(c["B"], c["C"], c["salt"]), _loss_inputs(c["B"], c["C"], c["salt"] + 100)
        z1 = torch.from_numpy(z1n).cuda().requires_grad_(True)
        z2 = torch.from_numpy(z2n).cuda().requires_grad_(True)
        loss = IID_loss(z1, z2, lamb=c["lamb"])
        loss.backward()
        assert abs(loss.item() - c["loss32"]) <= 1e-5, (c["B"], c["C"], loss.item(), c["loss32"])  # north-star tolerance
        assert abs(loss.item() - c["loss64"]) <= 2e-5 * max(1.0, abs(c["loss64"]))
        rows = np.asarray(c["rows"])
        d1, d2 = z1.grad.cpu().numpy()[rows], z2.grad.cpu().numpy()[rows]
        w1, w2 = np.asarray(c["dz1_rows64"]), np.asarray(c["dz2_rows64"])
        scale = max(np.abs(w1).max(), 1e-12)
        # gradients: the reference's own float32 autograd deviates from float64 by up to 6e-5 of
        # the largest entry on these cases (dz1_rows32 in the golden file); same class required
        assert np.abs(d1 - w1).max() <= 1e-4 * scale, (c["B"], c["C"], np.abs(d1 - w1).max(), scale)
        assert np.abs(d2 - w2).max() <= 1e-4 * max(np.abs(w2).max(), 1e-12)
        j = compute_joint(z1.detach(), z2.detach()).cpu().numpy()
        wj = orc.compute_joint(z1n.astype(np.float64), z2n.astype(np.float64))
        np.testing.assert_allclose(j, wj, rtol=1e-5, atol=1e-12)
        assert np.array_equal(j, j.T)


def test_iid_loss_clamped_and_deterministic():
    from idelucs_b200.LossFunctions import IID_loss
    torch.manual_seed(0)
    B, C = 300, 40
    z1 = torch.softmax(torch.randn(B, C, device="cuda") * 30, 1).requires_grad_(True)   # near one-hot -> clamps
    z2 = torch.softmax(torch.randn(B, C, device="cuda") * 30, 1).requires_grad_(True)
    l1 = IID_loss(z1, z2, lamb=2.8)
    l1.backward()
    g1 = z1.grad.clone()
    wl, wd1, wd2 = orc.IID_loss_grad(z1.detach().cpu().numpy(), z2.detach().cpu().numpy(), lamb=2.8)
    assert abs(l1.item() - wl) <= 1e-5 * max(1.0, abs(wl))
    np.testing.assert_allclose(g1.cpu().numpy(), wd1, rtol=1e-3, atol=2e-5 * np.abs(wd1).max())
    z1.grad = None
    l2 = IID_loss(z1, z2, lamb=2.8)
    l2.backward()
    assert l1.item() == l2.item() and torch.equal(g1, z1.grad)


def test_pc_kernel_equals_generic(ft, SeqSet):
    """the producer/consumer kernel (k=6, float outputs, >= 512 items) must reproduce the generic
    kernel bit for bit, including items it defers (too long for its staging buffer) and Ns"""
    rng = np.random.default_rng(21)
    alph = np.frombuffer(b"ACGTACGTACGTACGTACGTACGTN", dtype=np.uint8)
    lens = rng.integers(50, 12000, size=700)
    lens[[5, 77, 300]] = [20481, 30000, 66000]      # deferred to the generic kernel (66000: long path)
    lens[[9, 10]] = [0, 3]
    seqs = [alph[rng.integers(0, alph.size, size=int(L))].tobytes() for L in lens]
    ss = SeqSet.from_sequences(seqs)
    variants = [ft.VariantSpec(ft.KIND_CLEAN)] + ft.mimic_schedule(20)
    for i, v in enumerate(variants):
        v.rng_id = i
    sc_mean = torch.rand(4096, device="cuda") * 1e-4
    sc_scale = torch.rand(4096, device="cuda") * 1e-5 + 1e-6
    outs = {}
    prep = ft.prepare(ss, 6, variants, seed=99, seq_id0=7)      # the two-call fast path (idl_profiles_prepare / _prepared)
    for mode in ("pc", "generic"):
        kw = {"prepared": prep} if mode == "pc" else {}
        f = ft.profiles(ss, 6, variants, out_kind=ft.OUT_FREQ_F32, seed=99, seq_id0=7, **kw)
        s = ft.profiles(ss, 6, variants, out_kind=ft.OUT_STD_F32, seed=99, seq_id0=7, mean=sc_mean, scale=sc_scale, **kw)
        outs[mode] = (f, s)
    assert torch.equal(outs["pc"][0], outs["generic"][0])
    assert torch.equal(outs["pc"][1], outs["generic"][1])
    # and against the oracle on a few sequences
    c = ft.profiles(ss, 6, variants, out_kind=ft.OUT_COUNTS_I32, seed=99, seq_id0=7).cpu().numpy()
    idx = [0, 5, 9, 10, 123]
    f32 = outs["pc"][0].cpu().numpy()
    for i in idx:
        for v, spec in enumerate(variants):
            edits = orc.rng_variant_edits(99, 7 + i, v, spec.kind, orc.codes_of_seq(seqs[i]), len(seqs[i]), spec.p1, spec.p2, spec.n_bp)
            mut = bytearray(seqs[i])
            for pos, val in edits:
                mut[pos] = b"ACGTN"[val]
            cnt = np.zeros(4096, np.int32)
            orc.kmer_counts(mut, 6, cnt)
            assert np.array_equal(c[v, i], cnt), (i, v)
            assert np.array_equal(f32[v, i], ((cnt + 1) / (cnt + 1).sum()).astype(np.float32)), (i, v)


def test_profile_stats_equals_matrix_fit(golden_dir, fasta_files, ft, SeqSet):
    """in-kernel statistics (idl_profile_stats) == colstats over the materialised profiles, for
    rng-mode Bernoulli, Random_N, clean and explicit (reference mutations) variants; and the
    AugmentFasta x_train built from them is still bit-identical to the reference"""
    ss = SeqSet.from_fasta(fasta_files["Influenza-A"])
    for k, spec in ((6, ft.VariantSpec(ft.KIND_BOTH, 1e-2, 0.5e-2, rng_id=0)), (5, ft.VariantSpec(ft.KIND_RANDOM_N, n_bp=20, rng_id=3)),
                    (6, ft.VariantSpec(ft.KIND_CLEAN)), (4, ft.VariantSpec(ft.KIND_TRANSVERSION, p2=0.3, rng_id=2))):
        x = ft.profiles(ss, k, [spec], out_kind=ft.OUT_FREQ_F32, seed=17)[0]
        a, b = ft.Scaler.fit(x), ft.profile_stats(ss, k, spec, seed=17)
        assert torch.allclose(a.mean64, b.mean64, rtol=1e-13, atol=0)
        assert torch.allclose(a.scale64, b.scale64, rtol=1e-9, atol=0)
        assert float(((a.mean32 - b.mean32).abs() / a.mean32.abs()).max()) < 2e-7      # at most a last-ulp flip of the cast
        c = ft.profile_stats(ss, k, spec, seed=17)
        assert torch.equal(b.mean64, c.mean64) and torch.equal(b.scale64, c.scale64)  # run-to-run identical
    g = _golden(golden_dir)["files"]["Influenza-A"]["augment_seed0_nmimics3"]
    ed = np.load(os.path.join(golden_dir, "influenza_edits_seed0.npz"))
    n, offs, k, F = ss.n, ed["offsets"], 5, 1024
    lut = np.full(256, 4, np.int64)
    for i, ch in enumerate(b"ACGT"):
        lut[ch] = i
    explicit = [[(ed["pos"][offs[p * n + i]:offs[p * n + i + 1]], lut[ed["newbyte"][offs[p * n + i]:offs[p * n + i + 1]]])
                 for i in range(n)] for p in range(4)]
    lists = ft.pack_edit_lists(explicit, n, ss.device)
    variants = [ft.VariantSpec(ft.KIND_EXPLICIT, explicit_idx=p) for p in range(4)]
    sc = ft.profile_stats(ss, k, variants[0], edit_lists=lists)
    x = torch.empty((3 * n, 2, F), dtype=torch.float32, device=ss.device)
    ft.profiles(ss, k, variants, out_kind=ft.OUT_STD_F32, edit_lists=lists, mean=sc.mean32, scale=sc.scale32,
                out=x, out_off=[0] + [((j * n) * 2 + 1) * F for j in range(3)], out_stride=2 * F)
    x[n:2 * n, 0] = x[:n, 0]
    x[2 * n:, 0] = x[:n, 0]
    assert sha(x.cpu().numpy()) == g["k5"]["x_train_sha256"]


def test_prepared_stats_equal_generic_and_matrix_fit(ft, SeqSet):
    """the statistics of the prepare pass (k=6, prep.cuh: packed uint16 histograms of slot 0 + colstats16)
    against the generic OUT_STATS path and against colstats of the materialised float32 profiles
    (themselves bit-exact against the oracle): clean and Bernoulli slots, ragged lengths incl. 0 / < k /
    block and chunk boundaries / deferred long ones, Ns, and rates high enough that the on-chip edit and
    delta lists overflow (those items are deferred to the generic kernel)"""
    rng = np.random.default_rng(33)
    alph = np.frombuffer(b"ACGTACGTACGTACGTACGTACGTACGTN", dtype=np.uint8)
    lens = rng.integers(1, 12000, size=900)
    lens[[0, 1, 2, 3, 4, 450, 899]] = [0, 3, 5, 6, 16, 16385, 70001]
    lens[[200, 201, 202, 203, 204, 205]] = [16384, 16400, 33000, 16320, 16321, 16319]
    lens[[300, 301, 302, 303]] = [63, 64, 65, 128]
    seqs = [alph[rng.integers(0, alph.size, size=int(L))].tobytes() for L in lens]
    seqs[7] = b"N" * 500
    seqs[8] = b"ACGTAC" + b"N" * 40 + b"ACGTACG"
    ss = SeqSet.from_sequences(seqs)
    few = SeqSet.from_sequences(seqs[:40])
    specs = [ft.VariantSpec(ft.KIND_CLEAN), ft.VariantSpec(ft.KIND_BOTH, 1e-2, 0.5e-2, rng_id=0),
             ft.VariantSpec(ft.KIND_TRANSITION, p1=1e-2, rng_id=1), ft.VariantSpec(ft.KIND_TRANSVERSION, p2=0.5e-2, rng_id=2),
             ft.VariantSpec(ft.KIND_BOTH, 0.06, 0.05, rng_id=5),      # the longer items overflow the delta list: deferred
             ft.VariantSpec(ft.KIND_BOTH, 0.5, 0.4, rng_id=6)]        # nearly every item deferred
    for spec in specs:
        x = ft.profiles(ss, 6, [spec], out_kind=ft.OUT_FREQ_F32, seed=17, seq_id0=3)[0]
        a = ft.Scaler.fit(x)
        b = ft.profile_stats(ss, 6, spec, seed=17, seq_id0=3)                 # prepare pass + colstats16 (+ generic for deferred items)
        g = ft.profile_stats(ss, 6, spec, seed=17, seq_id0=3, fast=False)     # generic kernel only
        for other in (a, g):
            assert torch.allclose(other.mean64, b.mean64, rtol=1e-13, atol=0), spec
            assert torch.allclose(other.scale64, b.scale64, rtol=1e-9, atol=0), spec
            assert float(((other.mean32 - b.mean32).abs() / other.mean32.abs()).max()) < 2e-7
        c = ft.profile_stats(ss, 6, spec, seed=17, seq_id0=3)
        assert torch.equal(b.mean64, c.mean64) and torch.equal(b.scale64, c.scale64)      # run-to-run identical
        slab, ft.STATS_SLAB = ft.STATS_SLAB, 600                                          # slab-wise statistics of big sets (items through sidx)
        try:
            d = ft.profile_stats(ss, 6, spec, seed=17, seq_id0=3)
        finally:
            ft.STATS_SLAB = slab
        assert torch.allclose(d.mean64, b.mean64, rtol=1e-13, atol=0) and torch.allclose(d.scale64, b.scale64, rtol=1e-9, atol=0)
        # float64 sums of the float32 frequencies on a small set
        s = ft.profile_stats(few, 6, spec, seed=17)
        xf = ft.profiles(few, 6, [spec], out_kind=ft.OUT_FREQ_F32, seed=17)[0].double().cpu().numpy()
        np.testing.assert_allclose(s.mean64.cpu().numpy(), xf.mean(axis=0), rtol=1e-13, atol=0)
        np.testing.assert_allclose(s.var64.cpu().numpy(), xf.var(axis=0), rtol=1e-8, atol=1e-30)


def test_pc_kernel_repetitive_and_degenerate_sequences(ft, SeqSet):
    """fast kernel == generic kernel on inputs that stress its sparse fix-up logic: homopolymers and short tandem
    repeats (every Random_N removal of a variant hits the same few bins: multiplicities up to 120 in the biased
    uint8 scratch), all-N and N-rich sequences (window totals near the pseudocount floor, many equal totals),
    and lengths around the 64-base chunk / 128-base mask alignment boundaries"""
    rng = np.random.default_rng(5)
    seqs = []
    for i in range(640):
        L = int(rng.integers(1, 4000))
        kind = i % 8
        if kind == 0:
            s = b"A" * L
        elif kind == 1:
            s = (b"ACG" * (L // 3 + 1))[:L]
        elif kind == 2:
            s = b"N" * L
        elif kind == 3:
            a = np.frombuffer(b"ACGTNNNN", dtype=np.uint8)
            s = a[rng.integers(0, a.size, size=L)].tobytes()
        elif kind == 4:
            s = (b"AT" * (L // 2 + 1))[:L]
        elif kind == 5:
            s = b"G" * int(rng.choice([63, 64, 65, 127, 128, 129, 191, 192, 193]))
        else:
            a = np.frombuffer(b"ACGT", dtype=np.uint8)
            s = a[rng.integers(0, 4, size=L)].tobytes()
        seqs.append(s)
    ss = SeqSet.from_sequences(seqs)
    variants = ft.mimic_schedule(50)
    mean = torch.rand(4096, device="cuda") * 1e-3
    scale = torch.rand(4096, device="cuda") * 1e-4 + 1e-6
    outs = {}
    prep = ft.prepare(ss, 6, variants, seed=3)
    for mode in ("pc", "generic"):
        kw = {"prepared": prep} if mode == "pc" else {}
        outs[mode] = ft.profiles(ss, 6, variants, out_kind=ft.OUT_STD_F32, seed=3, mean=mean, scale=scale, **kw)
    # the statistics of the prepare pass == the generic in-kernel statistics (every sequence here is short: nothing deferred)
    a, b = prep.scaler(), ft.profile_stats(ss, 6, variants[0], seed=3, fast=False)
    assert torch.allclose(a.mean64, b.mean64, rtol=1e-13, atol=0) and torch.allclose(a.scale64, b.scale64, rtol=1e-9, atol=0)
    assert torch.equal(outs["pc"], outs["generic"])
    # mimic counts of a homopolymer against the oracle's mutate-and-recount
    c = ft.profiles(ss, 6, variants, out_kind=ft.OUT_COUNTS_I32, seed=3).cpu().numpy()
    for i in (0, 8, 1, 3):
        for v in (0, 1, 2, 3, 50):
            spec = variants[v]
            edits = orc.rng_variant_edits(3, i, v, spec.kind, orc.codes_of_seq(seqs[i]), len(seqs[i]), spec.p1, spec.p2, spec.n_bp)
            mut = bytearray(seqs[i])
            for pos, val in edits:
                mut[pos] = b"ACGTN"[val]
            cnt = np.zeros(4096, np.int32)
            orc.kmer_counts(mut, 6, cnt)
            assert np.array_equal(c[v, i], cnt), (i, v)


def _ref_style_info_nce(z1, z2, temperature):
    """the reference's mask-gather formulation (idelucs/LossFunctions.py:65-98), restated on the tensors' device"""
    n = z1.shape[0]
    dev = z1.device
    feats = torch.nn.functional.normalize(torch.cat((z1, z2), 0).float(), dim=1)
    lab = torch.cat([torch.arange(n, device=dev), torch.arange(n, device=dev)])
    lab = (lab.unsqueeze(0) == lab.unsqueeze(1))
    sim = feats @ feats.T
    eye = torch.eye(2 * n, dtype=torch.bool, device=dev)
    lab, sim = lab[~eye].view(2 * n, -1), sim[~eye].view(2 * n, -1)
    logits = torch.cat([sim[lab].view(2 * n, -1), sim[~lab].view(2 * n, -1)], dim=1) / temperature
    return torch.nn.functional.cross_entropy(logits, torch.zeros(2 * n, dtype=torch.long, device=dev))


def test_fused_info_nce_matches_reference_formulation():
    """SURVEY §8f rank 2: idl_info_nce (normalise + similarity + masked log-softmax + cross-entropy + gradient, three
    launches) against the reference's formulation and its autograd gradient, in float64 as the yardstick"""
    from idelucs_b200.LossFunctions import info_nce_loss, info_nce_loss_stacked
    torch.manual_seed(3)
    for n, d, scale in ((512, 64, 1.0), (256, 64, 30.0), (5, 64, 1.0), (37, 32, 0.1), (100, 128, 3.0), (1, 64, 1.0), (64, 256, 1.0), (33, 160, 2.0)):
        a = (torch.randn(n, d, device="cuda") * scale).requires_grad_(True)
        b = (torch.randn(n, d, device="cuda") * scale + 0.3 * a.detach()).requires_grad_(True)
        want = _ref_style_info_nce(a.double(), b.double(), 0.85)
        gwa, gwb = torch.autograd.grad(want, (a, b))
        got = info_nce_loss(a, b, 0.85)
        gga, ggb = torch.autograd.grad(got, (a, b))
        assert abs(want.item() - got.item()) < 1e-5, (n, d, want.item(), got.item())
        tol = 1e-4 * float(max(gwa.abs().max(), gwb.abs().max())) + 1e-9
        assert float((gwa - gga).abs().max()) < tol and float((gwb - ggb).abs().max()) < tol, (n, d)
        got2 = info_nce_loss_stacked(torch.cat((a, b), 0), 0.85)
        assert got2.item() == got.item()                                  # run-to-run identical (fixed-order reductions)
        # float32 reference formulation agrees to its own rounding
        w32 = _ref_style_info_nce(a, b, 0.85)
        assert abs(w32.item() - got.item()) < 1e-5


def test_iid_loss_small_kernel_equals_tiled_kernel_and_oracle():
    """C <= 16 takes the single-CTA kernel (train_ops.cu): same loss / joint / gradients as the oracle's closed form, for the
    shapes of the reference's configurations (C = 3, 5, 12; last ragged batch 332 / 287) and clamped entries"""
    from idelucs_b200.LossFunctions import IID_loss, compute_joint
    rng = np.random.default_rng(8)
    for B, C, lamb in ((512, 5, 2.8), (332, 5, 2.8), (287, 3, 2.5), (256, 12, 2.8), (64, 16, 1.0), (7, 1, 2.0), (512, 2, 2.8)):
        z1 = torch.softmax(torch.from_numpy(rng.normal(size=(B, C)).astype(np.float32) * 3), 1).cuda().requires_grad_(True)
        z2 = torch.softmax(torch.from_numpy(rng.normal(size=(B, C)).astype(np.float32) * 3), 1).cuda().requires_grad_(True)
        loss = IID_loss(z1, z2, lamb=lamb)
        loss.backward()
        wl, wd1, wd2 = orc.IID_loss_grad(z1.detach().cpu().numpy(), z2.detach().cpu().numpy(), lamb=lamb)
        assert abs(loss.item() - wl) < 1e-5, (B, C, loss.item(), wl)
        m = max(np.abs(wd1).max(), np.abs(wd2).max(), 1e-12)
        assert np.abs(z1.grad.cpu().numpy() - wd1).max() < 1e-4 * m and np.abs(z2.grad.cpu().numpy() - wd2).max() < 1e-4 * m, (B, C)
        np.testing.assert_allclose(compute_joint(z1, z2).cpu().numpy(), orc.compute_joint(z1.detach().cpu().numpy(), z2.detach().cpu().numpy()),
                                   rtol=1e-5, atol=1e-8)
    # a cluster nobody uses: clamped marginal and joint entries
    z1 = torch.zeros(64, 4, device="cuda"); z1[:, 0] = 0.5; z1[:, 1] = 0.5
    z2 = z1.clone()
    z1.requires_grad_(True); z2.requires_grad_(True)
    loss = IID_loss(z1, z2, lamb=2.8)
    loss.backward()
    wl, wd1, wd2 = orc.IID_loss_grad(z1.detach().cpu().numpy(), z2.detach().cpu().numpy(), lamb=2.8)
    assert abs(loss.item() - wl) < 1e-5
    assert np.abs(z1.grad.cpu().numpy() - wd1).max() < 1e-4 * max(np.abs(wd1).max(), 1e-12)


def test_weighted_training_loss_and_seeded_gradients():
    """train_losses_and_grads (idl_nce_softmax_xent_scaled + idl_iid_loss_scaled: the weights of idelucs/models.py:128 inside the
    kernels, the combined loss written by the IIC kernel) == (1 - w) info_nce + w IID_loss of the reference formulation in
    float64 and its autograd gradients — register kernel (C <= 8; one and several rows per thread), single-CTA kernel (C <= 16),
    GEMM route (C = 200), odd batch sizes (the scalar weights kernel)"""
    from idelucs_b200.LossFunctions import train_losses_and_grads, train_losses
    torch.manual_seed(11)
    for B, C, w, lamb in ((512, 5, 0.25, 2.8), (96, 3, 0.25, 2.8), (700, 5, 0.4, 2.5), (1300, 8, 0.25, 2.8), (333, 7, 0.1, 1.0), (512, 2, 0.9, 2.8),
                          (256, 12, 0.25, 2.8), (512, 200, 0.25, 2.8), (301, 1, 0.5, 2.0)):
        z = torch.softmax(torch.randn(2 * B, C, device="cuda") * 2, 1).requires_grad_(True)
        h = torch.randn(2 * B, 64, device="cuda").requires_grad_(True)
        zd, hd = z.detach().double().requires_grad_(True), h.detach().double().requires_grad_(True)
        want = (1 - w) * _ref_style_info_nce(hd[:B], hd[B:], 0.85) + w * _ref_iid64(zd[:B], zd[B:], lamb)
        gz, gh = torch.autograd.grad(want, (zd, hd))
        loss, dz, dh = train_losses_and_grads(z, h, lamb, w, 0.85)
        assert abs(loss.item() - want.item()) < 2e-5, (B, C, loss.item(), want.item())
        assert float((dz.double() - gz).abs().max()) < 1e-4 * float(gz.abs().max()) + 1e-9, (B, C)
        assert float((dh.double() - gh).abs().max()) < 1e-4 * float(gh.abs().max()) + 1e-9, (B, C)
        # the autograd node built on the same kernels, and a second run (fixed-order reductions)
        l2 = train_losses(z, h, lamb, w, 0.85)
        az, ah = torch.autograd.grad(l2, (z, h))
        assert l2.item() == loss.item() and torch.equal(az, dz) and torch.equal(ah, dh)


def test_iid_abi_route_equals_gemm_route_and_oracle():
    """C > 16: the Python layer issues the three contractions as GEMMs around idl_iid_joint_algebra; the C ABI's own idl_iid_loss
    issues them as its two contraction kernels around the same algebra.  Both against the oracle's closed form (loss, joint,
    gradients), incl. the weighting; the C ABI's joint is exactly symmetric and a second call repeats every output bit for bit."""
    import ctypes
    from idelucs_b200 import _lib
    from idelucs_b200.LossFunctions import _iid_device, _ws
    lib = _lib.load()
    rng = np.random.default_rng(21)
    for B, C, lamb in ((512, 200, 2.8), (96, 17, 1.0), (300, 64, 2.5), (64, 256, 2.8)):
        z1 = torch.softmax(torch.from_numpy(rng.normal(size=(B, C)).astype(np.float32) * 3), 1).cuda()
        z2 = torch.softmax(torch.from_numpy(rng.normal(size=(B, C)).astype(np.float32) * 3), 1).cuda()
        wl, wd1, wd2 = orc.IID_loss_grad(z1.cpu().numpy(), z2.cpu().numpy(), lamb=lamb)
        wj = orc.compute_joint(z1.cpu().numpy(), z2.cpu().numpy())
        m = max(np.abs(wd1).max(), np.abs(wd2).max())
        add = torch.tensor(0.5, device="cuda")
        # GEMM route (what IID_loss / train_losses take)
        loss, joint, d1, d2 = _iid_device(z1, z2, lamb, sys.float_info.epsilon, want_joint=True, grad_scale=0.25, loss_weight=0.25, add=add,
                                          add_weight=0.75)
        assert abs(loss.item() - (0.25 * wl + 0.75 * 0.5)) < 1e-5, (B, C)
        np.testing.assert_allclose(joint.cpu().numpy(), wj, rtol=1e-4, atol=1e-9)
        assert np.abs(d1.cpu().numpy() - 0.25 * wd1).max() < 1e-4 * 0.25 * m and np.abs(d2.cpu().numpy() - 0.25 * wd2).max() < 1e-4 * 0.25 * m
        # the C ABI on its own (contraction kernels)
        l2 = torch.empty((), device="cuda"); j2 = torch.empty((C, C), device="cuda"); e1 = torch.empty_like(z1); e2 = torch.empty_like(z2)
        ws = _ws(z1.device, C)
        _lib.check(lib.idl_iid_loss_scaled(_lib.ptr(z1), _lib.ptr(z2), B, C, lamb, sys.float_info.epsilon, 0.25, 0.25, _lib.ptr(add), 0.75, _lib.ptr(l2),
                                           _lib.ptr(j2), _lib.ptr(e1), _lib.ptr(e2), _lib.ptr(ws), ws.numel(), _lib.stream_ptr()))
        assert abs(l2.item() - (0.25 * wl + 0.75 * 0.5)) < 1e-5, (B, C)
        np.testing.assert_allclose(j2.cpu().numpy(), wj, rtol=1e-4, atol=1e-9)
        assert np.abs(e1.cpu().numpy() - 0.25 * wd1).max() < 1e-4 * 0.25 * m and np.abs(e2.cpu().numpy() - 0.25 * wd2).max() < 1e-4 * 0.25 * m
        assert torch.equal(j2, j2.t()), (B, C)
        l3 = torch.empty_like(l2); j3 = torch.empty_like(j2); f1 = torch.empty_like(e1); f2 = torch.empty_like(e2)
        _lib.check(lib.idl_iid_loss_scaled(_lib.ptr(z1), _lib.ptr(z2), B, C, lamb, sys.float_info.epsilon, 0.25, 0.25, _lib.ptr(add), 0.75, _lib.ptr(l3),
                                           _lib.ptr(j3), _lib.ptr(f1), _lib.ptr(f2), _lib.ptr(ws), ws.numel(), _lib.stream_ptr()))
        assert torch.equal(l3, l2) and torch.equal(j3, j2) and torch.equal(f1, e1) and torch.equal(f2, e2), (B, C)


def test_trainer_forward_backward_equals_plain_module():
    """ShardedTrainer._forward (_FirstLinear + _FlatLinear + fused ReLU - Dropout kernels: gradients written into the flat buffer,
    nothing zeroed or accumulated) against the plain NetLinear module + autograd.  Dropout off (eval mode, p = 0 in the fused
    kernels): same outputs, same gradient for every parameter — also on the second step, when the flat buffer still holds the previous
    gradients.  Dropout on: the masks come from the kernels' own counter-based stream, so the module is re-run with exactly those masks."""
    from idelucs_b200.seqset import SeqSet
    from idelucs_b200.train import ShardedTrainer
    rng = np.random.default_rng(3)
    seqs = [np.frombuffer(b"ACGT", dtype=np.uint8)[rng.integers(0, 4, size=600)].tobytes() for _ in range(700)]
    tr = ShardedTrainer(SeqSet.from_sequences(seqs), k=6, n_clusters=5, n_mimics=3, batch_sz=256, seed=1)
    params = [p for p in tr.net.parameters()]
    tr.net.eval()
    for step in range(2):
        x = torch.randn(512, 4096, device="cuda")
        gz, gh = torch.randn(512, 5, device="cuda"), torch.randn(512, 64, device="cuda")
        z, h = tr._forward(x)
        torch.autograd.backward((z, h), (gz, gh))
        got = [p.grad.detach().clone() for p in params]
        zo, ho = z.detach().clone(), h.detach().clone()
        for p in params:
            p.grad.zero_()
        z2, h2 = tr.net(x)
        torch.autograd.backward((z2, h2), (gz, gh))
        assert torch.allclose(zo, z2, rtol=1e-4, atol=1e-6) and torch.allclose(ho, h2, rtol=1e-4, atol=1e-4)
        for g, p in zip(got, params):
            assert float((g - p.grad).abs().max()) <= 2e-4 * float(p.grad.abs().max()) + 1e-7, (step, tuple(p.shape))
    # training mode: recover the masks the fused kernels drew and replay the module's arithmetic with them
    tr.net.train()
    lin1, lin2, lin3 = tr.net.layers[0], tr.net.layers[3], tr.net.classifier[2]
    x = torch.randn(512, 4096, device="cuda")
    gz, gh = torch.randn(512, 5, device="cuda"), torch.randn(512, 64, device="cuda")
    tr._step_no.fill_(5)
    z, h = tr._forward(x)
    torch.autograd.backward((z, h), (gz, gh))
    got = [p.grad.detach().clone() for p in params]
    with torch.no_grad():
        a1 = torch.addmm(lin1.bias, x, lin1.weight.t())
    from idelucs_b200.train import _relu_dropout_fwd
    d1 = _relu_dropout_fwd(a1.unsqueeze(0).contiguous(), 1, None, 512, 512, tr._drop(1))
    m1 = (d1 != 0) | (a1 <= 0)                       # kept (where the unit was active; irrelevant elsewhere)
    keep1 = float(((d1 != 0) & (a1 > 0)).sum()) / float((a1 > 0).sum())
    assert abs(keep1 - 0.5) < 0.01, keep1
    assert torch.equal(d1, torch.where((a1 > 0) & m1, a1 * 2.0, torch.zeros_like(a1)))
    d2k = _relu_dropout_fwd(h.detach().unsqueeze(0).contiguous(), 1, None, 512, 64, tr._drop(2))
    m2 = (d2k != 0) | (h.detach() <= 0)
    for p in params:
        p.grad.zero_()
    a1r = torch.addmm(lin1.bias, x, lin1.weight.t())
    h2 = torch.addmm(lin2.bias, torch.relu(a1r) * m1 * 2.0, lin2.weight.t())
    z2 = torch.softmax(torch.addmm(lin3.bias, torch.relu(h2) * m2 * 2.0, lin3.weight.t()), 1)
    torch.autograd.backward((z2, h2), (gz, gh))
    assert torch.allclose(z.detach(), z2, rtol=1e-4, atol=1e-6) and torch.allclose(h.detach(), h2, rtol=1e-4, atol=1e-4)
    for g, p in zip(got, params):
        assert float((g - p.grad).abs().max()) <= 2e-4 * float(p.grad.abs().max()) + 1e-7, tuple(p.shape)
    # another step number: another mask; the same step number: the same mask
    tr._step_no.fill_(6)
    d1b = _relu_dropout_fwd(a1.unsqueeze(0).contiguous(), 1, None, 512, 512, tr._drop(1))
    tr._step_no.fill_(5)
    d1c = _relu_dropout_fwd(a1.unsqueeze(0).contiguous(), 1, None, 512, 512, tr._drop(1))
    assert torch.equal(d1c, d1) and not torch.equal(d1b, d1)


def test_first_linear_split_equals_nn_linear():
    """train._FirstLinear (inner-dimension split of the first Linear's forward GEMM, weight gradient written into its slice of a flat
    buffer) against nn.Linear + autograd on the same weights: same output, same gradients (float32 summation order aside)"""
    from idelucs_b200.train import _FirstLinear
    torch.manual_seed(5)
    lin = torch.nn.Linear(4096, 512).cuda()
    x = torch.randn(1024, 4096, device="cuda") * 3
    dy = torch.randn(1024, 512, device="cuda")
    want = lin(x)
    want.backward(dy)
    flat = torch.full((512 * 4096 + 512,), 7.0, device="cuda")           # stale contents must be overwritten, not accumulated
    gw, gb = flat[:512 * 4096].view(512, 4096), flat[512 * 4096:]
    for ns in (1, 4, 8):
        flat.fill_(7.0)
        got = _FirstLinear.apply(x, lin.weight, lin.bias, gw, gb, ns)
        got.backward(dy)
        assert float((got - want).abs().max()) < 1e-3 * float(want.abs().max())
        assert float((gw - lin.weight.grad).abs().max()) < 1e-4 * float(lin.weight.grad.abs().max())
        assert float((gb - lin.bias.grad).abs().max()) < 1e-4 * float(lin.bias.grad.abs().max())


def _ref_iid64(x_out, x_tf_out, lamb, EPS=sys.float_info.epsilon):
    """idelucs/LossFunctions.py:20-62 in float64 torch ops (the yardstick of the test above)"""
    k = x_out.shape[1]
    p_i_j = (x_out.unsqueeze(2) * x_tf_out.unsqueeze(1)).sum(dim=0)
    p_i_j = (p_i_j + p_i_j.t()) / 2.0
    p_i_j = p_i_j / p_i_j.sum()
    p_i = p_i_j.sum(dim=1).view(k, 1).expand(k, k)
    p_j = p_i_j.sum(dim=0).view(1, k).expand(k, k)
    p_i_j = torch.where(p_i_j < EPS, torch.full_like(p_i_j, EPS), p_i_j)
    p_j = torch.where(p_j < EPS, torch.full_like(p_j, EPS), p_j)
    p_i = torch.where(p_i < EPS, torch.full_like(p_i, EPS), p_i)
    return (-p_i_j * (torch.log(p_i_j) - lamb * torch.log(p_j) - lamb * torch.log(p_i))).sum()


def test_rmsprop_step_matches_torch():
    """idl_rmsprop_step == torch.optim.RMSprop(lr, weight_decay=0.01) (idelucs/models.py:86) over several steps"""
    from idelucs_b200 import _lib
    lib = _lib.load()
    torch.manual_seed(1)
    n = 100003
    p_ref = torch.nn.Parameter(torch.randn(n, device="cuda"))
    p = p_ref.detach().clone()
    sq = torch.zeros(n, device="cuda")
    opt = torch.optim.RMSprop([p_ref], lr=1e-3, weight_decay=0.01)
    for step in range(5):
        g = torch.randn(n, device="cuda") * (10.0 ** (step - 2))
        p_ref.grad = g.clone()
        opt.step()
        _lib.check(lib.idl_rmsprop_step(_lib.ptr(p), _lib.ptr(g), _lib.ptr(sq), n, 1e-3, 0.99, 1e-8, 0.01, 1.0, _lib.stream_ptr()))
    assert torch.allclose(p, p_ref.detach(), rtol=2e-6, atol=1e-7)
    assert torch.allclose(sq, opt.state[p_ref]["square_avg"], rtol=2e-6, atol=0)
