"""GPU tests (-m gpu) of the canonical output kinds of the profile kernels (IDL_OUT_CANON_F32 / _STD_F32 / _F64): the
reverse-complement fold of --model_size small done in the row emission, compared by == with the composition it replaces,
normalize_counts(revcomp_fold(counts + 1)) (idelucs/utils.py:246-250), and with the oracle; and the canonical loader that
regenerates its batches instead of materialising every mimic."""
import os

import numpy as np
import pytest

import idelucs_oracle as orc

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

SEED = 0x5EED00CA11


@pytest.fixture(scope="module")
def ft():
    from idelucs_b200 import featurise
    return featurise


@pytest.fixture(scope="module")
def SeqSet():
    from idelucs_b200.seqset import SeqSet
    return SeqSet


def _rand_seq(rng, L, n_rate=0.002):
    """random ACGT bytes with scattered Ns and, from 64 bases on, N runs"""
    a = np.frombuffer(b"ACGT", dtype=np.uint8)[rng.integers(0, 4, size=L)].copy()
    if n_rate > 0 and L > 0:
        a[rng.random(L) < n_rate] = ord("N")
        for _ in range(min(3, L // 64)):
            p = int(rng.integers(0, L))
            a[p:p + int(rng.integers(1, min(200, L // 8) + 1))] = ord("N")
    return a.tobytes()


def _explicit_lists(rng, seqs):
    lists = []
    for s in seqs:
        L = len(s)
        if L == 0:
            lists.append((np.zeros(0, np.int64), np.zeros(0, np.int64)))
            continue
        pos = np.unique(np.concatenate([rng.integers(0, L, size=min(L, 200)), [0, L - 1, L // 2]]))
        lists.append((pos, rng.integers(0, 5, size=pos.size)))
    return lists


def _variants(ft):
    """every variant kind, plus rates high enough that one tile's edits overflow the on-chip list"""
    v = [ft.VariantSpec(ft.KIND_CLEAN), ft.VariantSpec(ft.KIND_TRANSITION, p1=1e-2), ft.VariantSpec(ft.KIND_TRANSVERSION, p2=0.5e-2),
         ft.VariantSpec(ft.KIND_BOTH, 1e-2, 0.5e-2), ft.VariantSpec(ft.KIND_RANDOM_N, n_bp=20), ft.VariantSpec(ft.KIND_RANDOM_N, n_bp=333),
         ft.VariantSpec(ft.KIND_EXPLICIT, explicit_idx=0), ft.VariantSpec(ft.KIND_BOTH, 0.2, 0.3)]
    for i, s in enumerate(v):
        s.rng_id = i
    return v


def _composition(ft, ss, k, variants, **kw):
    """the composition the canonical kinds replace: +1 counts -> revcomp_fold -> normalize_counts (float64, float32)"""
    c = ft.profiles(ss, k, variants, out_kind=ft.OUT_COUNTS_I32, pseudocount=1, **kw)
    return ft.normalize_counts(ft.revcomp_fold(c, k), want64=True, want32=True)


def _check_kinds(ft, ss, k, variants, **kw):
    """the three canonical kinds against the composition, by =="""
    w64, w32 = _composition(ft, ss, k, variants, **kw)
    assert torch.equal(ft.profiles(ss, k, variants, out_kind=ft.OUT_CANON_F64, **kw), w64)
    assert torch.equal(ft.profiles(ss, k, variants, out_kind=ft.OUT_CANON_F32, **kw), w32)
    sc = ft.Scaler.fit(w32[0].contiguous())
    wstd = sc.transform32(w32.clone())
    got = ft.profiles(ss, k, variants, out_kind=ft.OUT_CANON_STD_F32, mean=sc.mean32, scale=sc.scale32, **kw)
    assert torch.equal(got, wstd)
    return w64, w32, sc


@pytest.mark.parametrize("k", [1, 2, 3, 4, 5, 6])
def test_canonical_kinds_equal_the_composition(ft, SeqSet, k):
    """every variant kind at the lengths where the kernel changes paths (empty, shorter than a window, around one packed
    word, the shared-memory staging limit, the last uint16 short-path length, the int32 long path), a homopolymer whose bin
    holds 65 535 - (k - 1) windows, odd pair sums, seq_id0 != 0; at k = 6 both the chunked path and the generic kernel"""
    rng = np.random.default_rng(900 + k)
    lens = sorted(set([0, 1, max(k - 1, 0), k] + list(range(63, 130, 11)) + [129, 20479, 20480, 20481, 65535, 65536, 70001]))
    seqs = [_rand_seq(rng, L) for L in lens] + [b"A" * 65535, b"ACGT" * 5000]
    ss = SeqSet.from_sequences(seqs)
    explicit = [_explicit_lists(rng, seqs)]
    lists = ft.pack_edit_lists(explicit, len(seqs), ss.device)
    variants = _variants(ft)
    for chunked in ((None, False) if k == 6 else (None,)):
        w64, w32, sc = _check_kinds(ft, ss, k, variants, seed=SEED, seq_id0=17, edit_lists=lists, chunked=chunked)
    # the truncation of odd pair sums matters in these rows
    c = ft.profiles(ss, k, variants[:1], out_kind=ft.OUT_COUNTS_I32, pseudocount=1)[0].cpu().numpy()
    canon = ft.canonical_index(k, "cpu").numpy()
    rc = np.array([orc.reverse_complement(int(m), k) for m in canon])
    assert ((c[:, canon] + c[:, rc]) % 2 == 1).any()
    assert c[len(lens), 0] == 65535 - (k - 1) + 1                      # the homopolymer's bin is at the uint16 ceiling
    # selection mode: repeated and out-of-order items, random slots; unaligned offsets and an odd stride
    R = w64.shape[2]
    sidx = torch.tensor([5, 0, 5, len(seqs) - 1, 3, 12, len(lens) - 1, 0], dtype=torch.int32, device="cuda")
    sel = torch.from_numpy(rng.integers(0, len(variants), size=(sidx.numel(), 3)).astype(np.int32)).cuda()
    for kind, want in ((ft.OUT_CANON_F64, w64), (ft.OUT_CANON_F32, w32)):
        got = ft.profiles(ss, k, variants, out_kind=kind, seed=SEED, seq_id0=17, edit_lists=lists, sidx=sidx, sel=sel)
        assert torch.equal(got, want[sel.long().t(), sidx.long().unsqueeze(0)])
        stride, n = R + 3, sidx.numel()
        offs = [1 + s * (n * stride + 5) for s in range(3)]
        buf = torch.full((3 * (n * stride + 5) + 8,), float("nan"), dtype=want.dtype, device="cuda")
        ft.profiles(ss, k, variants, out_kind=kind, seed=SEED, seq_id0=17, edit_lists=lists, sidx=sidx, sel=sel, out=buf, out_off=offs,
                    out_stride=stride)
        for s in range(3):
            view = torch.as_strided(buf, (n, R), (stride, 1), offs[s])
            assert torch.equal(view, got[s])
        written = torch.zeros_like(buf, dtype=torch.bool)
        for s in range(3):
            torch.as_strided(written, (n, R), (stride, 1), offs[s]).fill_(True)
        assert bool(buf[~written].isnan().all())                          # nothing outside the rows is touched
    got = ft.profiles(ss, k, variants, out_kind=ft.OUT_CANON_STD_F32, seed=SEED, seq_id0=17, edit_lists=lists, sidx=sidx, sel=sel,
                      mean=sc.mean32, scale=sc.scale32)
    assert torch.equal(got, sc.transform32(w32.clone())[sel.long().t(), sidx.long().unsqueeze(0)])


def test_canonical_kinds_on_the_chunked_path(ft, SeqSet):
    """k = 6 with 20 kb - 1 Mb genomes: the canonical emission of ch_reduce_kernel against the composition and against
    the generic kernel's long path"""
    rng = np.random.default_rng(77)
    seqs = [_rand_seq(rng, L, n_rate=0.001) for L in (20000, 70001, 250000, 1000000, 65536, 30000, 131072)]
    ss = SeqSet.from_sequences(seqs)
    variants = ft.mimic_schedule(10)
    w64, w32, sc = _check_kinds(ft, ss, 6, variants, seed=SEED, seq_id0=3)
    for kind, want in ((ft.OUT_CANON_F64, w64), (ft.OUT_CANON_F32, w32)):
        assert torch.equal(ft.profiles(ss, 6, variants, out_kind=kind, seed=SEED, seq_id0=3, chunked=False), want)


def _fasta_seqs(path):
    return [bytes(r[1]) for r in orc.read_fasta(path)]


@pytest.mark.parametrize("stem", ["Influenza-A", "Actinopterygii"])
def test_augment_device_canonical_vs_composition_and_oracle(ft, stem, fasta_files):
    """augment_device(reduce=True) by == against the old composition (restated here from the public pieces) and, at
    k = 6 on the bundled FASTA files, against the oracle's mutate-and-recount, kmer_rev_comp and StandardScaler"""
    from idelucs_b200 import utils as U
    ss = U.load_seqset(fasta_files[stem])
    k, n_mimics, seed = 6, 3, 4321
    variants = ft.mimic_schedule(n_mimics)
    x, sc, _ = U.augment_device(ss, n_mimics, k=k, seed=seed, reduce=True)
    c = ft.profiles(ss, k, variants, out_kind=ft.OUT_COUNTS_I32, seed=seed, pseudocount=1)
    old32 = ft.normalize_counts(ft.revcomp_fold(c, k), want64=False, want32=True)
    old_sc = ft.Scaler.fit(old32[0])
    for name in ("mean64", "var64", "scale64", "mean32", "scale32"):
        assert torch.equal(getattr(sc, name), getattr(old_sc, name)), name
    V, n, R = old32.shape
    assert torch.equal(x, old_sc.transform32(old32.reshape(V * n, R)).reshape(V, n, R))
    seqs = _fasta_seqs(fasta_files[stem])
    oc = orc.rng_mimic_counts(seqs, k, seed, orc.schedule_kinds(n_mimics)) + 1
    fold = np.stack([np.stack([orc.kmer_rev_comp(r.copy(), k) for r in cv]) for cv in oc])
    x32 = (fold / fold.sum(axis=2, keepdims=True)).astype(np.float32)
    want = orc.standard_scaler_transform(x32.reshape(-1, R), sc.mean64.cpu().numpy(), sc.scale64.cpu().numpy()).reshape(x32.shape)
    assert np.array_equal(x.cpu().numpy(), want)
    # reduced_profiles / kmersFasta(reduce=True) through the canonical kinds
    f64 = ft.reduced_profiles(ss, k, [ft.VariantSpec(ft.KIND_CLEAN)])[0]
    _, ref = orc.kmersFasta(fasta_files[stem], k=k, reduce=True)
    assert np.array_equal(f64.cpu().numpy(), ref)
    names, got = U.kmersFasta(fasta_files[stem], k=k, reduce=True)
    assert np.array_equal(got, ref) and len(names) == ss.n


@pytest.mark.parametrize("k", [2, 5, 6])
def test_regenerating_canonical_loader_equals_the_materialised_one(ft, SeqSet, k):
    """PairBatchLoader(reduce=True, materialize_bytes=0) against the default (materialised) loader for the same pair ids:
    identical scaler and identical batches, the last partial batch included"""
    from idelucs_b200 import utils as U
    rng = np.random.default_rng(1000 + k)
    seqs = [_rand_seq(rng, int(L)) for L in rng.integers(k, 3000, size=297)] + [_rand_seq(rng, 70001), _rand_seq(rng, 0), _rand_seq(rng, 1)]
    ss = SeqSet.from_sequences(seqs)
    n_mimics, seed = 4, 555
    mat = U.PairBatchLoader(ss, n_mimics, k=k, seed=seed, reduce=True)
    reg = U.PairBatchLoader(ss, n_mimics, k=k, seed=seed, reduce=True, materialize_bytes=0)
    assert mat.profiles is not None and reg.profiles is None
    assert torch.equal(mat.scaler.mean32, reg.scaler.mean32) and torch.equal(mat.scaler.scale32, reg.scaler.scale32)
    perm = torch.from_numpy(rng.permutation(mat.n_pairs)).cuda()
    assert mat.n_pairs % 512 != 0 and len(reg) == (mat.n_pairs + 511) // 512
    for b in range(len(reg)):
        ids = perm[b * 512:(b + 1) * 512]
        a, r = mat.batch(ids), reg.batch(ids)
        assert r["true"].shape == (ids.numel(), ft.canonical_width(k))
        assert torch.equal(a["true"], r["true"]) and torch.equal(a["modified"], r["modified"]), b


def test_canonical_loader_at_scale_within_one_matrix(ft, SeqSet):
    """10^6 sequences of 2 kb with n_mimics 10 at k = 6: the materialised canonical path would need about 360 GB; the
    loader regenerates its batches and its peak is one [N, R] float32 matrix (the t_norm rows its scaler is fitted on).
    Three batches equal the composition computed for just their sequences with the same scaler."""
    from idelucs_b200 import utils as U
    N, L, n_mimics = 10 ** 6, 2000, 10
    g = torch.Generator(device="cuda").manual_seed(11)
    a = torch.randint(0, 4, (N * L,), dtype=torch.uint8, device="cuda", generator=g)
    ascii_u8 = 65 + 2 * a + 2 * (a == 2).to(torch.uint8) + 13 * (a == 3).to(torch.uint8)   # 0 1 2 3 -> A C G T
    del a
    ss = SeqSet.from_ascii(ascii_u8, np.arange(N + 1, dtype=np.int64) * L, validate=False)
    del ascii_u8
    torch.cuda.synchronize()
    R = ft.canonical_width(6)
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    loader = U.PairBatchLoader(ss, n_mimics, k=6, seed=SEED, reduce=True)
    torch.cuda.synchronize()
    peak = torch.cuda.max_memory_allocated() - base
    bound = N * R * 4 + (256 << 20)
    assert loader.profiles is None and peak <= bound, (peak, bound)
    rng = np.random.default_rng(3)
    for _ in range(3):
        ids = torch.from_numpy(rng.integers(0, loader.n_pairs, size=512)).cuda()
        got = loader.batch(ids)
        mim = torch.div(ids, N, rounding_mode="floor") + 1
        seq = ids - (mim - 1) * N
        uniq, inv = torch.unique(seq, return_inverse=True)
        _, w32 = _composition(ft, ss, 6, loader.variants, seed=SEED, sidx=uniq.to(torch.int32))
        std = loader.scaler.transform32(w32.contiguous())
        assert torch.equal(got["true"], std[0, inv]) and torch.equal(got["modified"], std[mim, inv])


def test_cli_small_regenerated_equals_materialised(golden_dir, fasta_files, tmp_path, monkeypatch):
    """the CLI with --model_size small on Influenza-A: a run whose loader regenerates every batch writes the same
    assignments.tsv as a run whose loader materialises the profiles"""
    from idelucs_b200 import __main__ as cli
    from idelucs_b200 import models
    from idelucs_b200 import utils as U

    def run(tag, materialize_bytes):
        d = tmp_path / tag
        d.mkdir()
        monkeypatch.chdir(d)
        made = []

        def create_dataloader(sequence_file, n_mimics, k=6, batch_size=512, GT_file=None, reduce=False):
            made.append(U.PairBatchLoader(U.load_seqset(sequence_file), n_mimics, k=k, batch_size=batch_size, reduce=reduce,
                                          **({} if materialize_bytes is None else dict(materialize_bytes=materialize_bytes))))
            return made[-1]
        monkeypatch.setattr(models, "create_dataloader", create_dataloader)
        args = dict(sequence_file=fasta_files["Influenza-A"], GT_file=os.path.join(golden_dir, "Influenza-A_GT.tsv"), n_clusters=4, k=6, n_mimics=3, batch_sz=256, optimizer="RMSprop",
                    weight=0.25, lr=1e-3, scheduler="None", plot=False, n_epochs=2, n_voters=1, model_size="small")
        args["lambda"] = 2.8
        torch.manual_seed(0); np.random.seed(0)
        cli.run(args)
        assert made and all((l.profiles is None) == (materialize_bytes == 0) for l in made)
        out = [os.path.join(dp, f) for dp, _, fs in os.walk(str(d)) for f in fs if f == "assignments.tsv"]
        assert len(out) == 1
        with open(out[0]) as fh:
            return fh.read()

    a, b = run("materialised", None), run("regenerated", 0)
    assert a.count("\n") == 1 + 949 and a == b
