"""K2/K3/K4 host API: k-mer profiles of a SeqSet for a list of mimic variants, scaler
statistics and standardisation.  Thin wrappers over the C ABI; all arithmetic is in CUDA."""
import ctypes

import numpy as np
import torch

from . import _lib
from ._lib import (KIND_BOTH, KIND_CLEAN, KIND_EXPLICIT, KIND_RANDOM_N, KIND_TRANSITION, KIND_TRANSVERSION,  # noqa: F401
                   OUT_CANON_F32, OUT_CANON_F64, OUT_CANON_STD_F32, OUT_COUNTS_I32, OUT_FREQ_F32, OUT_FREQ_F64, OUT_STD_F32)

_OUT_DTYPE = {OUT_COUNTS_I32: torch.int32, OUT_FREQ_F32: torch.float32, OUT_STD_F32: torch.float32,
              OUT_FREQ_F64: torch.float64, OUT_CANON_F32: torch.float32, OUT_CANON_STD_F32: torch.float32,
              OUT_CANON_F64: torch.float64}
CANON_KINDS = (OUT_CANON_F32, OUT_CANON_STD_F32, OUT_CANON_F64)

LONG_MIN = 65536   # items at least this long take the chunked path (csrc/chunked.cuh)
MAX_EDIT_POS = 1 << 29   # edit entries are pos << 3 | val in 32 bits: mutated variants need sequences shorter than this
MAX_PARTS = 2048   # scaler partials idl_profiles_prepare / idl_profile_stats may write (>= 8 per SM)

# hard-coded rates of the reference's AugmentFasta (idelucs/utils.py:330-349)
P_TRANSITION, P_TRANSVERSION, N_RANDOM_N = 1e-2, 0.5e-2, 20


class VariantSpec(object):
    """One mimic variant: kind + parameters (+ rng_id: its identity in the Philox counter)."""

    def __init__(self, kind, p1=0.0, p2=0.0, n_bp=0, rng_id=None, explicit_idx=0):
        self.kind, self.p1, self.p2, self.n_bp, self.rng_id, self.explicit_idx = kind, p1, p2, n_bp, rng_id, explicit_idx

    def __repr__(self):
        return "VariantSpec(kind=%d, p1=%g, p2=%g, n_bp=%d, rng_id=%s)" % (self.kind, self.p1, self.p2, self.n_bp, self.rng_id)


def mimic_schedule(n_mimics):
    """Variants of AugmentFasta's pass schedule (idelucs/utils.py:330-351): pass 0 =
    transition_transversion(1e-2, 0.5e-2) (t_norm, the 'true' column), pass 1 =
    transition(1e-2), pass 2 = transversion(0.5e-2), passes 3..n_mimics = Random_N(20).
    Like the reference, passes 0..2 always exist (n_mimics < 2 still yields 2 mimics)."""
    v = [VariantSpec(KIND_BOTH, P_TRANSITION, P_TRANSVERSION), VariantSpec(KIND_TRANSITION, p1=P_TRANSITION),
         VariantSpec(KIND_TRANSVERSION, p2=P_TRANSVERSION)]
    v += [VariantSpec(KIND_RANDOM_N, n_bp=N_RANDOM_N) for _ in range(n_mimics - 2)]
    for i, s in enumerate(v):
        s.rng_id = i
    return v


_workspaces = {}
_varr_cache = {}


def _variant_array(variants):
    """ctypes idl_variant[] of a VariantSpec list (cached per list object)"""
    key = id(variants)
    hit = _varr_cache.get(key)
    sig = tuple((v.kind, v.rng_id, v.n_bp, v.explicit_idx, v.p1, v.p2) for v in variants)
    if hit is not None and hit[0] == sig:
        return hit[1]
    varr = (_lib.Variant * len(variants))()
    for i, v in enumerate(variants):
        varr[i].kind, varr[i].rng_id, varr[i].n_bp = v.kind, (v.rng_id if v.rng_id is not None else i), v.n_bp
        varr[i].explicit_idx, varr[i].p1, varr[i].p2 = v.explicit_idx, v.p1, v.p2
    if len(_varr_cache) > 64:
        _varr_cache.clear()
    _varr_cache[key] = (sig, varr)
    return varr


def _workspace(device, nbytes, tag):
    key = (device.index if device.index is not None else torch.cuda.current_device(),
           torch.cuda.current_stream(device).cuda_stream, tag)
    ws = _workspaces.get(key)
    if ws is None or ws.numel() < nbytes:
        ws = torch.empty(nbytes, dtype=torch.uint8, device=device)
        _workspaces[key] = ws
    return ws


def _seqset_args(seqset):
    """(codes, nmask, chunk_off, len, n): the arguments the profile entry points start with"""
    return _lib.ptr(seqset.codes), _lib.ptr(seqset.nmask), _lib.ptr(seqset.chunk_off), _lib.ptr(seqset.len), seqset.n


def _seed(seed):
    return ctypes.c_uint64(seed & (2 ** 64 - 1))


def _workspace_args(lib, device):
    """(workspace, its size, stream): the arguments the profile entry points end with (inside ``torch.cuda.device(device)``)"""
    ws = _workspace(device, lib.idl_profiles_workspace_bytes(), "prof")
    return _lib.ptr(ws), ws.numel(), _lib.stream_ptr()


def _stats_buffers(F, device):
    return (torch.empty((MAX_PARTS, 2, F), dtype=torch.float64, device=device),
            torch.zeros((MAX_PARTS,), dtype=torch.float64, device=device))


def _scaler(parts, part_n, group):
    """Scaler of this process's partials, or of the whole torch.distributed group's (a collective) when group is given"""
    if group is not None:
        parts, part_n = gather_partials(parts, part_n, group)
    return Scaler.from_partials(parts, part_n)


def pack_edit_lists(explicit, n_seqs, device):
    """explicit: list (one per EXPLICIT variant) of per-sequence (pos, val) pairs, val in 0..4
    (A C G T N) -> CSR (int64 offsets, int32-typed uint32 entries pos<<3|val) on the device."""
    offs = [0]
    chunks = []
    for lists in explicit:
        assert len(lists) == n_seqs
        for pos, val in lists:
            pos = np.asarray(pos, dtype=np.int64)
            val = np.asarray(val, dtype=np.int64)
            order = np.argsort(pos, kind="stable")
            pos, val = pos[order], val[order]
            if pos.size and (np.diff(pos) <= 0).any():
                raise ValueError("explicit edit positions must be unique per sequence")
            if pos.size and (int(pos[-1]) >= MAX_EDIT_POS or int(pos[0]) < 0):
                raise ValueError("edit positions must be in [0, 2^29): entries are pos << 3 | val in 32 bits")
            chunks.append(((pos << 3) | val).astype(np.uint32))
            offs.append(offs[-1] + pos.size)
    ent = np.concatenate(chunks) if chunks else np.zeros(0, np.uint32)
    if ent.size == 0:
        ent = np.zeros(1, np.uint32)
    d_off = torch.from_numpy(np.asarray(offs, dtype=np.int64)).to(device)
    d_ent = torch.from_numpy(ent.view(np.int32)).to(device)
    return d_off, d_ent


class Prepared(object):
    """Result of ``prepare``: the device buffer the k = 6 fast path reads its Bernoulli deltas from, and the scaler
    partials of slot 0 computed on the way."""

    def __init__(self, buf, parts, part_n, key):
        self.buf, self.parts, self.part_n, self.key = buf, parts, part_n, key

    def scaler(self, group=None):
        return _scaler(self.parts, self.part_n, group)


def can_prepare(seqset, k, variants, n_items=None):
    """whether the two-call whole-schedule path (idl_profiles_prepare / idl_profiles_prepared) applies"""
    n_items = seqset.n if n_items is None else n_items
    bern = sum(1 for v in variants if v.kind in (KIND_TRANSITION, KIND_TRANSVERSION, KIND_BOTH))
    rates = set([v.p1 for v in variants if v.kind in (KIND_TRANSITION, KIND_BOTH)] + [v.p2 for v in variants if v.kind in (KIND_TRANSVERSION, KIND_BOTH)])
    v0 = variants[0]
    ok0 = v0.kind in (KIND_CLEAN, KIND_TRANSITION, KIND_TRANSVERSION, KIND_BOTH) or (v0.kind == KIND_RANDOM_N and v0.n_bp <= 0)
    return (k == 6 and n_items >= 512 and len(variants) <= 64 and bern <= 3 and len(rates) <= 4 and ok0
            and not any(v.kind == KIND_EXPLICIT for v in variants))


def prepare(seqset, k, variants, seed=0, seq_id0=0, pseudocount=1, want_stats=True, sidx=None, buf=None):
    """idl_profiles_prepare over the SeqSet (or the items ``sidx``): ONE pass that generates the Bernoulli mimics' histogram
    deltas for the profile pass (``profiles(..., prepared=...)``) and the scaler statistics of variants[0]."""
    lib = _lib.load()
    device = seqset.device
    F = 4 ** k
    n = seqset.n if sidx is None else int(sidx.numel())
    nbytes = lib.idl_prepare_bytes(n)
    if buf is None or buf.numel() < nbytes:
        buf = torch.empty(nbytes, dtype=torch.uint8, device=device)
    parts, part_n = _stats_buffers(F, device) if want_stats else (None, None)
    n_parts = ctypes.c_int(0)
    status = torch.zeros((max(n, 1),), dtype=torch.int32, device=device)
    varr = _variant_array(variants)
    with torch.cuda.device(device):
        _lib.check(lib.idl_profiles_prepare(*_seqset_args(seqset), _lib.ptr(sidx), n, int(seq_id0), k, varr, len(variants), _seed(seed),
                                            int(pseudocount), _lib.ptr(buf), buf.numel(), _lib.ptr(parts), _lib.ptr(part_n), MAX_PARTS,
                                            ctypes.byref(n_parts), _lib.ptr(status), *_workspace_args(lib, device)))
    if want_stats:
        parts, part_n = parts[: n_parts.value], part_n[: n_parts.value]
    return Prepared(buf, parts, part_n, (id(seqset), k, seed, seq_id0, pseudocount, len(variants)) if sidx is None else None)


STATS_SLAB = 131072   # sequences per prepare call when only the statistics are wanted (2.4 GB of scratch, reused)


def profiles(seqset, k, variants, out_kind=OUT_FREQ_F32, seed=0, out=None, out_off=None, out_stride=None,
             mean=None, scale=None, sidx=None, sel=None, S=None, edit_lists=None, seq_id0=0, pseudocount=None,
             accumulate=False, status=None, prepared=None, chunked=None, max_long=None, cta_cap=0):
    """Run K2+K3.  Default output: tensor [S, n_items, 4^k] (variant-major) of the out_kind's
    dtype; [S, n_items, R] (R = canonical_width(k)) for the canonical kinds OUT_CANON_*.  See
    include/idelucs_b200.h::idl_profiles for the argument meaning.  The standardised kinds equal IEEE float32 division by
    ``scale`` when every scale is a finite, normal float (``Scaler`` guarantees that for frequency columns); a zero or
    infinite scale, or a subnormal one whose reciprocal overflows, gives NaN instead.  ``prepared`` (from ``prepare`` with the
    same SeqSet / variants / seed / seq_id0) routes float32 outputs through idl_profiles_prepared (k = 6 fast path).  Sets with
    sequences of >= 65 536 bases go through idl_profiles_chunked (k = 6; chunked=False forces the generic kernel).  ``cta_cap`` > 0
    caps the generic kernel at that many CTAs per SM (room for a concurrent stream)."""
    lib = _lib.load()
    device = seqset.device
    F = canonical_width(k) if out_kind in CANON_KINDS else 4 ** k
    n_items = int(sidx.numel()) if sidx is not None else seqset.n
    nv = len(variants)
    if S is None:
        S = nv if sel is None else int(sel.shape[1])
    if pseudocount is None:
        pseudocount = 0 if out_kind == OUT_COUNTS_I32 else 1
    if out is None:
        out = torch.empty((S, n_items, F), dtype=_OUT_DTYPE[out_kind], device=device)
        out_off = [s * n_items * F for s in range(S)]
        out_stride = F
    assert out.dtype == _OUT_DTYPE[out_kind] and out.is_contiguous()
    if seqset.n and int(seqset.lengths.max()) >= MAX_EDIT_POS and any(v.kind != KIND_CLEAN for v in variants):
        raise _lib.IdelucsB200Error("mimic variants need sequences shorter than 2^29 bases (32-bit edit entries); clean counting takes any length < 2^31")
    varr = _variant_array(variants)
    offs = (ctypes.c_int64 * S)(*[int(o) for o in out_off])
    d_eoff, d_ent = (None, None) if edit_lists is None else edit_lists
    with torch.cuda.device(device):
        if prepared is not None:
            assert sidx is None and sel is None and edit_lists is None and out_kind in (OUT_FREQ_F32, OUT_STD_F32)
            assert prepared.key == (id(seqset), k, seed, seq_id0, pseudocount, nv), "prepared for a different call"
            if status is None:
                status = torch.zeros(n_items, dtype=torch.int32, device=device)
            _lib.check(lib.idl_profiles_prepared(
                *_seqset_args(seqset), None, n_items, int(seq_id0), k, varr, nv, _seed(seed), out_kind, _lib.ptr(out), offs,
                int(out_stride), int(pseudocount), _lib.ptr(mean), _lib.ptr(scale), _lib.ptr(status), _lib.ptr(prepared.buf),
                prepared.buf.numel(), *_workspace_args(lib, device)))
            return out
        # long sequences (>= 65 536 bases, k = 6): tiles shared by the whole grid instead of one CTA per sequence
        n_long = int((seqset.lengths >= LONG_MIN).sum()) if (k == 6 and sidx is None and chunked is not False) else 0
        if n_long > 0 and max_long is not None:
            n_long = int(max_long)   # (tests: a scratch sized for fewer long items than there are makes the device fall back)
        if n_long > 0:
            nbytes = lib.idl_profiles_chunked_bytes(n_items, n_long, varr, nv, S)
            if nbytes > 0:
                scratch = _workspace(device, nbytes, "chunk")
                _lib.check(lib.idl_profiles_chunked(
                    *_seqset_args(seqset), None, n_items, int(seq_id0), k, varr, nv, _lib.ptr(sel), S, _seed(seed),
                    _lib.ptr(d_eoff), _lib.ptr(d_ent), out_kind, _lib.ptr(out), offs, int(out_stride), int(pseudocount),
                    1 if accumulate else 0, _lib.ptr(mean), _lib.ptr(scale), _lib.ptr(scratch), scratch.numel(), n_long,
                    *_workspace_args(lib, device)))
                return out
        _lib.check(lib.idl_profiles(
            *_seqset_args(seqset), _lib.ptr(sidx), n_items, int(seq_id0), k, varr, nv, _lib.ptr(sel), S, _seed(seed),
            _lib.ptr(d_eoff), _lib.ptr(d_ent), out_kind, _lib.ptr(out), offs, int(out_stride), int(pseudocount),
            (1 if accumulate else 0) | ((int(cta_cap) & 0xFF) << 8), _lib.ptr(mean), _lib.ptr(scale), _lib.ptr(status),
            *_workspace_args(lib, device)))
    return out


def schedule_profiles(seqset, k, variants, out_kind=OUT_STD_F32, seed=0, seq_id0=0, group=None, out=None, out_off=None,
                      out_stride=None, fast=True):
    """The AugmentFasta computation on the device (idelucs/utils.py:330-366): statistics of variants[0]'s float32 frequencies
    -> every variant's profile (standardised with them when out_kind is OUT_STD_F32).  Returns (profiles, Scaler).
    fast=False keeps everything on the generic kernels (any k; the parity tests compare the two)."""
    if fast and k == 6 and seqset.n > 0 and int(seqset.lengths.max()) >= LONG_MIN:
        # long genomes (BASELINE configs[4]): integer counts of every slot through the chunked path (mutations generated once),
        # then float32(count / total) (idl_normalize_counts: the reference's float64 division + cast), statistics of slot 0,
        # standardisation — all elementwise passes over a small [V, N, 4096] matrix
        c = profiles(seqset, k, variants, out_kind=OUT_COUNTS_I32, seed=seed, seq_id0=seq_id0, pseudocount=1)
        x = normalize_counts(c, want64=False, want32=True)
        del c
        sc = Scaler.fit(x[0], group=group)
        if out_kind == OUT_STD_F32:
            sc.transform32(x.view(-1, x.shape[-1]))
        if out is not None:
            F = x.shape[-1]
            for s_i, o in enumerate(out_off):
                torch.as_strided(out.view(-1), (x.shape[1], F), (int(out_stride), 1), int(o)).copy_(x[s_i])
            return out, sc
        return x, sc
    if fast and can_prepare(seqset, k, variants):
        prep = prepare(seqset, k, variants, seed=seed, seq_id0=seq_id0)
        sc = prep.scaler(group)
        x = profiles(seqset, k, variants, out_kind=out_kind, seed=seed, seq_id0=seq_id0, mean=sc.mean32, scale=sc.scale32,
                     out=out, out_off=out_off, out_stride=out_stride, prepared=prep)
        return x, sc
    sc = profile_stats(seqset, k, variants[0], seed=seed, seq_id0=seq_id0, group=group, fast=False)
    x = profiles(seqset, k, variants, out_kind=out_kind, seed=seed, seq_id0=seq_id0, mean=sc.mean32, scale=sc.scale32,
                 out=out, out_off=out_off, out_stride=out_stride)
    return x, sc


def profile_stats(seqset, k, variant, seed=0, seq_id0=0, edit_lists=None, group=None, pseudocount=1, fast=True):
    """Scaler statistics of one variant's float32 frequency profiles over the whole SeqSet, computed
    inside the featurisation kernels (no [N, 4^k] matrix is written or re-read).  Equivalent to
    ``Scaler.fit(profiles(seqset, k, [variant], OUT_FREQ_F32)[0], group)``."""
    if fast and edit_lists is None and can_prepare(seqset, k, [variant]):
        if seqset.n <= STATS_SLAB:
            return prepare(seqset, k, [variant], seed=seed, seq_id0=seq_id0, pseudocount=pseudocount).scaler(group)
        # big sets (configs[3]: 10^6 sequences): slab by slab through one reused scratch buffer; the parts are merged in slab order
        parts, part_n, buf = [], [], None
        for lo in range(0, seqset.n, STATS_SLAB):
            idx = torch.arange(lo, min(lo + STATS_SLAB, seqset.n), dtype=torch.int32, device=seqset.device)
            pr = prepare(seqset, k, [variant], seed=seed, seq_id0=seq_id0, pseudocount=pseudocount, sidx=idx, buf=buf)
            buf = pr.buf
            parts.append(pr.parts.clone()); part_n.append(pr.part_n.clone())
        return _scaler(torch.cat(parts), torch.cat(part_n), group)
    lib = _lib.load()
    device = seqset.device
    F = 4 ** k
    parts, part_n = _stats_buffers(F, device)
    varr = _variant_array([variant])
    n_parts = ctypes.c_int(0)
    d_eoff, d_ent = (None, None) if edit_lists is None else edit_lists
    with torch.cuda.device(device):
        _lib.check(lib.idl_profile_stats(*_seqset_args(seqset), None, seqset.n, int(seq_id0), k, varr, _seed(seed),
                                         _lib.ptr(d_eoff), _lib.ptr(d_ent), int(pseudocount), _lib.ptr(parts), _lib.ptr(part_n),
                                         MAX_PARTS, ctypes.byref(n_parts), None, *_workspace_args(lib, device)))
    parts, part_n = parts[: n_parts.value].contiguous(), part_n[: n_parts.value].contiguous()
    if seqset.n == 0:
        parts, part_n = torch.zeros((1, 2, F), dtype=torch.float64, device=device), torch.zeros((1,), dtype=torch.float64, device=device)
    return _scaler(parts, part_n, group)


def kmer_counts_batch(seqset, k, counts=None):
    """int32 counts [n, 4^k] of every sequence (idelucs/kmers.pyx:2-50 per sequence)."""
    lib = _lib.load()
    accumulate = counts is not None
    if counts is None:
        counts = torch.empty((seqset.n, 4 ** k), dtype=torch.int32, device=seqset.device)
    with torch.cuda.device(seqset.device):
        _lib.check(lib.idl_kmer_counts(*_seqset_args(seqset), k, _lib.ptr(counts), 1 if accumulate else 0, *_workspace_args(lib, seqset.device)))
    return counts


def cgr_batch(counts, k, cgr=None):
    """FCGR cell counts [n, 4^k] (idelucs/kmers.pyx:53-123) from the k-mer counts of the same windows: a fixed
    permutation of the count vector (idl_cgr_map); accumulates into ``cgr`` when given."""
    lib = _lib.load()
    accumulate = cgr is not None
    if cgr is None:
        cgr = torch.empty_like(counts)
    assert counts.dtype == torch.int32 and counts.is_contiguous() and cgr.is_contiguous()
    with torch.cuda.device(counts.device):
        _lib.check(lib.idl_cgr_map(_lib.ptr(counts), counts.shape[0], k, _lib.ptr(cgr), 1 if accumulate else 0, _lib.stream_ptr()))
    return cgr


_canon_cache = {}


def canonical_index(k, device):
    """int32 device tensor of the canonical k-mers of kmer_rev_comp (idelucs/utils.py:208-221), increasing"""
    key = (k, str(device))
    if key not in _canon_cache:
        lib = _lib.load()
        import numpy as np
        h = np.empty(4 ** k, np.int32)
        R = lib.idl_revcomp_canonical(k, ctypes.c_void_p(h.ctypes.data))
        _canon_cache[key] = torch.from_numpy(h[:R].copy()).to(device)
    return _canon_cache[key]


def canonical_width(k):
    """R: the number of canonical k-mers, the width of a row of the canonical output kinds (idl_revcomp_canonical)"""
    return _lib.load().idl_revcomp_canonical(k, None)


def revcomp_fold(counts, k):
    """kmer_rev_comp on int32 counts [..., 4^k] (pseudocount included) -> int32 [..., R] (idl_revcomp_fold)"""
    lib = _lib.load()
    canon = canonical_index(k, counts.device)
    flat = counts.reshape(-1, 4 ** k).contiguous()
    out = torch.empty((flat.shape[0], canon.numel()), dtype=torch.int32, device=counts.device)
    with torch.cuda.device(counts.device):
        _lib.check(lib.idl_revcomp_fold(_lib.ptr(flat), flat.shape[0], k, _lib.ptr(canon), canon.numel(), _lib.ptr(out), _lib.stream_ptr()))
    return out.reshape(tuple(counts.shape[:-1]) + (canon.numel(),))


def normalize_counts(counts, want64=True, want32=False):
    """counts / np.sum(counts) per row of an int32 [..., R] tensor (idelucs/utils.py:250, 272): float64 and / or
    float32(float64) (idl_normalize_counts)"""
    lib = _lib.load()
    R = counts.shape[-1]
    flat = counts.reshape(-1, R).contiguous()
    o64 = torch.empty(flat.shape, dtype=torch.float64, device=counts.device) if want64 else None
    o32 = torch.empty(flat.shape, dtype=torch.float32, device=counts.device) if want32 else None
    with torch.cuda.device(counts.device):
        _lib.check(lib.idl_normalize_counts(_lib.ptr(flat), flat.shape[0], R, _lib.ptr(o64), _lib.ptr(o32), _lib.stream_ptr()))
    res = tuple(t.reshape(counts.shape) for t in (o64, o32) if t is not None)
    return res[0] if len(res) == 1 else res


def reduced_profiles(seqset, k, variants, seed=0, edit_lists=None, seq_id0=0, want64=True, want32=False):
    """reduce=True path of kmersFasta (idelucs/utils.py:246-250): +1-pseudocount counts of every variant ->
    canonical folding -> counts / sum, folded in the profile kernel's row emission (OUT_CANON_F64 / OUT_CANON_F32: the
    values of ``normalize_counts(revcomp_fold(counts + 1))`` without the [V, N, 4^k] counts).  Returns [V, N, R] float64
    and / or float32."""
    kinds = ([OUT_CANON_F64] if want64 else []) + ([OUT_CANON_F32] if want32 else [])
    res = tuple(profiles(seqset, k, variants, out_kind=o, seed=seed, edit_lists=edit_lists, seq_id0=seq_id0, pseudocount=1) for o in kinds)
    return res[0] if len(res) == 1 else res


class Scaler(object):
    """StandardScaler statistics on the device (idelucs/utils.py:358-359, 404-405)."""

    def __init__(self, mean64, var64, scale64, mean32, scale32, n):
        self.mean64, self.var64, self.scale64, self.mean32, self.scale32, self.n = mean64, var64, scale64, mean32, scale32, n

    @staticmethod
    def partials(x):
        """(partials [P,2,F] float64, part_n [P] float64) of a row-major [n, F] float32/float64 matrix"""
        lib = _lib.load()
        assert x.dim() == 2 and x.is_contiguous() and x.dtype in (torch.float32, torch.float64)
        n, F = x.shape
        P = lib.idl_colstats_parts(n)
        parts = torch.empty((P, 2, F), dtype=torch.float64, device=x.device)
        part_n = torch.empty((P,), dtype=torch.float64, device=x.device)
        with torch.cuda.device(x.device):
            _lib.check(lib.idl_colstats(_lib.ptr(x), 1 if x.dtype == torch.float64 else 0, n, F, _lib.ptr(parts),
                                        _lib.ptr(part_n), _lib.stream_ptr()))
        return parts, part_n

    @classmethod
    def from_partials(cls, parts, part_n):
        lib = _lib.load()
        P, _, F = parts.shape
        dev = parts.device
        mean64, var64, scale64 = (torch.empty(F, dtype=torch.float64, device=dev) for _ in range(3))
        mean32, scale32 = (torch.empty(F, dtype=torch.float32, device=dev) for _ in range(2))
        with torch.cuda.device(dev):
            _lib.check(lib.idl_scaler_finalize(_lib.ptr(parts), _lib.ptr(part_n), P, F, _lib.ptr(mean64), _lib.ptr(var64),
                                               _lib.ptr(scale64), _lib.ptr(mean32), _lib.ptr(scale32), _lib.stream_ptr()))
        return cls(mean64, var64, scale64, mean32, scale32, None)

    @classmethod
    def fit(cls, x, group=None):
        """Statistics of x's columns.  group=None: this process only.  With a torch.distributed
        group the per-rank partials are all-gathered (rank order) and merged identically on
        every rank (a collective: every rank of the group must call it)."""
        return _scaler(*cls.partials(x), group)

    def transform32(self, x, out=None):
        lib = _lib.load()
        assert x.dtype == torch.float32 and x.is_contiguous()
        F = x.shape[-1]
        out = x if out is None else out
        with torch.cuda.device(x.device):
            _lib.check(lib.idl_standardize_f32(_lib.ptr(x), _lib.ptr(out), x.numel() // F, F, _lib.ptr(self.mean32),
                                               _lib.ptr(self.scale32), _lib.stream_ptr()))
        return out

    def transform64(self, x, want32=False):
        lib = _lib.load()
        assert x.dtype == torch.float64 and x.is_contiguous()
        F = x.shape[-1]
        out64 = None if want32 else torch.empty_like(x)
        out32 = torch.empty(x.shape, dtype=torch.float32, device=x.device) if want32 else None
        with torch.cuda.device(x.device):
            _lib.check(lib.idl_standardize_f64(_lib.ptr(x), _lib.ptr(out64), _lib.ptr(out32), x.numel() // F, F,
                                               _lib.ptr(self.mean64), _lib.ptr(self.scale64), _lib.stream_ptr()))
        return out32 if want32 else out64


def _merge_local(parts, part_n):
    """this rank's parts -> ONE (mean, M2, rows) part, fixed-order Chan merge (idl_scaler_finalize on the device; the
    same recurrence in torch for host tensors, which only the gloo host-logic tests use)"""
    if parts.is_cuda:
        s = Scaler.from_partials(parts, part_n)
        n = part_n.sum()
        # M2 = var * rows: one float64 rounding away from the merge's own M2 (far below the 1e-9 the scale is compared
        # at); a constant column keeps its exact 0
        return s.mean64, s.var64 * n, n
    F = parts.shape[2]
    na, ma, M2 = 0.0, torch.zeros(F, dtype=torch.float64), torch.zeros(F, dtype=torch.float64)
    for g in range(parts.shape[0]):
        nb = float(part_n[g])
        if nb <= 0:
            continue
        delta = parts[g, 0] - ma
        nt = na + nb
        ma = ma + delta * (nb / nt)
        M2 = M2 + parts[g, 1] + delta * delta * (na * nb / nt)
        na = nt
    return ma, M2, torch.tensor(na, dtype=torch.float64)


def gather_partials(parts, part_n, group=None):
    """Scaler partials of the whole group: every rank first merges its own parts into one, then the ranks exchange
    2·F + 1 doubles each (all-gather, rank order) — no host synchronisation, 64 KB per rank at k = 6 instead of
    one part per CTA.  Returns ([world, 2, F], [world])."""
    import torch.distributed as dist
    world = dist.get_world_size(group)
    F = parts.shape[2]
    mean, M2, n = _merge_local(parts, part_n)
    packed = torch.cat([mean.reshape(-1), M2.reshape(-1), n.reshape(1)]).contiguous()
    out = [torch.empty_like(packed) for _ in range(world)]
    dist.all_gather(out, packed, group=group)
    out = torch.stack(out, 0)
    return out[:, : 2 * F].reshape(world, 2, F).contiguous(), out[:, 2 * F].contiguous()
