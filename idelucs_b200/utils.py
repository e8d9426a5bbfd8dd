"""Featurisation front-end with the reference's names and signatures (idelucs/utils.py).

``kmersFasta`` / ``AugmentFasta`` / ``create_dataloader`` / ``SequenceDataset`` parse the
FASTA file ONCE, keep the sequences packed on the GPU and produce profiles with the sm_100a
kernels (featurise.py -> C ABI).  Mutations ("mimics") come from the counter-based device
RNG; passing any *other* callable as ``transform`` (for instance the reference's own
transform objects, which draw from numpy's global MT19937 stream) is honoured exactly by
running it on the host bytes, diffing, and feeding the edits to the device as explicit edit
lists — that path reproduces the reference bit for bit.
"""
import os

import numpy as np
import torch

from . import _lib
from . import featurise as ft
from .seqset import SeqSet, read_fasta_raw

_A, _C, _G, _T, _N = (ord(c) for c in "ACGTN")
# check_sequence's alphabet (idelucs/utils.py:42-46) as one 256-entry table: canonical byte,
# 0 = deleted whitespace, 255 = left as is (invalid unless already ACGTN)
_CANON = np.arange(256, dtype=np.uint8)
for _src, _dst in ((b"acgtuU", b"ACGTTT"), (b"swkmyrbdhvnSWKMYRBDHV-", b"N" * 22)):
    for _s, _d in zip(_src, _dst):
        _CANON[_s] = _d


def check_sequence(header, seq):
    """idelucs/utils.py:26-51: header checks, alphabet normalisation, ValueError on an invalid
    byte.  Host helper kept for API compatibility (the device packer applies the same mapping)."""
    if len(header) > 0 and (header[0] in (">", "#") or header[0].isspace()):
        raise ValueError("Bad character in sequence header")
    if "\t" in header:
        raise ValueError("tab included in header")
    a = np.frombuffer(bytes(seq), dtype=np.uint8)
    a = a[~np.isin(a, np.frombuffer(b" \t\n\r", dtype=np.uint8))]
    a = _CANON[a]
    bad = ~np.isin(a, np.frombuffer(b"ACGTN", dtype=np.uint8))
    if bad.any():
        raise ValueError("Invalid DNA byte in sequence {}: '{}'".format(header, chr(int(a[np.argmax(bad)]))))
    return bytearray(a.tobytes())


# ---- transform descriptors (idelucs/utils.py:54-135) ---------------------------------------
class _DeviceTransform(object):
    """Marker base: kmersFasta maps these to device RNG variants instead of calling them."""
    kind = ft.KIND_CLEAN
    p1 = p2 = 0.0
    n_bp = 0

    def spec(self, rng_id):
        return ft.VariantSpec(self.kind, p1=self.p1, p2=self.p2, n_bp=self.n_bp, rng_id=rng_id)


class transition(_DeviceTransform):
    """A<->G, C<->T with probability ``threshold`` per base (idelucs/utils.py:54-76)."""
    kind = ft.KIND_TRANSITION

    def __init__(self, threshold):
        self.threshold = self.p1 = threshold

    def __call__(self, seq):  # host compatibility path, numpy global RNG like the reference
        x = np.random.random(len(seq))
        for i in np.where(x < self.threshold)[0]:
            seq[i] = {_A: _G, _G: _A, _T: _C, _C: _T}.get(seq[i], seq[i])


class transversion(_DeviceTransform):
    """purine <-> random pyrimidine with probability ``threshold`` (idelucs/utils.py:98-118)."""
    kind = ft.KIND_TRANSVERSION

    def __init__(self, threshold):
        self.threshold = self.p2 = threshold

    def __call__(self, seq):
        import random
        x = np.random.random(len(seq))
        table = {_A: (_T, _C), _G: (_T, _C), _T: (_A, _G), _C: (_A, _G)}
        for i in np.where(x < self.threshold)[0]:
            seq[i] = random.choice(table.get(seq[i], (_N,)))


class transition_transversion(_DeviceTransform):
    """transition(threshold_1) then transversion(threshold_2) (idelucs/utils.py:120-135)."""
    kind = ft.KIND_BOTH

    def __init__(self, threshold_1, threshold_2):
        self.tf1, self.tf2 = transition(threshold_1), transversion(threshold_2)
        self.p1, self.p2 = threshold_1, threshold_2

    def __call__(self, seq):
        self.tf1(seq)
        self.tf2(seq)


class Random_N(_DeviceTransform):
    """``n_bp`` uniformly drawn positions (with replacement) become N (idelucs/utils.py:78-95)."""
    kind = ft.KIND_RANDOM_N

    def __init__(self, n_bp):
        self.n_bp = n_bp

    def __call__(self, seq):
        for i in np.random.randint(0, len(seq), self.n_bp):
            seq[i] = _N


# ---- seeds ------------------------------------------------------------------------------------
def _draw_seed():
    """Device RNG seed drawn from numpy's global stream, so ``np.random.seed(s)`` (which the
    reference does at import, models.py:18-21) makes a run reproducible here too."""
    return int(np.random.randint(0, 2 ** 31 - 1)) * (2 ** 31) + int(np.random.randint(0, 2 ** 31 - 1))


_seqset_cache = {}


def _to_host(t):
    """device tensor -> numpy through a pinned staging buffer (PyTorch's caching host allocator recycles it): a pageable
    `.cpu()` of the 93 MB x_train of Influenza-A at k = 6 takes 40 ms, the pinned copy 2 ms"""
    host = torch.empty(t.shape, dtype=t.dtype, pin_memory=True)
    host.copy_(t, non_blocking=True)
    torch.cuda.current_stream(t.device).synchronize()
    return host.numpy()


def load_seqset(fname, device=None):
    """Parse + pack a FASTA file once per (path, mtime, device)."""
    device = torch.device(device if device is not None else "cuda")
    key = (os.path.abspath(fname), os.path.getmtime(fname), str(device))
    ss = _seqset_cache.get(key)
    if ss is None:
        ss = SeqSet.from_fasta(fname, device=device)
        ss._host_seqs = None
        _seqset_cache.clear()
        _seqset_cache[key] = ss
    return ss


def _explicit_lists_from_callable(fname, ss, transform):
    """Run an arbitrary host transform on every record (file order, like kmersFasta does) and
    return its effect as device edit lists."""
    names, seqs = read_fasta_raw(fname)
    lut = np.full(256, 4, np.int64)
    for i, ch in enumerate(b"ACGT"):
        lut[ch] = i
    lists = []
    for name, raw in zip(names, seqs):
        before = check_sequence(name, raw)
        after = bytearray(before)
        transform(after)
        if len(after) != len(before):
            raise ValueError("transform changed the sequence length")
        b, a = np.frombuffer(bytes(before), np.uint8), np.frombuffer(bytes(after), np.uint8)
        pos = np.nonzero(a != b)[0]
        lists.append((pos, lut[a[pos]]))
    return ft.pack_edit_lists([lists], ss.n, ss.device)


def kmersFasta(fname, k=6, transform=None, reduce=False):
    """idelucs/utils.py:224-277 -> (names, float64[N, 4^k]) with the +1 pseudocount (reduce=True: float64
    [N, R] over the canonical k-mers, utils.py:246-247)."""
    ss = load_seqset(fname)
    if transform is None:
        variants, lists, seed = [ft.VariantSpec(ft.KIND_CLEAN)], None, 0
    elif isinstance(transform, _DeviceTransform):
        variants, lists, seed = [transform.spec(0)], None, _draw_seed()
    else:
        variants, lists, seed = [ft.VariantSpec(ft.KIND_EXPLICIT, explicit_idx=0)], _explicit_lists_from_callable(fname, ss, transform), 0
    if reduce:
        out = ft.reduced_profiles(ss, k, variants, seed=seed, edit_lists=lists)
    else:
        out = ft.profiles(ss, k, variants, out_kind=ft.OUT_FREQ_F64, seed=seed, edit_lists=lists)
    return list(ss.names), _to_host(out[0])


def reverse_complement(x, k):
    """idelucs/utils.py:191-206: index of the reverse complement of k-mer index x (A0 C1 G2 T3, first base most significant)"""
    x, r = (4 ** k - 1) - int(x), 0
    for _ in range(k):
        r = (r << 2) | (x & 3)
        x >>= 2
    return r


def kmer_rev_comp(kmer_counts, k):
    """idelucs/utils.py:208-221 on a host vector: canonical k-mers (kmer <= reverse complement, increasing) with
    ``(c[kmer] + c[revcomp]) * 0.5`` written back IN PLACE like the reference (an integer array truncates the product);
    returns the canonical entries.  Batches on the device: ``featurise.revcomp_fold``."""
    index = []
    for kmer in range(4 ** k):
        rc = reverse_complement(kmer, k)
        if kmer <= rc:
            index.append(kmer)
            kmer_counts[kmer] += kmer_counts[rc]
            kmer_counts[kmer] *= 0.5
    return kmer_counts[index]


def cgrFasta(fname, k=6, transform=None):
    """idelucs/utils.py:279-318 -> (names, float64[N, 4^k]): FCGR cell frequencies with the +1 pseudocount (the k-mer
    profile of kmersFasta under the fixed cell permutation of idelucs/kmers.pyx:110-123)."""
    ss = load_seqset(fname)
    if transform is None:
        variants, lists, seed = [ft.VariantSpec(ft.KIND_CLEAN)], None, 0
    elif isinstance(transform, _DeviceTransform):
        variants, lists, seed = [transform.spec(0)], None, _draw_seed()
    else:
        variants, lists, seed = [ft.VariantSpec(ft.KIND_EXPLICIT, explicit_idx=0)], _explicit_lists_from_callable(fname, ss, transform), 0
    counts = ft.profiles(ss, k, variants, out_kind=ft.OUT_COUNTS_I32, seed=seed, edit_lists=lists, pseudocount=0)[0]
    # the reference seeds the cell array with ones and cgr() adds the window counts (utils.py:292-295)
    cells = ft.cgr_batch(counts, k, cgr=torch.ones_like(counts))
    return list(ss.names), _to_host(ft.normalize_counts(cells))


def canonical_scaler(ss, k, variants, seed, seq_id0=0, group=None):
    """Scaler of the t_norm slot's float32 canonical rows: the [N, R] matrix is written (OUT_CANON_F32) and fitted by
    idl_colstats like every other matrix, then freed"""
    x0 = ft.profiles(ss, k, variants[:1], out_kind=ft.OUT_CANON_F32, seed=seed, seq_id0=seq_id0)[0]
    return ft.Scaler.fit(x0, group=group)


def augment_device(ss, n_mimics, k=6, seed=None, group=None, seq_id0=0, reduce=False):
    """Device-resident AugmentFasta: returns (profiles float32 [n_mimics+1, N, 4^k] — slot 0 =
    t_norm, slot j = mimic j — standardised with the t_norm statistics, and the Scaler).
    reduce=True: the canonical-k-mer profiles [n_mimics+1, N, R] (utils.py:246-247 applied to every pass)."""
    seed = _draw_seed() if seed is None else seed
    variants = ft.mimic_schedule(n_mimics)
    if reduce:
        sc = canonical_scaler(ss, k, variants, seed, seq_id0, group)
        out = ft.profiles(ss, k, variants, out_kind=ft.OUT_CANON_STD_F32, seed=seed, seq_id0=seq_id0, mean=sc.mean32, scale=sc.scale32)
        return out, sc, seed
    # t_norm statistics (never materialised) and all standardised slots; k = 6: the prepare pass generates the Bernoulli
    # mimics once for both
    out, sc = ft.schedule_profiles(ss, k, variants, out_kind=ft.OUT_STD_F32, seed=seed, seq_id0=seq_id0, group=group)
    return out, sc, seed


def AugmentFasta(sequence_file, n_mimics, k=6, reduce=False):
    """idelucs/utils.py:321-368 -> float32 numpy [n_pairs, 2, 4^k], mimic-major, column 0 =
    standardised t_norm, column 1 = standardised mimic (n_pairs = max(n_mimics, 2) * N)."""
    ss = load_seqset(sequence_file)
    prof, _, _ = augment_device(ss, n_mimics, k=k, reduce=reduce)
    V, n, F = prof.shape
    x = torch.empty((V - 1, n, 2, F), dtype=torch.float32, device=prof.device)
    x[:, :, 0, :] = prof[0].unsqueeze(0)
    x[:, :, 1, :] = prof[1:]
    return _to_host(x.reshape((V - 1) * n, 2, F))


class AugmentedDataset(torch.utils.data.Dataset):
    """idelucs/utils.py:370-389."""

    def __init__(self, data):
        self.data = data

    def __len__(self):
        return self.data.shape[0]

    def __getitem__(self, idx):
        if torch.is_tensor(idx):
            idx = idx.tolist()
        return {"true": self.data[idx, 0, :], "modified": self.data[idx, 1, :]}


class PairBatchLoader(object):
    """Replaces DataLoader(AugmentedDataset, shuffle=True, num_workers=4) (utils.py:422-429):
    yields ``{'true': [B,F], 'modified': [B,F]}`` float32 CUDA tensors.  Pairs are
    (sequence i, mimic j); the pair set is fixed for the whole run like the reference's
    (same seed => same mimic).  When the standardised profiles fit ``materialize_bytes`` they
    are produced once and batches are gathers; otherwise every batch is regenerated from the
    packed sequences by the mimic kernel (selection mode), which gives identical values.
    reduce=True (model_size 'small') follows the same rule with the canonical-k-mer rows (R columns)."""

    def __init__(self, ss, n_mimics, k=6, batch_size=512, seed=None, materialize_bytes=8 << 30, group=None,
                 seq_id0=0, drop_last=False, reduce=False):
        self.ss, self.k, self.batch_size, self.drop_last = ss, k, batch_size, drop_last
        self.variants = ft.mimic_schedule(n_mimics)
        self.n_pairs = (len(self.variants) - 1) * ss.n
        self.seed = _draw_seed() if seed is None else seed
        self.seq_id0 = seq_id0
        self.out_kind = ft.OUT_CANON_STD_F32 if reduce else ft.OUT_STD_F32
        F = ft.canonical_width(k) if reduce else 4 ** k
        if len(self.variants) * ss.n * F * 4 <= materialize_bytes:
            self.profiles, self.scaler, _ = augment_device(ss, n_mimics, k, seed=self.seed, group=group, seq_id0=seq_id0, reduce=reduce)
        else:
            if reduce:
                self.scaler = canonical_scaler(ss, k, self.variants, self.seed, seq_id0, group)
            else:
                self.scaler = ft.profile_stats(ss, k, self.variants[0], seed=self.seed, seq_id0=seq_id0, group=group)
            self.profiles = None

    def __len__(self):
        return self.n_pairs // self.batch_size if self.drop_last else (self.n_pairs + self.batch_size - 1) // self.batch_size

    def batch(self, pair_ids, cta_cap=0):
        """pair id = (mimic-1) * N + sequence  (the reference's mimic-major row order)"""
        n = self.ss.n
        if self.profiles is not None:
            mim = torch.div(pair_ids, n, rounding_mode="floor") + 1
            sidx = pair_ids - (mim - 1) * n
            return {"true": self.profiles[0][sidx], "modified": self.profiles[mim, sidx]}
        # regenerated batch: item = sequence, slots (0, mimic) — the index arithmetic is one launch (idl_pair_selection)
        B = int(pair_ids.numel())
        sidx = torch.empty(B, dtype=torch.int32, device=pair_ids.device)
        sel = torch.empty((B, 2), dtype=torch.int32, device=pair_ids.device)
        ids = pair_ids if (pair_ids.dtype == torch.int64 and pair_ids.is_contiguous()) else pair_ids.to(torch.int64).contiguous()
        lib = _lib.load()
        with torch.cuda.device(pair_ids.device):
            _lib.check(lib.idl_pair_selection(_lib.ptr(ids), B, n, _lib.ptr(sidx), _lib.ptr(sel), _lib.stream_ptr()))
        out = ft.profiles(self.ss, self.k, self.variants, out_kind=self.out_kind, seed=self.seed, sidx=sidx,
                          sel=sel, mean=self.scaler.mean32, scale=self.scaler.scale32, seq_id0=self.seq_id0, cta_cap=cta_cap)
        return {"true": out[0], "modified": out[1], "both": out.view(-1, out.shape[-1])}   # 'both' = the two sides stacked, no copy

    def __iter__(self):
        perm = torch.randperm(self.n_pairs, device=self.ss.device)
        for b in range(len(self)):
            yield self.batch(perm[b * self.batch_size:(b + 1) * self.batch_size])


def create_dataloader(sequence_file, n_mimics, k=6, batch_size=512, GT_file=None, reduce=False):
    """idelucs/utils.py:422-429 -> iterable of {'true','modified'} batches (shuffled every epoch)."""
    return PairBatchLoader(load_seqset(sequence_file), n_mimics, k=k, batch_size=batch_size, reduce=reduce)


def SummaryFasta(fname, GT_file=None):
    """idelucs/utils.py:137-188 -> (names, lengths, ground_truth, cluster_dis)."""
    ss = load_seqset(fname)
    ground_truth = cluster_dis = None
    if GT_file:
        import pandas as pd
        df = pd.read_csv(GT_file, sep="\t")
        gt = dict(zip(df.sequence_id, df.cluster_id))
        cluster_dis = df["cluster_id"].value_counts().to_dict()
        for name in ss.names:
            if name not in gt:
                raise ValueError("Check GT for sequence {}".format(name))
        ground_truth = [gt[name] for name in ss.names]
    return list(ss.names), [int(x) for x in ss.lengths], ground_truth, cluster_dis


class SequenceDataset(torch.utils.data.Dataset):
    """idelucs/utils.py:391-420: clean float64 profiles + their own StandardScaler.  ``kmers``
    is a float64 numpy array like the reference's; ``kmers32`` is the float32 CUDA tensor the
    trainer feeds to the network (models.py:163 casts to float32)."""

    def __init__(self, fasta_file, k=6, transform=None, GT_file=None, reduce=False, group=None):
        self.names, self.lengths, self.GT, self.cluster_dis = SummaryFasta(fasta_file, GT_file)
        ss = load_seqset(fasta_file)
        if transform is None and not reduce:
            f64 = ft.profiles(ss, k, [ft.VariantSpec(ft.KIND_CLEAN)], out_kind=ft.OUT_FREQ_F64)[0]
        elif transform is None:
            f64 = ft.reduced_profiles(ss, k, [ft.VariantSpec(ft.KIND_CLEAN)])[0]
        else:
            f64 = torch.from_numpy(kmersFasta(fasta_file, k, transform, reduce=reduce)[1]).to(ss.device)
        sc = ft.Scaler.fit(f64, group=group)
        self._k64 = sc.transform64(f64)
        self.kmers32 = sc.transform64(f64, want32=True)
        self._kmers = None

    @property
    def kmers(self):
        if self._kmers is None:
            self._kmers = _to_host(self._k64)
        return self._kmers

    def __len__(self):
        return len(self.lengths)

    def __getitem__(self, idx):
        if torch.is_tensor(idx):
            idx = idx.tolist()
        sample = {"kmer": self.kmers[idx, :], "name": self.names[idx]}
        if self.GT:
            sample["cluster_id"] = self.GT[idx]
        return sample


def label_features(predictions, n_clusters):
    """Vote ensemble of idelucs/utils.py:582-602: k-means (k-means++, n_init=10) over the centred one-hot votes of the
    voters; returns (labels, fuzzy membership maxima) — inverse squared distances to the centres, normalised per row."""
    from sklearn.cluster import KMeans
    from sklearn.metrics.pairwise import euclidean_distances
    predictions = np.asarray(predictions)
    n_v, n = predictions.shape
    feats = np.zeros((n, n_v * n_clusters))
    for v in range(n_v):
        for j in range(n_clusters):
            feats[predictions[v] == j, v * n_clusters + j] = 1.0
    feats = feats - np.sum(feats, axis=0) / n
    km = KMeans(n_clusters=n_clusters, init="k-means++", n_init=10)
    y = km.fit_predict(feats)
    with np.errstate(divide="ignore", invalid="ignore"):
        D = 1.0 / euclidean_distances(feats, km.cluster_centers_, squared=True)
        D /= np.sum(D, axis=1)[:, np.newaxis]
    return np.array(y), D.max(axis=1)


def compute_results(y_pred, data, y_true=None, devices=None):
    """idelucs/utils.py:606-625: internal (and, with ground truth, external) clustering metrics -> (dict, assignment).
    A CUDA tensor `data` gets its silhouette score on the GPU (metrics.silhouette_score_device, split over `devices` when
    that is a list of CUDA devices) and its Davies-Bouldin score from sklearn on a float64 host copy; numpy `data` goes to
    sklearn for both."""
    from sklearn import metrics
    if torch.is_tensor(data) and data.is_cuda:
        from .metrics import silhouette_score_device
        host = data.cpu().numpy().astype(np.float64)
        d = {"Davies-Boulding": metrics.davies_bouldin_score(host, y_pred), "Silhouette-Score": silhouette_score_device(data, y_pred, devices)}
    else:
        d = {"Davies-Boulding": metrics.davies_bouldin_score(data, y_pred), "Silhouette-Score": metrics.silhouette_score(data, y_pred)}
    if y_true is not None:
        ext, ind = external_results(y_pred, y_true)
        d.update(ext)
        return d, ind
    return d, None


def external_results(y_pred, y_true):
    """the ground-truth part of compute_results -> ({NMI, ARI, Homogeneity, Completeness, ACC}, assignment)"""
    from sklearn import metrics
    d = {"NMI": metrics.adjusted_mutual_info_score(y_true, y_pred), "ARI": metrics.adjusted_rand_score(y_true, y_pred),
         "Homogeneity": metrics.homogeneity_score(y_true, y_pred), "Completeness": metrics.completeness_score(y_true, y_pred)}
    ind, d["ACC"] = cluster_acc(y_true, y_pred)
    return d, ind


def cluster_acc(y_true, y_pred):
    """Hungarian-matched clustering accuracy (idelucs/utils.py:489-508) -> (assignment, acc)."""
    from scipy.optimize import linear_sum_assignment
    y_true = np.asarray(y_true).astype(np.int64)
    y_pred = np.asarray(y_pred).astype(np.int64)
    D = int(max(y_pred.max(), y_true.max())) + 1
    w = np.zeros((D, D), dtype=np.int64)
    np.add.at(w, (y_pred, y_true), 1)
    rows, cols = linear_sum_assignment(w.max() - w)
    return np.stack([rows, cols], axis=1), float(w[rows, cols].sum()) / y_pred.size
