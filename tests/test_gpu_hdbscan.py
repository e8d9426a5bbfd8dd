"""hdbscan_device and its two kernels against scikit-learn's HDBSCAN (the implementation the --n_clusters 0 path used before):
core distances and MST weights compare by ==, labels and probabilities by array equality."""
import os
import warnings

import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

from sklearn.cluster import HDBSCAN  # noqa: E402
from sklearn.cluster._hdbscan._linkage import mst_from_data_matrix  # noqa: E402
from sklearn.metrics import DistanceMetric  # noqa: E402
from sklearn.neighbors import NearestNeighbors  # noqa: E402


def _blobs(n, d, centers, seed, spread=1.0):
    rng = np.random.default_rng(seed)
    c = rng.normal(0.0, 10.0, size=(centers, d))
    return (c[rng.integers(0, centers, size=n)] + rng.normal(0.0, spread, size=(n, d))).astype(np.float32)


def _with_duplicates(x, seed):
    """every 7th row copied over a random other row: ties and zero distances with multiplicity"""
    rng = np.random.default_rng(seed)
    x = x.copy()
    src = np.arange(0, len(x), 7)
    x[rng.integers(0, len(x), size=len(src))] = x[src]
    return x


def _sk_core(x, k):
    """what sklearn's HDBSCAN computes: a KD-tree kNN query of float64 data, distance to the k-th neighbour"""
    x64 = x.astype(np.float64)
    return NearestNeighbors(n_neighbors=k, algorithm="kd_tree").fit(x64).kneighbors(x64, k)[0][:, -1]


def _device(x):
    return torch.from_numpy(x).cuda()


def _spans(n, src, dst):
    parent = list(range(n))

    def find(a):
        while parent[a] != a:
            parent[a] = parent[parent[a]]
            a = parent[a]
        return a
    for a, b in zip(src, dst):
        ra, rb = find(int(a)), find(int(b))
        if ra == rb:
            return False
        parent[ra] = rb
    return len({find(i) for i in range(n)}) == 1


CORE_CASES = [(n, d, k, dup) for n in (2, 257, 5000) for d in (3, 64) for dup in (False, True)
              for k in sorted({1, 2, 31, n // 100 + 1, n}) if k <= n]


@pytest.mark.parametrize("n,d,k,dup", CORE_CASES, ids=["n%d-d%d-k%d%s" % (n, d, k, "-dup" if dup else "") for n, d, k, dup in CORE_CASES])
def test_core_distances_equal_sklearn(n, d, k, dup):
    from idelucs_b200.hdbscan import core_distances
    x = _blobs(n, d, max(2, n // 50), seed=n + d)
    if dup:
        x = _with_duplicates(x, seed=k)
    got = core_distances(_device(x), k).cpu().numpy()
    assert np.array_equal(got, _sk_core(x, k))


MST_CASES = [(257, 64, 1, False), (257, 3, 5, True), (2000, 64, 1, False), (2000, 37, 21, False), (2000, 64, 21, True), (4000, 64, 41, False)]


@pytest.mark.parametrize("n,d,s,dup", MST_CASES, ids=["n%d-d%d-s%d%s" % (n, d, s, "-dup" if dup else "") for n, d, s, dup in MST_CASES])
def test_mst_weights_equal_sklearn(n, d, s, dup):
    from idelucs_b200.hdbscan import core_distances, mreach_mst
    x = _blobs(n, d, 20, seed=3 * n + s)
    if dup:
        x = _with_duplicates(x, seed=s)
    xd = _device(x)
    core = core_distances(xd, s)
    src, dst, w = (t.cpu().numpy() for t in mreach_mst(xd, core))
    assert len(w) == n - 1 and _spans(n, src, dst)
    ref = HDBSCAN(min_cluster_size=max(s, 2), min_samples=s, copy=True).fit(x.astype(np.float64))._single_linkage_tree_["value"]
    assert np.array_equal(np.sort(w), np.sort(ref))
    # every weight is the mutual-reachability distance of its own edge
    c = core.cpu().numpy()
    x64 = x.astype(np.float64)
    d2 = np.zeros(n - 1)
    for t in range(d):   # sequential sum, like sklearn's EuclideanDistance
        diff = x64[src, t] - x64[dst, t]
        d2 = d2 + diff * diff
    assert np.array_equal(w, np.maximum(np.maximum(c[src], c[dst]), np.sqrt(d2)))


@pytest.mark.parametrize("n,d", [(1000, 64), (3000, 16)])
def test_mst_edges_equal_prim_without_ties(n, d):
    """min_samples = 1 (core distance 0) on continuous random data: all weights distinct, so the MST is unique"""
    from idelucs_b200.hdbscan import core_distances, mreach_mst
    x = np.random.default_rng(n).random((n, d), dtype=np.float32)
    xd = _device(x)
    core = core_distances(xd, 1)
    src, dst, w = (t.cpu().numpy() for t in mreach_mst(xd, core))
    assert len(np.unique(w)) == n - 1
    ref = mst_from_data_matrix(x.astype(np.float64), core.cpu().numpy(), DistanceMetric.get_metric("euclidean"), 1.0)
    edges = {(min(a, b), max(a, b)): wt for a, b, wt in zip(ref["current_node"], ref["next_node"], ref["distance"])}
    assert edges == {(min(int(a), int(b)), max(int(a), int(b))): wt for a, b, wt in zip(src, dst, w)}
    # oriented like Prim's edges from point 0: the first endpoint is the parent
    assert {(int(a), int(b)) for a, b in zip(src, dst)} == {(int(a), int(b)) for a, b in zip(ref["current_node"], ref["next_node"])}


def _compare_with_sklearn(x, min_cluster_size, min_samples=None, latent=None):
    """labels and probabilities of hdbscan_device (on `latent`, default: x on the device) and of sklearn.  sklearn's own labels
    depend on the order of tied MST weights (it sorts its Prim-ordered edges with an unstable argsort), so where they differ
    the test shows that the two MSTs agree except for that order: same weights, same edges wherever a weight is unique, and
    (when the edge sets are equal) sklearn's labels again once the device edges are put in sklearn's order."""
    from idelucs_b200.hdbscan import core_distances, hdbscan_device, labels_from_mst, mreach_mst
    dev = _device(x) if latent is None else latent
    labels, probs = hdbscan_device(dev, min_cluster_size, min_samples)
    x64 = x.astype(np.float64)
    sk = HDBSCAN(min_cluster_size=min_cluster_size, min_samples=min_samples, copy=True).fit(x64)
    if np.array_equal(labels, sk.labels_) and np.array_equal(probs, sk.probabilities_):
        return
    k = min_cluster_size if min_samples is None else min_samples
    core = core_distances(dev, k)
    src, dst, w = (t.cpu().numpy() for t in mreach_mst(dev, core))
    ref = mst_from_data_matrix(x64, core.cpu().numpy(), DistanceMetric.get_metric("euclidean"), 1.0)
    assert np.array_equal(np.sort(w), np.sort(ref["distance"]))
    ties = len(w) - len(np.unique(w))
    assert ties > 0, "labels differ from sklearn's without any tied MST weight"
    ours = {(int(a), int(b)): wt for a, b, wt in zip(src, dst, w)}
    theirs = {(int(a), int(b)): wt for a, b, wt in zip(ref["current_node"], ref["next_node"], ref["distance"])}
    # two spanning trees of equal total order statistics that differ only by exchanging edges of equal weight
    assert sorted(ours[e] for e in set(ours) - set(theirs)) == sorted(theirs[e] for e in set(theirs) - set(ours))
    if ours == theirs:   # the device's edges in sklearn's Prim order: labels_from_mst then sorts them exactly as sklearn does
        l2, p2 = labels_from_mst(ref["current_node"], ref["next_node"],
                                 np.array([ours[(int(a), int(b))] for a, b in zip(ref["current_node"], ref["next_node"])]), min_cluster_size)
        assert np.array_equal(l2, sk.labels_) and np.array_equal(p2, sk.probabilities_)
    warnings.warn("labels differ from sklearn's at %d points; the MST has %d tied weights; edge sets equal: %s"
                  % (int((labels != sk.labels_).sum()), ties, ours == theirs))


def test_labels_blobs_cli_parameters():
    n = 20000
    x = _blobs(n, 64, 200, seed=7)
    _compare_with_sklearn(x, n // 100 + 1)


@pytest.mark.parametrize("m", [5, 15, 40])
def test_labels_tie_free_random(m):
    """min_samples = 1 on continuous random data: every mutual-reachability weight is a distinct distance"""
    x = np.random.default_rng(m).random((3000, 8), dtype=np.float32)
    _compare_with_sklearn(x, m, 1)


def _trained_latent(fasta, n_epochs=4):
    from idelucs_b200 import models
    from idelucs_b200.utils import SummaryFasta
    torch.manual_seed(0)
    np.random.seed(0)
    args = dict(sequence_file=fasta, GT_file=None, n_clusters=200, k=6, n_mimics=3, batch_sz=256, optimizer="RMSprop", weight=0.25,
                lr=1e-3, model_size="linear", scheduler="None", n_epochs=n_epochs, n_voters=1)
    args["lambda"] = 2.8
    model = models.IID_model(args)
    model.names, model.lengths, model.GT, model.cluster_dis = SummaryFasta(model.sequence_file, model.GT_file)
    model.build_dataloader()
    for _ in range(n_epochs):
        model.contrastive_training_epoch()
    latent = model.predict(device_latent=True)[2]
    assert latent.is_cuda and latent.dtype == torch.float32
    return latent


@pytest.mark.parametrize("stem", ["Influenza-A", "Actinopterygii"])
def test_labels_trained_latent(fasta_files, stem):
    latent = _trained_latent(fasta_files[stem])
    n = latent.shape[0]
    _compare_with_sklearn(latent.cpu().numpy(), max(n // 100 + 1, 2), latent=latent)


@pytest.mark.parametrize("args,text", [
    (dict(min_cluster_size=1), "The 'min_cluster_size' parameter of HDBSCAN must be an int in the range [2, inf). Got 1 instead."),
    (dict(min_cluster_size=5, min_samples=0), "The 'min_samples' parameter of HDBSCAN must be an int in the range [1, inf) or None. Got 0 instead."),
    (dict(min_cluster_size=5, min_samples=11), "min_samples (11) must be at most the number of samples in X (10)"),
    (dict(min_cluster_size=11), "min_samples (11) must be at most the number of samples in X (10)"),
])
def test_parameter_errors(args, text):
    from idelucs_b200.hdbscan import hdbscan_device
    with pytest.raises(ValueError) as e:
        hdbscan_device(np.random.default_rng(0).random((10, 4), dtype=np.float32), **args)
    assert str(e.value) == text


def test_single_sample_and_non_finite_errors():
    from idelucs_b200.hdbscan import hdbscan_device
    with pytest.raises(ValueError, match=r"^n_samples=1 while HDBSCAN requires more than one sample$"):
        hdbscan_device(torch.ones((1, 4), device="cuda"), 2)
    x = torch.rand((50, 4), device="cuda")
    x[3, 1] = float("nan")
    with pytest.raises(ValueError, match=r"^Input X contains NaN\.$"):
        hdbscan_device(x, 2)
    x[3, 1] = float("inf")
    with pytest.raises(ValueError, match=r"^Input X contains infinity"):
        hdbscan_device(x.cpu().numpy(), 2)


def test_cli_default_mode_writes_sklearn_labels(golden_dir, fasta_files, tmp_path, monkeypatch):
    """run(n_clusters=0) without the hdbscan package: assignments.tsv holds sklearn's HDBSCAN labels (+1) of the latent"""
    import sys
    from idelucs_b200 import __main__ as cli
    from idelucs_b200 import models
    monkeypatch.chdir(tmp_path)
    monkeypatch.setitem(sys.modules, "hdbscan", None)   # import hdbscan -> ImportError
    seen = []
    predict = models.IID_model.predict

    def spy(self, *a, **kw):
        out = predict(self, *a, **kw)
        seen.append(out[2])
        return out
    monkeypatch.setattr(models.IID_model, "predict", spy)
    base = dict(sequence_file=fasta_files["Actinopterygii"], GT_file=os.path.join(golden_dir, "Actinopterygii_GT.tsv"), k=6, n_mimics=3,
                batch_sz=256, optimizer="RMSprop", weight=0.25, lr=1e-3, scheduler="None", plot=False, model_size="linear")
    base["lambda"] = 2.8
    torch.manual_seed(0)
    np.random.seed(0)
    cli.run(dict(base, n_clusters=0, n_epochs=4, n_voters=1))
    assert len(seen) == 1 and torch.is_tensor(seen[0]) and seen[0].is_cuda
    latent = seen[0].cpu().numpy().astype(np.float64)
    sk = HDBSCAN(min_cluster_size=max(len(latent) // 100 + 1, 2), copy=True).fit(latent)
    out = [os.path.join(dp, f) for dp, _, fs in os.walk(str(tmp_path)) for f in fs if f == "assignments.tsv"]
    assert len(out) == 1
    rows = [line.rstrip("\n").split("\t") for line in open(out[0])][1:]
    assert [int(r[1]) for r in rows] == list(sk.labels_ + 1)
    assert [r[2] for r in rows] == [f"{float(p):.6f}" for p in sk.probabilities_]
