"""silhouette_samples_device / silhouette_score_device and the CLI's metrics.tsv.

The per-sample values compare by == with a numpy oracle that follows the arithmetic contract of idl_silhouette_samples
(include/idelucs_b200.h): fp64 distances summed in order over the dimensions, cluster sums as sequential folds in index
order.  Against sklearn, which forms its distances with a matrix product, they agree within 1e-9 on duplicate-free data."""
import os
import sys

import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

from sklearn import metrics as skm  # noqa: E402


def _blobs(n, d, centers, seed, spread=1.0):
    """(float32 [n, d] points, int64 [n] index of the centre each point was drawn around)"""
    rng = np.random.default_rng(seed)
    c = rng.normal(0.0, 10.0, size=(centers, d))
    lab = rng.integers(0, centers, size=n)
    return (c[lab] + rng.normal(0.0, spread, size=(n, d))).astype(np.float32), lab


def _oracle(x, labels, rows=None, block=256):
    """silhouette of the given rows (default: all) by the contract of idl_silhouette_samples"""
    x64 = x.astype(np.float64)
    n, D = x64.shape
    _, enc = np.unique(labels, return_inverse=True)
    m = int(enc.max()) + 1
    members = [np.flatnonzero(enc == c) for c in range(m)]   # increasing index order
    size = np.array([len(p) for p in members])
    rows = np.arange(n) if rows is None else np.asarray(rows)
    out = np.zeros(len(rows))
    for b0 in range(0, len(rows), block):
        rb = rows[b0:b0 + block]
        d2 = np.zeros((len(rb), n))
        for t in range(D):   # sequential sum over the dimensions
            diff = x64[rb, t][:, None] - x64[None, :, t]
            d2 = d2 + diff * diff
        d = np.sqrt(d2)
        S = np.stack([np.cumsum(d[:, p], axis=1)[:, -1] if len(p) else np.zeros(len(rb)) for p in members], axis=1)
        for q, i in enumerate(rb):
            own = enc[i]
            if size[own] == 1:
                continue
            intra = S[q, own] / (size[own] - 1)
            inter = min(S[q, c] / size[c] for c in range(m) if c != own and size[c] > 0)
            with np.errstate(invalid="ignore"):
                s = (inter - intra) / max(intra, inter)
            out[b0 + q] = 0.0 if np.isnan(s) else s
    return out


def _distances(x):
    """the exact [n, n] distance matrix of the contract (fp64, sequential over the dimensions)"""
    x64 = x.astype(np.float64)
    d2 = np.zeros((len(x64), len(x64)))
    for t in range(x64.shape[1]):
        diff = x64[:, t][:, None] - x64[None, :, t]
        d2 = d2 + diff * diff
    return np.sqrt(d2)


def _device(x):
    return torch.from_numpy(x).cuda()


def _weird(labels, seed):
    """the same partition under unsorted, non-contiguous, negative label values"""
    values = np.random.default_rng(seed).permutation(np.arange(len(np.unique(labels))) * 7 - 5)
    return values[np.unique(labels, return_inverse=True)[1]]


CASES = []
for n in (3, 64, 65, 257, 5000):
    for d in ((1, 3, 64, 100) if n < 5000 else (3, 64)):
        CASES.append((n, d, 2, "blobs"))
        if n > 200:
            CASES.append((n, d, 200, "blobs"))
        if n <= 257 and n > 3:
            CASES.append((n, d, n - 1, "blobs"))
CASES += [(5000, 64, 2, "weird"), (5000, 64, 200, "weird"), (257, 3, 2, "noise"), (5000, 16, 40, "noise"),
          (1000, 8, 2, "sorted"), (1000, 8, 10, "dup"), (1000, 8, 10, "dup_all"), (300, 5, 3, "equal_rows")]


def _case_data(n, d, k, kind):
    x, lab = _blobs(n, d, min(k, n), seed=31 * n + d + k)
    if kind == "blobs" and k >= n - 1:   # n - 1 clusters: one pair, every other point alone
        lab = np.arange(n)
        lab[-1] = 0
    if kind == "blobs" and len(np.unique(lab)) < 2:
        lab[0] = 1 - lab[0]
    if kind == "weird":
        lab = _weird(lab, n + k)
    if kind == "noise":   # -1 for about a fifth of the points, as HDBSCAN labels noise
        lab = _weird(lab, k)
        lab[np.random.default_rng(k).random(n) < 0.2] = -1
    if kind == "sorted":   # clusters of 500 contiguous points: each one spans many column tiles
        lab = np.arange(n) // 500
    if kind == "dup":   # duplicate rows, mostly in other clusters: zero distances across clusters
        src = np.arange(0, n, 3)
        x[np.random.default_rng(n).permutation(n)[:len(src)]] = x[src]
    if kind == "dup_all":   # every point of the first half has a twin in another cluster
        src = np.arange(n // 2)
        x[src + n // 2] = x[src]
        lab[src + n // 2] = (lab[src] + 1) % k
    if kind == "equal_rows":   # every distance is 0: intra = inter = 0 -> 0
        x[:] = x[0]
    return x, lab


@pytest.mark.parametrize("n,d,k,kind", CASES, ids=["n%d-d%d-c%d-%s" % c for c in CASES])
def test_samples_equal_oracle(n, d, k, kind):
    from idelucs_b200.metrics import silhouette_samples_device
    x, lab = _case_data(n, d, k, kind)
    got = silhouette_samples_device(_device(x), lab)
    assert got.dtype == np.float64 and got.shape == (n,)
    ref = _oracle(x, lab)
    bad = np.flatnonzero(got != ref)
    assert len(bad) == 0, (bad[:5], got[bad[:5]], ref[bad[:5]])
    if kind == "equal_rows":
        assert np.all(got == 0.0)


def test_samples_at_scale_equal_oracle():
    from idelucs_b200.metrics import silhouette_samples_device
    n = 300000
    x, lab = _blobs(n, 64, 200, seed=5)
    got = silhouette_samples_device(_device(x), lab)
    rows = np.random.default_rng(1).choice(n, size=64, replace=False)
    assert np.array_equal(got[rows], _oracle(x, lab, rows))


@pytest.mark.parametrize("n,k", [(2000, 2), (3000, 60), (20000, 200)])
def test_samples_and_score_agree_with_sklearn(n, k):
    from idelucs_b200.metrics import silhouette_samples_device, silhouette_score_device
    x, lab = _blobs(n, 64, k, seed=n + k)
    assert len(np.unique(x, axis=0)) == n
    got = silhouette_samples_device(_device(x), lab)
    assert np.max(np.abs(got - skm.silhouette_samples(x.astype(np.float64), lab))) <= 1e-9
    score = silhouette_score_device(x, lab)   # numpy input: rounded to float32, which x already is
    assert isinstance(score, float) and abs(score - skm.silhouette_score(x.astype(np.float64), lab)) <= 1e-9
    assert score == float(np.mean(got))


def test_repeatable():
    from idelucs_b200.metrics import silhouette_samples_device
    x, lab = _blobs(5000, 64, 200, seed=2)
    xd = _device(x)
    a, b = silhouette_samples_device(xd, lab), silhouette_samples_device(xd, lab)
    assert a.tobytes() == b.tobytes()


def test_label_count_errors():
    from idelucs_b200.metrics import silhouette_samples_device, silhouette_score_device
    x = torch.rand((10, 4), device="cuda")
    with pytest.raises(ValueError) as e:
        silhouette_samples_device(x, np.zeros(10, dtype=np.int64))
    assert str(e.value) == "Number of labels is 1. Valid values are 2 to n_samples - 1 (inclusive)"
    with pytest.raises(ValueError) as e:
        silhouette_score_device(x, np.arange(10))
    assert str(e.value) == "Number of labels is 10. Valid values are 2 to n_samples - 1 (inclusive)"


def test_input_errors():
    from idelucs_b200.metrics import silhouette_samples_device
    x = torch.rand((50, 4), device="cuda")
    lab = np.arange(50) % 3
    with pytest.raises(ValueError, match=r"^Found input variables with inconsistent numbers of samples: \[50, 49\]$"):
        silhouette_samples_device(x, lab[:49])
    x[3, 1] = float("nan")
    with pytest.raises(ValueError, match=r"^Input X contains NaN\.$"):
        silhouette_samples_device(x, lab)
    x[3, 1] = float("inf")
    with pytest.raises(ValueError, match=r"^Input X contains infinity"):
        silhouette_samples_device(x.cpu().numpy(), lab)


def test_out_of_range_label_rejected_before_any_launch():
    from idelucs_b200 import _lib
    lib = _lib.load()
    n, D, m = 100, 8, 3
    x = torch.rand((n, D), device="cuda")
    lab = torch.from_numpy((np.arange(n) % m).astype(np.int32)).cuda()
    lab[37] = m
    out = torch.full((n,), 7.0, dtype=torch.float64, device="cuda")
    ws = torch.empty(lib.idl_silhouette_workspace_bytes(n, m), dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()
    launches = lib.idl_launch_count()
    rc = lib.idl_silhouette_samples(_lib.ptr(x), _lib.ptr(lab), n, D, m, _lib.ptr(out), _lib.ptr(ws), ws.numel(), _lib.stream_ptr())
    assert rc == 1
    assert lib.idl_last_error().decode() == "idl_silhouette_samples: label 3 outside 0..2 at position 37"
    lab[37] = -1
    rc = lib.idl_silhouette_samples(_lib.ptr(x), _lib.ptr(lab), n, D, m, _lib.ptr(out), _lib.ptr(ws), ws.numel(), _lib.stream_ptr())
    assert rc == 1 and lib.idl_last_error().decode() == "idl_silhouette_samples: label -1 outside 0..2 at position 37"
    assert lib.idl_launch_count() == launches and bool((out == 7.0).all())


def test_compute_results_on_device_matches_numpy():
    from idelucs_b200.utils import compute_results
    x, lab = _blobs(4000, 64, 30, seed=9)
    y_true = (lab + np.random.default_rng(3).integers(0, 2, size=len(lab))) % 30   # a noisy ground truth
    x64 = x.astype(np.float64)
    for gt in (None, y_true):
        got, got_ind = compute_results(lab, _device(x), gt)
        ref, ref_ind = compute_results(lab, x64, gt)
        assert list(got) == list(ref)
        for key in ("Davies-Boulding", "Silhouette-Score"):
            assert abs(got[key] - ref[key]) <= 1e-9, key
        for key in set(ref) - {"Davies-Boulding", "Silhouette-Score"}:
            assert got[key] == ref[key], key
        assert (got_ind is None and ref_ind is None) or np.array_equal(np.asarray(got_ind), np.asarray(ref_ind))


def _cli_run(golden_dir, fasta_files, tmp_path, monkeypatch, n_clusters, n_voters):
    """run() on Actinopterygii with its GT file -> (y_pred, last latent the CLI saw, y_true, assignments rows, metrics.tsv lines)"""
    from idelucs_b200 import __main__ as cli
    from idelucs_b200 import models
    out_root = tmp_path / ("run%d" % n_clusters)
    out_root.mkdir()
    monkeypatch.chdir(out_root)
    monkeypatch.setitem(sys.modules, "hdbscan", None)   # import hdbscan -> ImportError: the device path
    seen = []
    predict = models.IID_model.predict

    def spy(self, *a, **kw):
        out = predict(self, *a, **kw)
        seen.append(out[2])
        return out
    monkeypatch.setattr(models.IID_model, "predict", spy)
    gt = os.path.join(golden_dir, "Actinopterygii_GT.tsv")
    args = dict(sequence_file=fasta_files["Actinopterygii"], GT_file=gt, k=6, n_mimics=3, batch_sz=256, optimizer="RMSprop", weight=0.25,
                lr=1e-3, scheduler="None", plot=False, model_size="linear", n_clusters=n_clusters, n_epochs=4, n_voters=n_voters)
    args["lambda"] = 2.8
    torch.manual_seed(0)
    np.random.seed(0)
    y_pred = cli.run(args)
    assert len(seen) == n_voters and all(torch.is_tensor(t) and t.is_cuda for t in seen)
    found = {f: os.path.join(dp, f) for dp, _, fs in os.walk(str(out_root)) for f in fs}
    assert set(found) == {"assignments.tsv", "metrics.tsv"}
    assert os.path.dirname(found["assignments.tsv"]) == os.path.dirname(found["metrics.tsv"])
    rows = [line.rstrip("\n").split("\t") for line in open(found["assignments.tsv"])]
    lines = open(found["metrics.tsv"]).read().splitlines()
    from idelucs_b200.utils import SummaryFasta
    true = SummaryFasta(fasta_files["Actinopterygii"], gt)[2]
    ids = {c: i for i, c in enumerate(sorted(set(true)))}
    return np.asarray(y_pred), seen[-1], np.array([ids[c] for c in true]), rows, lines


@pytest.mark.parametrize("n_clusters,n_voters", [(0, 1), (3, 2)])
def test_cli_writes_metrics_tsv(golden_dir, fasta_files, tmp_path, monkeypatch, capsys, n_clusters, n_voters):
    from idelucs_b200.utils import cluster_acc, compute_results
    y_pred, latent, y_true, rows, lines = _cli_run(golden_dir, fasta_files, tmp_path, monkeypatch, n_clusters, n_voters)
    latent64 = latent.cpu().numpy().astype(np.float64)
    # assignments.tsv: the format and labels of before
    assert rows[0] == ["sequence_id", "assignment", "confidence_score"] and len(rows) == 1 + len(y_pred)
    assert [int(r[1]) for r in rows[1:]] == list(y_pred)
    if n_clusters == 0:
        from sklearn.cluster import HDBSCAN
        sk = HDBSCAN(min_cluster_size=max(len(latent64) // 100 + 1, 2), copy=True).fit(latent64)
        assert list(y_pred) == list(sk.labels_ + 1)
    ref, _ = compute_results(y_pred, latent64, y_true)
    assert len(lines) == 2 and lines[0].split("\t") == list(ref)
    got = dict(zip(lines[0].split("\t"), (float(v) for v in lines[1].split("\t"))))
    assert lines[1].split("\t") == [repr(v) for v in got.values()]
    for key in ref:
        if key != "Silhouette-Score":   # Davies-Bouldin and the ground-truth metrics: the same sklearn calls on the same data
            assert got[key] == ref[key], key
    # Actinopterygii holds duplicate sequences, whose latents are identical rows.  sklearn's GEMM distances
    # (|x|^2 - 2 x.y + |y|^2) put them about 3e-7 apart instead of 0, so its score differs from the exact one by ~1e-8.
    # The exact score: the oracle by ==, and sklearn's own formula on the exact distances
    sil = got["Silhouette-Score"]
    assert sil == float(np.mean(_oracle(latent.cpu().numpy(), y_pred)))
    assert abs(sil - skm.silhouette_score(_distances(latent.cpu().numpy()), y_pred, metric="precomputed")) <= 1e-12
    assert abs(sil - ref["Silhouette-Score"]) <= 1e-6
    printed = capsys.readouterr().out
    assert f"ACC \t {cluster_acc(y_true, y_pred)[1]:.5f}\n" in printed
    assert f"ARI \t {skm.adjusted_rand_score(y_true, y_pred):.5f}\nNMI \t {skm.adjusted_mutual_info_score(y_true, y_pred):.5f}\n" in printed
    assert f"Silhouette \t {got['Silhouette-Score']:.5f}\nDavies-Bouldin \t {got['Davies-Boulding']:.5f}\n" in printed


def test_cli_single_cluster_writes_nan(golden_dir, fasta_files, tmp_path, monkeypatch, capsys):
    """HDBSCAN calls every point noise: one label, so no silhouette or Davies-Bouldin; the run still finishes"""
    from idelucs_b200 import hdbscan as hd
    from idelucs_b200.utils import external_results
    monkeypatch.setattr(hd, "hdbscan_device", lambda latent, mcs, ms=None: (np.full(latent.shape[0], -1), np.zeros(latent.shape[0])))
    y_pred, _, y_true, rows, lines = _cli_run(golden_dir, fasta_files, tmp_path, monkeypatch, 0, 1)
    assert set(y_pred) == {0} and [r[1] for r in rows[1:]] == ["0"] * len(y_pred)
    ext, _ = external_results(y_pred, y_true)
    assert lines[0].split("\t") == ["Davies-Boulding", "Silhouette-Score"] + list(ext)
    assert lines[1].split("\t") == ["nan", "nan"] + [repr(float(v)) for v in ext.values()]
    printed = capsys.readouterr().out
    assert "Silhouette \t nan\nDavies-Bouldin \t nan\n" in printed
    assert "Silhouette and Davies-Bouldin need 2 to %d clusters, got 1: written as nan\n" % (len(y_pred) - 1) in printed
