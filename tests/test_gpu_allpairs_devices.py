"""The HDBSCAN and silhouette all-pairs passes split over several devices (``devices=[...]``) against the one-device result
(``devices=None``) on the same float32 input.  Every row's arithmetic is the same wherever it runs and the MST is unique
under its strict edge order (w, min(i, j), max(i, j)), so every comparison is exact.

A device may appear more than once in the list, so on one GPU ``devices=[0] * P`` exercises all of the splitting, the
per-round reduction over the parts and the combining; the tests that need distinct GPUs skip where there is only one."""
import os
import sys

import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

N_GPUS = torch.cuda.device_count() if torch.cuda.is_available() else 0
needs2 = pytest.mark.skipif(N_GPUS < 2, reason="needs at least 2 GPUs (found %d)" % N_GPUS)

SIZES = [(n, d) for n in (2, 63, 64, 65, 130, 1000, 20011) for d in (1, 3, 64)]
PARTS = (1, 2, 3, 8)


def _blobs(n, d, seed):
    rng = np.random.default_rng(seed)
    c = rng.normal(0.0, 10.0, size=(max(2, n // 50), d))
    return (c[rng.integers(0, len(c), size=n)] + rng.normal(0.0, 1.0, size=(n, d))).astype(np.float32)


def _grid(n, d, seed):
    """integer-grid points with duplicated rows: many equal distances, so many MST weights tie across the parts"""
    rng = np.random.default_rng(seed)
    x = rng.integers(0, 3, size=(n, d)).astype(np.float32)
    x[rng.integers(0, n, size=n // 5)] = x[rng.integers(0, n, size=n // 5)]
    return x


def _ks(n):
    return sorted(k for k in {1, 2, n // 100 + 1, n} if k <= n)


def _labels(n, n_labels, seed):
    return np.random.default_rng(seed).permutation(np.arange(n) % n_labels)


_REF = {}


def _ref(key, fn):
    """the devices=None result, computed once per input"""
    if key not in _REF:
        _REF[key] = fn()
    return _REF[key]


def _mst(x, k, devices):
    from idelucs_b200.hdbscan import core_distances, mreach_mst
    core = core_distances(x, k, devices=devices)
    return tuple(t.cpu() for t in (core,) + mreach_mst(x, core, devices=devices))


def _same_tensors(a, b):
    assert len(a) == len(b)
    for u, v in zip(a, b):
        assert u.dtype == v.dtype and torch.equal(u, v)


def _ids(cases):
    return ["n%d-d%d-P%d" % c for c in cases]


CASES = [(n, d, P) for n, d in SIZES for P in PARTS]


@pytest.mark.parametrize("n,d,P", CASES, ids=_ids(CASES))
def test_core_distances_split_equal_one_device(n, d, P):
    from idelucs_b200.hdbscan import core_distances
    x = torch.from_numpy(_blobs(n, d, seed=n + d)).cuda()
    for k in _ks(n):
        want = _ref(("core", n, d, k), lambda: core_distances(x, k).cpu())
        got = core_distances(x, k, devices=[0] * P)
        assert got.device == x.device
        assert torch.equal(got.cpu(), want), (k, P)


@pytest.mark.parametrize("n,d,P", CASES, ids=_ids(CASES))
def test_mst_split_equal_one_device(n, d, P):
    """src, dst and w element for element and in order"""
    x = torch.from_numpy(_blobs(n, d, seed=n + d)).cuda()
    k = max(n // 100 + 1, 2)
    want = _ref(("mst", n, d), lambda: _mst(x, k, None))
    got = _mst(x, k, [0] * P)
    _same_tensors(got, want)


@pytest.mark.parametrize("n,d,P", CASES, ids=_ids(CASES))
def test_hdbscan_split_equal_one_device(n, d, P):
    from idelucs_b200.hdbscan import hdbscan_device
    x = torch.from_numpy(_blobs(n, d, seed=n + d)).cuda()
    m = max(n // 100 + 1, 2)
    want = _ref(("hdbscan", n, d), lambda: hdbscan_device(x, m))
    labels, probs = hdbscan_device(x, m, devices=[0] * P)
    assert np.array_equal(labels, want[0]) and np.array_equal(probs, want[1])


SIL = [(n, d, P, L) for n, d in SIZES for P in PARTS for L in (2, 7, 200) if L < n]


@pytest.mark.parametrize("n,d,P,L", SIL, ids=["n%d-d%d-P%d-L%d" % c for c in SIL])
def test_silhouette_split_equal_one_device(n, d, P, L):
    from idelucs_b200.metrics import silhouette_samples_device, silhouette_score_device
    x = torch.from_numpy(_blobs(n, d, seed=n + d)).cuda()
    lab = _labels(n, L, seed=n + L)
    want = _ref(("sil", n, d, L), lambda: silhouette_samples_device(x, lab))
    assert np.array_equal(silhouette_samples_device(x, lab, devices=[0] * P), want)
    assert silhouette_score_device(x, lab, devices=[0] * P) == silhouette_score_device(x, lab)


TIES = [(n, d, P) for n, d in ((300, 2), (2000, 3), (5000, 8)) for P in (2, 3, 8)]


@pytest.mark.parametrize("n,d,P", TIES, ids=_ids(TIES))
def test_tie_heavy_inputs_split_equal_one_device(n, d, P):
    """integer grids with duplicated rows: tied weights whose order across the parts decides the tree"""
    from idelucs_b200.hdbscan import hdbscan_device
    from idelucs_b200.metrics import silhouette_samples_device
    xh = _grid(n, d, seed=n + P)
    x = torch.from_numpy(xh).cuda()
    for k in (1, 5, n // 100 + 1):
        want = _mst(x, k, None)
        w = want[3].numpy()
        assert len(w) - len(np.unique(w)) > n // 4   # the input does tie
        _same_tensors(_mst(x, k, [0] * P), want)
    m = n // 100 + 1
    labels, probs = hdbscan_device(x, m, devices=[0] * P)
    ref = hdbscan_device(x, m)
    assert np.array_equal(labels, ref[0]) and np.array_equal(probs, ref[1])
    lab = _labels(n, 7, seed=n)
    assert np.array_equal(silhouette_samples_device(x, lab, devices=[0] * P), silhouette_samples_device(x, lab))


def test_numpy_input_and_device_forms():
    """a numpy latent, and devices given as ints, strings and torch.device"""
    from idelucs_b200.hdbscan import hdbscan_device
    xh = _blobs(3000, 16, seed=4)
    want = hdbscan_device(xh, 31)
    for devices in ([0, 0], ["cuda:0", "cuda"], [torch.device("cuda", 0)] * 3, range(1)):
        got = hdbscan_device(xh, 31, devices=devices)
        assert np.array_equal(got[0], want[0]) and np.array_equal(got[1], want[1]), devices


def test_rejected_device_lists():
    from idelucs_b200.hdbscan import core_distances, hdbscan_device, mreach_mst
    from idelucs_b200.metrics import silhouette_samples_device
    x = torch.from_numpy(_blobs(200, 4, seed=1)).cuda()
    lab = _labels(200, 3, seed=1)
    core = core_distances(x, 3)
    calls = [lambda dv: core_distances(x, 3, devices=dv), lambda dv: mreach_mst(x, core, devices=dv),
             lambda dv: hdbscan_device(x, 3, devices=dv), lambda dv: silhouette_samples_device(x, lab, devices=dv)]
    for call in calls:
        with pytest.raises(ValueError, match=r"^devices must be a non-empty list of CUDA devices$"):
            call([])
        with pytest.raises(ValueError, match=r"^devices must be CUDA devices, got 'cpu'$"):
            call([0, "cpu"])


def test_side_stream_and_current_device_kept():
    """on a non-default stream of the current device: same results, and that stream is still current afterwards"""
    from idelucs_b200.hdbscan import hdbscan_device
    from idelucs_b200.metrics import silhouette_samples_device
    xh = _blobs(4000, 32, seed=9)
    lab = _labels(4000, 7, seed=9)
    want = hdbscan_device(xh, 41), silhouette_samples_device(xh, lab)
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        x = torch.from_numpy(xh).cuda()
        got = hdbscan_device(x, 41, devices=[0] * 3), silhouette_samples_device(x, lab, devices=[0] * 3)
        assert torch.cuda.current_stream() == s and torch.cuda.current_device() == 0
    assert np.array_equal(got[0][0], want[0][0]) and np.array_equal(got[0][1], want[0][1]) and np.array_equal(got[1], want[1])


def test_silhouette_rows_abi_empty_middle_cluster():
    """idl_silhouette_samples_rows over three row ranges (one empty) with label 1 unused equals one idl_silhouette_samples call"""
    from idelucs_b200 import _lib
    lib = _lib.load()
    n, D, L = 1000, 24, 3
    x = torch.from_numpy(_blobs(n, D, seed=3)).cuda()
    lab = torch.from_numpy(np.where(_labels(n, 2, seed=3) == 0, 0, 2).astype(np.int32)).cuda()
    ws = torch.empty(lib.idl_silhouette_workspace_bytes(n, L), dtype=torch.uint8, device="cuda")
    one = torch.empty(n, dtype=torch.float64, device="cuda")
    _lib.check(lib.idl_silhouette_samples(_lib.ptr(x), _lib.ptr(lab), n, D, L, _lib.ptr(one), _lib.ptr(ws), ws.numel(), _lib.stream_ptr()))
    split = torch.full((n,), float("nan"), dtype=torch.float64, device="cuda")
    for b, e in ((0, 333), (333, 333), (333, n)):
        _lib.check(lib.idl_silhouette_samples_rows(_lib.ptr(x), _lib.ptr(lab), n, D, L, b, e, _lib.ptr(split), _lib.ptr(ws), ws.numel(),
                                                   _lib.stream_ptr()))
    assert torch.equal(split, one)


def test_core_rows_abi_leaves_other_rows():
    """idl_core_distances_rows writes its rows only"""
    from idelucs_b200 import _lib
    from idelucs_b200.hdbscan import _workspace, core_distances
    lib = _lib.load()
    n, D = 777, 5
    x = torch.from_numpy(_blobs(n, D, seed=5)).cuda()
    ws = _workspace(x)
    core = torch.full((n,), -1.0, dtype=torch.float64, device="cuda")
    _lib.check(lib.idl_core_distances_rows(_lib.ptr(x), n, D, 8, 100, 300, _lib.ptr(core), _lib.ptr(ws), ws.numel(), _lib.stream_ptr()))
    want = core_distances(x, 8)
    assert torch.equal(core[100:300], want[100:300])
    assert bool((core[:100] == -1).all()) and bool((core[300:] == -1).all())


def test_row_parts_rule():
    from idelucs_b200.hdbscan import row_parts
    assert row_parts(1000, 1) == [(0, 1000)]
    assert row_parts(1000, 4) == [(0, 256), (256, 512), (512, 768), (768, 1000)]   # 16 tiles, 4 each
    assert row_parts(130, 8) == [(0, 0), (0, 0), (0, 64), (64, 64), (64, 64), (64, 128), (128, 128), (128, 130)]
    for n in (1, 63, 64, 65, 20011):
        for P in (1, 2, 3, 8, 100):
            parts = row_parts(n, P)
            assert len(parts) == P and parts[0][0] == 0 and parts[-1][1] == n
            assert all(a[1] == b[0] for a, b in zip(parts, parts[1:]))
            assert all(b % 64 == 0 for b, _ in parts if b < n)


# --- distinct GPUs

MULTI = [[0, 1], [1, 0], "all", [0, 1, 0]]


def _multi(devices):
    return list(range(N_GPUS)) if devices == "all" else devices


@needs2
@pytest.mark.parametrize("devices", MULTI, ids=["0-1", "1-0", "all", "0-1-0"])
def test_distinct_devices_equal_one_device(devices):
    from idelucs_b200.hdbscan import hdbscan_device
    from idelucs_b200.metrics import silhouette_samples_device
    devices = _multi(devices)
    for n, d in ((65, 3), (1000, 64), (20011, 64)):
        x = torch.from_numpy(_blobs(n, d, seed=n + d)).cuda()
        k = n // 100 + 1
        _same_tensors(_mst(x, k, devices), _mst(x, k, None))
        m = max(k, 2)
        got, want = hdbscan_device(x, m, devices=devices), hdbscan_device(x, m)
        assert np.array_equal(got[0], want[0]) and np.array_equal(got[1], want[1])
        lab = _labels(n, 7, seed=n)
        assert np.array_equal(silhouette_samples_device(x, lab, devices=devices), silhouette_samples_device(x, lab))
    x = torch.from_numpy(_grid(3000, 3, seed=1)).cuda()
    _same_tensors(_mst(x, 5, devices), _mst(x, 5, None))


@needs2
def test_input_on_second_device_results_come_back_there():
    from idelucs_b200.hdbscan import core_distances, mreach_mst
    xh = _blobs(2000, 16, seed=2)
    x1 = torch.from_numpy(xh).to("cuda:1")
    core = core_distances(x1, 21, devices=[0, 1])
    src, dst, w = mreach_mst(x1, core, devices=[0])
    assert core.device == x1.device and src.device == x1.device and w.device == x1.device
    _same_tensors((core.cpu(), src.cpu(), dst.cpu(), w.cpu()), _mst(torch.from_numpy(xh).cuda(), 21, None))


@needs2
def test_current_device_and_stream_unchanged():
    from idelucs_b200.hdbscan import core_distances, hdbscan_device, mreach_mst
    from idelucs_b200.metrics import silhouette_samples_device
    xh = _blobs(3000, 8, seed=6)
    lab = _labels(3000, 5, seed=6)
    for dev in (0, 1):
        with torch.cuda.device(dev):
            s = torch.cuda.Stream()
            with torch.cuda.stream(s):
                x = torch.from_numpy(xh).cuda()
                core = core_distances(x, 31, devices=[1, 0])
                assert torch.cuda.current_device() == dev and torch.cuda.current_stream() == s
                mreach_mst(x, core, devices=[0, 1, 0])
                assert torch.cuda.current_device() == dev and torch.cuda.current_stream() == s
                hdbscan_device(x, 31, devices=[1, 0, 1])
                assert torch.cuda.current_device() == dev and torch.cuda.current_stream() == s
                silhouette_samples_device(x, lab, devices=[0, 1])
                assert torch.cuda.current_device() == dev and torch.cuda.current_stream() == s


@needs2
def test_cli_all_devices_equal_one_device(golden_dir, fasta_files, tmp_path, monkeypatch):
    """run(n_clusters=0) splits HDBSCAN and the silhouette over every visible GPU: assignments.tsv and metrics.tsv equal what
    one device computes from the same latent"""
    from idelucs_b200 import __main__ as cli
    from idelucs_b200 import models
    from idelucs_b200.hdbscan import hdbscan_device
    from idelucs_b200.utils import compute_results
    monkeypatch.chdir(tmp_path)
    monkeypatch.setitem(sys.modules, "hdbscan", None)   # import hdbscan -> ImportError: the GPU HDBSCAN
    seen = []
    predict = models.IID_model.predict

    def spy(self, *a, **kw):
        out = predict(self, *a, **kw)
        seen.append(out[2])
        return out
    monkeypatch.setattr(models.IID_model, "predict", spy)
    args = dict(sequence_file=fasta_files["Influenza-A"], GT_file=None, k=6, n_mimics=3, batch_sz=256, optimizer="RMSprop", weight=0.25,
                lr=1e-3, scheduler="None", plot=False, model_size="linear", n_clusters=0, n_epochs=2, n_voters=1)
    args["lambda"] = 2.8
    torch.manual_seed(0)
    np.random.seed(0)
    cli.run(args)
    assert len(seen) == 1 and seen[0].is_cuda
    latent = seen[0]
    n = latent.shape[0]
    labels, probs = hdbscan_device(latent, max(n // 100 + 1, 2))
    y_pred = labels + 1
    out = {f: os.path.join(dp, f) for dp, _, fs in os.walk(str(tmp_path)) for f in fs if f in ("assignments.tsv", "metrics.tsv")}
    rows = [line.rstrip("\n").split("\t") for line in open(out["assignments.tsv"])][1:]
    assert [int(r[1]) for r in rows] == list(y_pred)
    assert [r[2] for r in rows] == [f"{float(p):.6f}" for p in probs]
    assert 1 < len(np.unique(y_pred)) < n, "the run must have a defined silhouette"
    results, _ = compute_results(y_pred, latent, None)
    want = "\t".join(results) + "\n" + "\t".join(repr(float(v)) for v in results.values()) + "\n"
    assert open(out["metrics.tsv"]).read() == want


def test_default_devices_context():
    """inside default_devices a devices=None call splits over the list; outside it computes on the input's device"""
    from idelucs_b200.hdbscan import _parts, default_devices, hdbscan_device
    from idelucs_b200.metrics import silhouette_samples_device
    x = torch.from_numpy(_blobs(1000, 8, seed=8)).cuda()
    lab = _labels(1000, 7, seed=8)
    want = hdbscan_device(x, 11), silhouette_samples_device(x, lab)
    with default_devices([0] * 3):
        assert len(_parts(x, None)) == 3 and len(_parts(x, [0])) == 1
        got = hdbscan_device(x, 11), silhouette_samples_device(x, lab)
    assert len(_parts(x, None)) == 1
    assert np.array_equal(got[0][0], want[0][0]) and np.array_equal(got[0][1], want[0][1]) and np.array_equal(got[1], want[1])
