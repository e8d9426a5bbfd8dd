"""HDBSCAN of the latent space (idelucs/__main__.py:149-156, the --n_clusters 0 mode) with its all-pairs work on the GPU.

Results equal ``sklearn.cluster.HDBSCAN(min_cluster_size, min_samples).fit(X)`` (Euclidean metric, alpha 1, excess-of-mass
selection): idl_core_distances and idl_mreach_mst compute the core distances and the mutual-reachability minimum spanning
tree with sklearn's own fp64 arithmetic, and sklearn's host code (make_single_linkage, tree_to_labels) turns the tree into
labels and probabilities, exactly as sklearn's ``_process_mst`` and ``fit`` do.  Ties between MST weights are the only
source of a difference: sklearn orders tied edges by an unstable argsort of its Prim order, this module by an unstable
argsort of the Borůvka order.

Every entry point takes ``devices``: None computes on the input's device; a list of CUDA devices (a device may appear more
than once) splits the rows of every all-pairs pass into contiguous parts (``row_parts``), one per entry, each on its device
with its own replica of the data.  Every row's arithmetic is the same wherever it runs and the MST is unique under its
strict edge order, so the results are bit-identical to one device's.  Inside ``default_devices(list)`` a call with
devices=None uses that list."""
import contextlib
import contextvars
import ctypes

import numpy as np

from . import _lib

_SK = "HDBSCAN"   # sklearn's parameter-validation texts name the estimator


def _as_device_matrix(latent):
    import torch
    x = latent if torch.is_tensor(latent) else torch.from_numpy(np.ascontiguousarray(latent))
    if x.dim() != 2:
        raise ValueError("expected a 2-d [N, D] latent matrix, got shape %s" % (tuple(x.shape),))
    dev = x.device if x.is_cuda else torch.device("cuda", torch.cuda.current_device())
    # values are rounded to float32 (the dtype of the model's latent); float32 data keeps sklearn's float64 results
    return x.to(device=dev, dtype=torch.float32).contiguous()


def _check_finite(x):
    import torch
    if not bool(torch.isfinite(x).all()):
        if bool(torch.isnan(x).any()):
            raise ValueError("Input X contains NaN.")
        raise ValueError("Input X contains infinity or a value too large for dtype('float32').")


def _workspace(x):
    import torch
    n, D = x.shape
    return torch.empty(_lib.load().idl_hdbscan_workspace_bytes(n, D), dtype=torch.uint8, device=x.device)


def row_parts(n, n_parts):
    """[(row_begin, row_end)] of n_parts contiguous parts of the rows 0..n-1: equal shares of the 64-row tiles the all-pairs
    kernels give one CTA each (part p takes tiles p T // n_parts .. (p + 1) T // n_parts - 1 of T = ceil(n / 64)); parts
    beyond the number of tiles are empty"""
    tiles = -(-n // 64)
    cut = [min(n, 64 * (p * tiles // n_parts)) for p in range(n_parts + 1)]
    return list(zip(cut[:-1], cut[1:]))


_DEFAULT_DEVICES = contextvars.ContextVar("idelucs_b200_default_devices", default=None)


@contextlib.contextmanager
def default_devices(devices):
    """Within the block, the entry points of this module and of ``metrics`` that are called with devices=None split over
    `devices`.  The CLI uses it so that its hdbscan_device call keeps the (latent, min_cluster_size) form that replacements
    of hdbscan_device rely on."""
    token = _DEFAULT_DEVICES.set(None if devices is None else list(devices))
    try:
        yield
    finally:
        _DEFAULT_DEVICES.reset(token)


def _parts(x, devices):
    """[(torch.device, row_begin, row_end)] of every part: one part on x's device for devices=None (outside
    default_devices), else the rows split by row_parts over the given list of CUDA devices (ints, strings or torch.device;
    repeats allowed)"""
    import torch
    n = x.shape[0]
    devices = _DEFAULT_DEVICES.get() if devices is None else devices
    if devices is None:
        return [(x.device, 0, n)]
    devs = []
    for d in devices:
        dev = torch.device(d)
        if dev.type != "cuda":
            raise ValueError("devices must be CUDA devices, got %r" % (d,))
        devs.append(torch.device("cuda", torch.cuda.current_device()) if dev.index is None else dev)
    if not devs:
        raise ValueError("devices must be a non-empty list of CUDA devices")
    return [(d, b, e) for d, (b, e) in zip(devs, row_parts(n, len(devs)))]


def _workspaces(xs, parts, ws=None):
    """one workspace per part; a caller's ws serves a single part on its device"""
    if ws is not None and len(parts) == 1 and parts[0][0] == ws.device:
        return [ws]
    return [_workspace(xs[d]) for d, _, _ in parts]


def _replicas(t, parts):
    """{device: t on that device} for every distinct device of the parts"""
    return {d: t if t.device == d else t.to(d) for d, _, _ in parts}


def _core_parts(xs, parts, k, wss):
    """every part's rows of the core distances on its device, then the other parts' slices copied into each device's array
    -> {device: full float64 [N] core}"""
    import torch
    lib = _lib.load()
    n, D = next(iter(xs.values())).shape
    cores = {d: torch.empty(n, dtype=torch.float64, device=d) for d in xs}
    for (d, b, e), ws in zip(parts, wss):
        with torch.cuda.device(d):
            _lib.check(lib.idl_core_distances_rows(_lib.ptr(xs[d]), n, D, int(k), b, e, _lib.ptr(cores[d]), _lib.ptr(ws), ws.numel(),
                                                   _lib.stream_ptr()))
    for d, b, e in parts:
        for d2 in cores:
            if d2 != d and e > b:
                cores[d2][b:e].copy_(cores[d][b:e])
    return cores


def _mst_parts(xs, cores, parts, wss):
    """idl_mreach_mst_parts -> (src, dst, w) on the first part's device"""
    import torch
    n, D = next(iter(xs.values())).shape
    out = parts[0][0]
    src = torch.empty(n - 1, dtype=torch.int64, device=out)
    dst = torch.empty(n - 1, dtype=torch.int64, device=out)
    w = torch.empty(n - 1, dtype=torch.float64, device=out)
    P = len(parts)

    def arr(ctype, values):
        return (ctype * P)(*values)
    _lib.check(_lib.load().idl_mreach_mst_parts(
        P, arr(ctypes.c_int, [d.index for d, _, _ in parts]), arr(ctypes.c_void_p, [xs[d].data_ptr() for d, _, _ in parts]),
        arr(ctypes.c_void_p, [cores[d].data_ptr() for d, _, _ in parts]), arr(ctypes.c_int64, [b for _, b, _ in parts]),
        arr(ctypes.c_int64, [e for _, _, e in parts]), n, D, _lib.ptr(src), _lib.ptr(dst), _lib.ptr(w),
        arr(ctypes.c_void_p, [ws.data_ptr() for ws in wss]), arr(ctypes.c_size_t, [ws.numel() for ws in wss]),
        arr(ctypes.c_void_p, [torch.cuda.current_stream(d).cuda_stream for d, _, _ in parts])))
    return src, dst, w


def core_distances(x, k, ws=None, devices=None):
    """float64 [N] CUDA tensor on x's device: the distance of every row of the float32 CUDA matrix x to its k-th nearest row,
    itself included (NearestNeighbors.kneighbors(X, k)[0][:, -1]).  ws: a workspace (_workspace(x)), used when there is
    one part on its device; devices: see the module text."""
    parts = _parts(x, devices)
    xs = _replicas(x, parts)
    wss = _workspaces(xs, parts, ws)
    cores = _core_parts(xs, parts, k, wss)
    return cores[x.device] if x.device in cores else cores[parts[0][0]].to(x.device)


def mreach_mst(x, core, ws=None, devices=None):
    """the N-1 edges (src int64, dst int64, weight float64; CUDA tensors on x's device, Borůvka order) of the minimum
    spanning tree of the mutual-reachability graph max(core[i], core[j], d(i, j)) of the float32 CUDA matrix x.  ws: a
    workspace (_workspace(x)), used when there is one part on its device; devices: see the module text."""
    parts = _parts(x, devices)
    xs = _replicas(x, parts)
    wss = _workspaces(xs, parts, ws)
    return tuple(t.to(x.device) for t in _mst_parts(xs, _replicas(core, parts), parts, wss))


def labels_from_mst(src, dst, w, min_cluster_size):
    """sklearn's host tail: _process_mst (argsort by weight, make_single_linkage), then tree_to_labels with excess-of-mass
    selection -> (labels int64[N], -1 = noise; probabilities float64[N])"""
    from sklearn.cluster._hdbscan._linkage import MST_edge_dtype, make_single_linkage
    from sklearn.cluster._hdbscan._tree import tree_to_labels
    mst = np.empty(len(w), dtype=MST_edge_dtype)
    mst["current_node"], mst["next_node"], mst["distance"] = src, dst, w
    mst = mst[np.argsort(mst["distance"])]
    tree = make_single_linkage(mst)
    return tree_to_labels(tree, min_cluster_size, "eom", False, 0.0, None)


def _check_params(min_cluster_size, min_samples):
    if isinstance(min_cluster_size, bool) or not isinstance(min_cluster_size, (int, np.integer)) or min_cluster_size < 2:
        raise ValueError("The 'min_cluster_size' parameter of %s must be an int in the range [2, inf). Got %r instead."
                         % (_SK, min_cluster_size))
    if min_samples is not None and (isinstance(min_samples, bool) or not isinstance(min_samples, (int, np.integer)) or min_samples < 1):
        raise ValueError("The 'min_samples' parameter of %s must be an int in the range [1, inf) or None. Got %r instead."
                         % (_SK, min_samples))


def hdbscan_device(latent, min_cluster_size, min_samples=None, devices=None):
    """sklearn.cluster.HDBSCAN(min_cluster_size=min_cluster_size, min_samples=min_samples).fit(latent) ->
    (labels int64[N], -1 = noise; probabilities float64[N]) for a float32 [N, D] CUDA tensor or a numpy array (rounded to
    float32).  min_samples counts the point itself and defaults to min_cluster_size, as in sklearn.  Unlike sklearn,
    non-finite values are rejected with ValueError instead of being given special labels.  devices: None (the tensor's
    device, or the current one for a numpy array) or a list of CUDA devices to split the all-pairs passes over; the
    results do not depend on it."""
    _check_params(min_cluster_size, min_samples)
    x = _as_device_matrix(latent)
    _check_finite(x)
    n = x.shape[0]
    if n == 1:
        raise ValueError("n_samples=1 while HDBSCAN requires more than one sample")
    k = min_cluster_size if min_samples is None else min_samples
    if k > n:
        raise ValueError(f"min_samples ({k}) must be at most the number of samples in X ({n})")
    parts = _parts(x, devices)
    xs = _replicas(x, parts)
    wss = _workspaces(xs, parts)   # each part's workspace serves both passes
    src, dst, w = _mst_parts(xs, _core_parts(xs, parts, k, wss), parts, wss)
    return labels_from_mst(src.cpu().numpy(), dst.cpu().numpy(), w.cpu().numpy(), int(min_cluster_size))
