"""HDBSCAN of the latent space (idelucs/__main__.py:149-156, the --n_clusters 0 mode) with its all-pairs work on the GPU.

Results equal ``sklearn.cluster.HDBSCAN(min_cluster_size, min_samples).fit(X)`` (Euclidean metric, alpha 1, excess-of-mass
selection): idl_core_distances and idl_mreach_mst compute the core distances and the mutual-reachability minimum spanning
tree with sklearn's own fp64 arithmetic, and sklearn's host code (make_single_linkage, tree_to_labels) turns the tree into
labels and probabilities, exactly as sklearn's ``_process_mst`` and ``fit`` do.  Ties between MST weights are the only
source of a difference: sklearn orders tied edges by an unstable argsort of its Prim order, this module by an unstable
argsort of the Borůvka order."""
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


def core_distances(x, k, ws=None):
    """float64 [N] CUDA tensor: the distance of every row of the float32 CUDA matrix x to its k-th nearest row, itself
    included (NearestNeighbors.kneighbors(X, k)[0][:, -1])."""
    import torch
    n, D = x.shape
    ws = _workspace(x) if ws is None else ws
    core = torch.empty(n, dtype=torch.float64, device=x.device)
    with torch.cuda.device(x.device):
        _lib.check(_lib.load().idl_core_distances(_lib.ptr(x), n, D, int(k), _lib.ptr(core), _lib.ptr(ws), ws.numel(), _lib.stream_ptr()))
    return core


def mreach_mst(x, core, ws=None):
    """the N-1 edges (src int64, dst int64, weight float64; CUDA tensors, Borůvka order) of the minimum spanning tree of
    the mutual-reachability graph max(core[i], core[j], d(i, j)) of the float32 CUDA matrix x"""
    import torch
    n, D = x.shape
    ws = _workspace(x) if ws is None else ws
    src = torch.empty(n - 1, dtype=torch.int64, device=x.device)
    dst = torch.empty(n - 1, dtype=torch.int64, device=x.device)
    w = torch.empty(n - 1, dtype=torch.float64, device=x.device)
    with torch.cuda.device(x.device):
        _lib.check(_lib.load().idl_mreach_mst(_lib.ptr(x), _lib.ptr(core), n, D, _lib.ptr(src), _lib.ptr(dst), _lib.ptr(w), _lib.ptr(ws),
                                              ws.numel(), _lib.stream_ptr()))
    return src, dst, w


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


def hdbscan_device(latent, min_cluster_size, min_samples=None):
    """sklearn.cluster.HDBSCAN(min_cluster_size=min_cluster_size, min_samples=min_samples).fit(latent) ->
    (labels int64[N], -1 = noise; probabilities float64[N]) for a float32 [N, D] CUDA tensor or a numpy array (rounded to
    float32).  min_samples counts the point itself and defaults to min_cluster_size, as in sklearn.  Unlike sklearn,
    non-finite values are rejected with ValueError instead of being given special labels."""
    _check_params(min_cluster_size, min_samples)
    x = _as_device_matrix(latent)
    _check_finite(x)
    n = x.shape[0]
    if n == 1:
        raise ValueError("n_samples=1 while HDBSCAN requires more than one sample")
    k = min_cluster_size if min_samples is None else min_samples
    if k > n:
        raise ValueError(f"min_samples ({k}) must be at most the number of samples in X ({n})")
    ws = _workspace(x)
    core = core_distances(x, k, ws)
    src, dst, w = mreach_mst(x, core, ws)
    return labels_from_mst(src.cpu().numpy(), dst.cpu().numpy(), w.cpu().numpy(), int(min_cluster_size))
