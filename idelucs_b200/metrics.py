"""Silhouette coefficients of a clustering (sklearn.metrics.silhouette_samples / silhouette_score, Euclidean metric) with
the all-pairs work on the GPU.

idl_silhouette_samples computes every distance in fp64 exactly as the HDBSCAN kernels do (the sklearn EuclideanDistance
arithmetic) and sums them per cluster in index order, as sklearn's np.bincount does.  sklearn itself forms its distances
with a matrix product, so the two agree to about 1e-14, not bit for bit; identical rows, which that product puts about 3e-7
apart instead of 0, are the exception."""
import numpy as np

from . import _lib
from .hdbscan import _as_device_matrix, _check_finite, _parts, _replicas


def silhouette_samples_device(X, labels, devices=None):
    """sklearn.metrics.silhouette_samples(X, labels) -> float64 [N] numpy array, for a float32 [N, D] CUDA tensor or a
    numpy array (rounded to float32).  labels: any integer array of length N, encoded densely as sklearn's LabelEncoder
    does; 2 to N - 1 distinct labels.  Non-finite values of X are rejected with ValueError.  devices: None (the tensor's
    device, or the current one for a numpy array) or a list of CUDA devices (repeats allowed) over which the rows are split
    as in hdbscan.row_parts; the values do not depend on it."""
    import torch
    x = _as_device_matrix(X)
    _check_finite(x)
    n, D = x.shape
    labels = np.ravel(labels.cpu().numpy() if torch.is_tensor(labels) else labels)
    if len(labels) != n:
        raise ValueError("Found input variables with inconsistent numbers of samples: [%d, %d]" % (n, len(labels)))
    uniq, enc = np.unique(labels, return_inverse=True)
    n_labels = len(uniq)
    if not 1 < n_labels < n:
        raise ValueError("Number of labels is %d. Valid values are 2 to n_samples - 1 (inclusive)" % n_labels)
    lib = _lib.load()
    parts = _parts(x, devices)
    xs = _replicas(x, parts)
    labs = _replicas(torch.from_numpy(enc.astype(np.int32)), parts)
    outs = {d: torch.empty(n, dtype=torch.float64, device=d) for d in xs}
    for d, b, e in parts:   # every call synchronises its stream once (the label check), then leaves its kernel running
        ws = torch.empty(lib.idl_silhouette_workspace_bytes(n, n_labels), dtype=torch.uint8, device=d)
        with torch.cuda.device(d):
            _lib.check(lib.idl_silhouette_samples_rows(_lib.ptr(xs[d]), _lib.ptr(labs[d]), n, D, n_labels, b, e, _lib.ptr(outs[d]),
                                                       _lib.ptr(ws), ws.numel(), _lib.stream_ptr()))
    out = np.empty(n, dtype=np.float64)
    for d, b, e in parts:
        out[b:e] = outs[d][b:e].cpu().numpy()
    return out


def silhouette_score_device(X, labels, devices=None):
    """sklearn.metrics.silhouette_score(X, labels) (all samples, Euclidean metric): the mean of silhouette_samples_device,
    taken on the host as sklearn takes it."""
    return float(np.mean(silhouette_samples_device(X, labels, devices)))
