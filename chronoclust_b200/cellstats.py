"""Per-group cell statistics computed on the device: cell counts, means, exact medians and linear quantiles per marker
(ccb_group_stats / ccb_cluster_stats in include/chronoclust_b200.h).

`group_statistics` is the stateless form over any rows; HDDStream.cluster_statistics groups the cells of its last
timepoint by cluster; app.run(cluster_statistics=True) writes the per-timepoint medians and means to cluster_statistics.csv.
"""
import collections
import ctypes as C

import numpy as np

from . import _lib

# count [G] int64; mean / median [G][D] float64; quantiles [nq][G][D] float64
GroupStats = collections.namedtuple("GroupStats", "count mean median quantiles")


def quantile_array(quantiles):
    """The requested quantiles as a contiguous float64 vector; ValueError unless every one lies in [0, 1] (NaN does not)."""
    q = np.ascontiguousarray(np.asarray(quantiles, dtype=np.float64).reshape(-1))
    if not np.all((q >= 0.0) & (q <= 1.0)):
        raise ValueError(f"quantiles must lie in [0, 1], got {q.tolist()}")
    return q


def _outputs(G, D, nq):
    return GroupStats(np.empty(G, np.int64), np.empty((G, D), np.float64), np.empty((G, D), np.float64),
                      np.empty((nq, G, D), np.float64))


def _pointers(out, q):
    return (_lib.ptr(q) if len(q) else None, _lib.ptr(out.count), _lib.ptr(out.mean), _lib.ptr(out.median),
            _lib.ptr(out.quantiles) if len(q) else None)


def group_statistics(X, groups, n_groups, quantiles=()):
    """Count, mean, median and the requested quantiles of every marker of every group, computed on the GPU.

    X: [N, D] rows (D <= 64) -- a CUDA tensor (float32 or float64 rows with unit column stride go in as they are,
    row-strided views included), or a numpy array / CPU tensor, which is copied to the current CUDA device first.
    groups: [N] integers, -1 = leave the row out, else the row's group in [0, n_groups).  The call runs after the work
    queued on the current torch stream of X's device and waits for its own.

    Returns GroupStats(count [G], mean [G, D], median [G, D], quantiles [nq, G, D]): the median is np.median and each
    quantile np.quantile(..., method="linear") of the group's values bit for bit, the mean np.mean up to rounding (the
    same bits on every call).  A group without rows has count 0 and NaN elsewhere; a NaN in a marker makes that marker's
    mean, median and quantiles NaN."""
    import torch

    q = quantile_array(quantiles)
    G = int(n_groups)
    if G < 1:
        raise ValueError(f"n_groups must be >= 1, got {n_groups}")
    if not isinstance(X, torch.Tensor):
        X = torch.from_numpy(np.asarray(X))
    if X.dim() != 2:
        raise ValueError(f"X must be 2-D, got shape {tuple(X.shape)}")
    N, D = X.shape
    if not 1 <= D <= 64:
        raise ValueError(f"X has {D} markers; 1 to 64 are supported")
    if isinstance(groups, torch.Tensor):
        if groups.is_floating_point() or groups.is_complex() or groups.dtype == torch.bool:
            raise ValueError("groups must hold integers")
        g_host = None
    else:
        g_host = np.asarray(groups)
        if g_host.dtype.kind not in "iu":
            raise ValueError("groups must hold integers")
        groups = g_host
    if tuple(groups.shape) != (N,):
        raise ValueError(f"groups must have shape ({N},), got {tuple(groups.shape)}")
    if N and g_host is not None and (int(g_host.min()) < -1 or int(g_host.max()) >= G):
        raise ValueError(f"groups must lie in [-1, {G})")
    dev = X.device if X.is_cuda else torch.device("cuda", torch.cuda.current_device())
    if N and g_host is None:
        lo, hi = int(groups.min()), int(groups.max())
        if lo < -1 or hi >= G:
            raise ValueError(f"groups must lie in [-1, {G})")

    if X.dtype not in (torch.float32, torch.float64):
        X = X.to(torch.float64)
    X = X.to(dev)
    if N and (X.stride(1) != 1 or (N > 1 and X.stride(0) < D)):
        X = X.contiguous()
    ld = X.stride(0) if N > 1 else D
    gd = torch.as_tensor(groups).to(device=dev, dtype=torch.int32).contiguous()
    code = _lib.DTYPE_F32 if X.dtype == torch.float32 else _lib.DTYPE_F64
    out = _outputs(G, D, len(q))
    stream = torch.cuda.current_stream(dev)
    with torch.cuda.device(dev):
        _lib.check(_lib.lib().ccb_group_stats(dev.index, C.c_void_p(stream.cuda_stream), X.data_ptr() if N else None,
                                              code, N, ld, D, gd.data_ptr() if N else None, G, len(q), *_pointers(out, q)))
    return out


def cluster_statistics(h, D, group_of_pcore, G, quantiles=()):
    """ccb_cluster_stats on handle h: G + 1 rows, the last one the cells in no group (see HDDStream.cluster_statistics).
    D: the width of the rows of the handle's last ingest (W after a column-subset ingest)."""
    q = quantile_array(quantiles)
    gop = np.ascontiguousarray(group_of_pcore, dtype=np.int32)
    out = _outputs(G + 1, D, len(q))
    _lib.check(_lib.lib().ccb_cluster_stats(h, _lib.ptr(gop) if len(gop) else None, len(gop), G, len(q),
                                            *_pointers(out, q)), h)
    return out


def statistics_rows(timepoint, labels, stats):
    """The cluster_statistics.csv rows of one timepoint: [timepoint, label, cell_count, medians..., means...] for every
    lineage label but 'None' (labels[1:], group g = labels[g + 1]; a label past the groups of `stats` has no cells), then
    the 'None' row from the last row of `stats`.  Floats go out as Python floats: csv.writer writes their repr, which
    reads back to the same bits."""
    G, D = len(stats.count) - 1, stats.mean.shape[1]
    rows = []
    for g, label in enumerate(labels[1:]):
        if g < G:
            rows.append([timepoint, label, int(stats.count[g])] + stats.median[g].tolist() + stats.mean[g].tolist())
        else:
            rows.append([timepoint, label, 0] + [float("nan")] * (2 * D))
    rows.append([timepoint, "None", int(stats.count[G])] + stats.median[G].tolist() + stats.mean[G].tolist())
    return rows
