"""Statistical outlier removal on the GPU (csrc/s9_knn.cu): the role of Open3D's
PointCloud.remove_statistical_outlier in the reference's clean_point_cloud (mesh_handler.py:89-94).

For every point, avg = mean distance to its k nearest points of the cloud (itself included); a point is kept iff
0 < avg < mean + std_ratio * std, with mean / std taken over the points with avg > 0 but divided by the full point count
(Bessel's correction for std).  The kNN is exact.  The one host sync is the read of the kept count (and the statistics
with it) that sizes the outputs.
"""
import ctypes

import torch

from . import capi


def _prepare(points):
    capi.require_cuda(points)
    if points.dim() != 2 or points.shape[1] != 3:
        raise capi.G2pcError(f"points must be (n, 3), got {tuple(points.shape)}")
    if points.dtype != torch.float32:
        raise capi.G2pcError(f"points must be float32, got {points.dtype}")
    return points.contiguous()


def _workspace(nbytes, device):
    return torch.empty((max(int(nbytes), 256),), dtype=torch.uint8, device=device)


def knn_mean_distance(points, k=20):
    """(n,) float64: mean distance of each point to its k nearest points (itself included; all n when n < k).  Points
    with a non-finite coordinate get NaN.  No host sync."""
    pts = _prepare(points)
    n = pts.shape[0]
    if not 1 <= int(k) <= 32:
        raise capi.G2pcError(f"k must be in [1, 32], got {k}")
    avg = torch.empty((n,), dtype=torch.float64, device=pts.device)
    ws = _workspace(capi.load().g2pc_knn_workspace_bytes(n, int(k)), pts.device)
    capi.call("g2pc_knn_mean_distance", capi.ptr(pts), n, int(k), capi.ptr(avg), capi.ptr(ws), ws.numel(),
              capi.stream_ptr(pts.device))
    return avg


def select_inliers(points, nb_neighbors=20, std_ratio=10.0):
    """(index int32 ascending, stats dict) of the points remove_statistical_outlier keeps.  Raises G2pcError on a
    non-finite coordinate.  One host sync."""
    if not std_ratio > 0:
        raise capi.G2pcError(f"std_ratio must be > 0, got {std_ratio}")
    if nb_neighbors < 1:
        raise capi.G2pcError(f"nb_neighbors must be >= 1, got {nb_neighbors}")
    pts = _prepare(points)
    n, dev = pts.shape[0], pts.device
    st = capi.stream_ptr(dev)
    avg = knn_mean_distance(pts, nb_neighbors)
    keep = torch.empty((max(n, 1),), dtype=torch.uint8, device=dev)
    # one device buffer for everything the host reads: [kept count as int64 | mean, std, threshold, non-finite count]
    out = torch.zeros((5,), dtype=torch.float64, device=dev)
    stats4 = out[1:]
    ws = _workspace(capi.load().g2pc_outlier_workspace_bytes(n), dev)
    capi.call("g2pc_outlier_mask", capi.ptr(avg), n, float(std_ratio), capi.ptr(keep), capi.ptr(stats4), capi.ptr(ws),
              ws.numel(), st)
    index = torch.empty((max(n, 1),), dtype=torch.int32, device=dev)
    cws = _workspace(capi.load().g2pc_cull_workspace_bytes(n), dev)
    capi.call("g2pc_cull_select", None, 0.0, None, 0.0, None, None, None, None, None, capi.ptr(keep), 0, n, n,
              capi.ptr(index), out.data_ptr(), capi.ptr(cws), cws.numel(), st)
    host = out.cpu()  # the one host read
    m = int(host[:1].view(torch.int64)[0])
    mean, std, thr, nonfinite = (float(v) for v in host[1:])
    if nonfinite > 0:
        raise capi.G2pcError(f"{int(nonfinite)} points have a non-finite coordinate")
    return index[:m], {"mean": mean, "std": std, "threshold": thr, "n": n, "kept": m}


def remove_statistical_outliers(points, nb_neighbors=20, std_ratio=10.0):
    """(index int64 ascending, stats) — the indices Open3D's remove_statistical_outlier returns alongside its cloud.
    stats: {"mean", "std", "threshold", "n", "kept"}."""
    index, stats = select_inliers(points, nb_neighbors, std_ratio)
    return index.to(torch.int64), stats


def gather_rows(index, tensors):
    """Rows `index` (int32, device) of each tensor (None passes through), compacted by g2pc_gather_rows."""
    m = index.shape[0]
    srcs = [None if t is None else t.contiguous() for t in tensors]
    dsts = [None if s is None else torch.empty((m,) + tuple(s.shape[1:]), dtype=s.dtype, device=s.device) for s in srcs]
    live = [(s, d) for s, d in zip(srcs, dsts) if s is not None]
    if m > 0 and live:
        k = len(live)
        sp = (ctypes.c_void_p * k)(*[s.data_ptr() for s, _ in live])
        dp = (ctypes.c_void_p * k)(*[d.data_ptr() for _, d in live])
        rb = (ctypes.c_int32 * k)(*[int(s[0].numel() * s.element_size()) for s, _ in live])
        capi.call("g2pc_gather_rows", capi.ptr(index), m, k, sp, dp, rb, capi.stream_ptr(index.device))
    return dsts
