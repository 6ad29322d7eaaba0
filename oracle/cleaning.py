"""Oracle restatement of point-cloud cleaning (TEST INFRASTRUCTURE, see oracle/__init__.py).

The reference's clean_point_cloud (mesh_handler.py:42-64, 89-94; called from gauss_to_pc.py:743-759) hands the cloud to
Open3D's PointCloud.remove_statistical_outlier(nb_neighbors=20, std_ratio=10) — the CLI never passes std_ratio.  Open3D
is not available where this project runs, so this module is pinned to the written statement of Open3D's
RemoveStatisticalOutliers below, NOT to a live Open3D run:

  1. points are widened to float64 (exact for a float32 cloud);
  2. avg[i] = mean of the Euclidean distances from point i to its k = nb_neighbors nearest points of the cloud, the point
     itself included (distance 0); k_eff = N when N < k.  Ties at the k-th distance do not change avg;
  3. valid = N (every point has at least one neighbour: itself);
  4. mean = sum of avg[i] over avg[i] > 0, divided by valid (exact duplicates, avg == 0, still count in the divisor);
  5. std = sqrt(sum over avg[i] > 0 of (avg[i] - mean)^2 / (valid - 1))  (two passes, Bessel's correction);
  6. threshold = mean + std_ratio * std;
  7. keep i iff avg[i] > 0 and avg[i] < threshold (strict; avg == 0 is dropped);
  8. kept rows stay in ascending original order;
  9. N = 0 -> empty; N = 1 -> empty (threshold is NaN); all points identical -> empty; nb_neighbors < 1 or
     std_ratio <= 0 -> error;
 10. colours come out as int32(trunc(clamp(c, 0, 255))) (the /255 ... *255 round trip through Open3D is exact for every
     integer 0..255 in float64); the reference returns points and normals as float64.

The kNN is an exact brute-force search in float64, chunked, that skips only blocks of points proven too far away;
`queries` restricts the rows whose avg is computed (each still searched against the whole cloud).
"""
import numpy as np
import torch


def _spread10(v):
    v = v.astype(np.uint64) & np.uint64(0x3FF)
    out = np.zeros_like(v)
    for b in range(10):
        out |= ((v >> np.uint64(b)) & np.uint64(1)) << np.uint64(3 * b)
    return out


def _spatial_order(P):
    """A Morton order of the rows (10 bits per axis): consecutive rows are close in space.  Only the speed of the search
    depends on it."""
    lo = P.min(0)
    ext = float((P.max(0) - lo).max()) or 1.0
    q = np.clip(((P - lo) / ext * 1023.0), 0, 1023).astype(np.uint64)
    key = (_spread10(q[:, 0]) << np.uint64(2)) | (_spread10(q[:, 1]) << np.uint64(1)) | _spread10(q[:, 2])
    return np.argsort(key, kind="stable")


def _topk_d2(Q, C, ke, point_chunk=1 << 20):
    """(q, ke) smallest float64 squared distances from the rows of Q to the rows of C (brute force, chunked)."""
    best = None
    for p0 in range(0, C.shape[0], point_chunk):
        Cc = C[p0:p0 + point_chunk]
        d2 = ((Q[:, None, 0] - Cc[None, :, 0]) ** 2 + (Q[:, None, 1] - Cc[None, :, 1]) ** 2
              + (Q[:, None, 2] - Cc[None, :, 2]) ** 2)
        d2 = torch.topk(d2, min(ke, d2.shape[1]), dim=1, largest=False).values
        best = d2 if best is None else torch.topk(torch.cat([best, d2], 1), ke, dim=1, largest=False).values
    return best


def knn_mean_distance(points, k=20, queries=None, block=512, query_chunk=32):
    """avg (len(queries) or N,) float64: the k smallest float64 distances of each query row to every point of the cloud
    (itself included), averaged over k_eff = min(k, N).

    Brute force over blocks of `block` spatially consecutive points: a block is searched exhaustively unless its exact
    bounding-box distance exceeds an upper bound of the query's k-th distance (the k-th distance among the 2 * block
    points around the query), so the result equals the all-pairs search (tests/test_cleaning_cpu.py checks that)."""
    if k < 1:
        raise ValueError("nb_neighbors must be >= 1")
    P = np.asarray(points, dtype=np.float64).reshape(-1, 3)
    n = P.shape[0]
    rows = np.arange(n) if queries is None else np.asarray(queries, dtype=np.int64).reshape(-1)
    out = np.empty((rows.shape[0],), dtype=np.float64)
    if n == 0 or rows.shape[0] == 0:
        return out
    ke = min(k, n)
    order = _spatial_order(P)
    rank = np.empty(n, dtype=np.int64)
    rank[order] = np.arange(n)
    S = torch.from_numpy(P[order])
    nblk = (n + block - 1) // block
    pad = torch.cat([S, S[-1:].expand(nblk * block - n, 3)]).view(nblk, block, 3)  # repeats a real point: boxes exact
    blo, bhi = pad.min(1).values, pad.max(1).values
    qorder = np.argsort(rank[rows], kind="stable")  # group the queries spatially
    for q0 in range(0, rows.shape[0], query_chunk):
        sel = qorder[q0:q0 + query_chunk]
        Q = torch.from_numpy(P[rows[sel]])
        # upper bound of each query's k-th squared distance: the k-th among the points around its own sorted position
        up2 = torch.empty(Q.shape[0], dtype=torch.float64)
        for j, r in enumerate(rank[rows[sel]]):
            a = max(0, min(int(r) - block, n - 2 * block))
            up2[j] = _topk_d2(Q[j:j + 1], S[a:a + 2 * block], ke)[0, -1]
        gap = torch.clamp(blo[None] - Q[:, None], min=0) + torch.clamp(Q[:, None] - bhi[None], min=0)
        lb2 = (gap ** 2).sum(-1)
        need = (lb2 * (1 - 1e-9) <= up2[:, None] * (1 + 1e-9)).any(0)
        C = pad[need].reshape(-1, 3)
        last = int(torch.nonzero(need)[-1]) if bool(need[-1]) else -1
        if last == nblk - 1:  # drop the padding copies of the last block
            C = C[: C.shape[0] - (nblk * block - n)]
        best = _topk_d2(Q, C, ke)
        out[sel] = (torch.sqrt(torch.sort(best, dim=1).values).sum(1) / ke).numpy()
    return out


def knn_mean_distance_all_pairs(points, k=20):
    """The same as knn_mean_distance by a plain all-pairs search (small clouds: the check of the blocked search)."""
    P = torch.as_tensor(np.asarray(points, dtype=np.float64)).reshape(-1, 3)
    n = P.shape[0]
    if n == 0:
        return np.empty(0)
    ke = min(k, n)
    out = [torch.sqrt(torch.sort(_topk_d2(P[i:i + 256], P, ke), dim=1).values).sum(1) / ke for i in range(0, n, 256)]
    return torch.cat(out).numpy()


def outlier_stats(avg, std_ratio):
    """(mean, std, threshold, keep mask) from the per-point mean distances (steps 3-7)."""
    if not std_ratio > 0:
        raise ValueError("std_ratio must be > 0")
    avg = np.asarray(avg, dtype=np.float64)
    valid = avg.shape[0]
    if valid == 0:
        return 0.0, 0.0, 0.0, np.zeros(0, dtype=bool)
    pos = avg > 0
    mean = avg[pos].sum() / valid
    with np.errstate(invalid="ignore", divide="ignore"):
        std = float(np.sqrt(((avg[pos] - mean) ** 2).sum() / (valid - 1)))
    thr = mean + std_ratio * std
    keep = pos & (avg < thr)
    return float(mean), std, float(thr), keep


def remove_statistical_outliers(points, nb_neighbors=20, std_ratio=10.0):
    """(index int64 ascending, {"mean", "std", "threshold", "avg"}) of the kept points."""
    if nb_neighbors < 1:
        raise ValueError("nb_neighbors must be >= 1")
    if not std_ratio > 0:
        raise ValueError("std_ratio must be > 0")
    avg = knn_mean_distance(points, nb_neighbors)
    mean, std, thr, keep = outlier_stats(avg, std_ratio)
    return np.nonzero(keep)[0].astype(np.int64), {"mean": mean, "std": std, "threshold": thr, "avg": avg}


def convert_colours(colours):
    """int32(trunc(clamp(c, 0, 255))) — the reference's colours after the Open3D round trip (mesh_handler.py:47,51,60)."""
    c = torch.clamp(torch.as_tensor(np.asarray(colours)), min=0, max=255).to(torch.int32)
    return c.numpy()


def clean_point_cloud(points, colours, normals, std_ratio=10):
    """mesh_handler.py:89-94 restated: (points float64, colours int32, normals float64 or None) of the kept rows."""
    idx, _ = remove_statistical_outliers(points, 20, std_ratio)
    pts = np.asarray(points, dtype=np.float64)[idx]
    cols = convert_colours(colours)[idx]
    nrm = None if normals is None else np.asarray(normals, dtype=np.float64)[idx]
    return pts, cols, nrm
