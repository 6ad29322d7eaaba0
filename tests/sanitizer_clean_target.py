"""Tiny run of point-cloud cleaning (kNN mean distances, outlier mask, compaction), meant to be executed under
compute-sanitizer (tests/test_cleaning_sanitizer_gpu.py): memcheck over the kNN build / query kernels and the
reductions, racecheck over the shared-memory reductions and the bottom-up tree build."""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "3dgs-to-pc_b200"))
import torch  # noqa: E402

import mesh_handler  # noqa: E402
from g2pc import outliers  # noqa: E402

dev = "cuda:0"
g = torch.Generator().manual_seed(5)
# a cluster, a few far points and an odd size (partial last bucket, empty leaves in the tree)
pts = torch.cat([torch.randn(3000, 3, generator=g), 40 * torch.randn(37, 3, generator=g)]).to(dev)
cols = torch.rand(pts.shape[0], 3, generator=g).to(dev) * 255
nrm = torch.randn(pts.shape[0], 3, generator=g).to(dev)
for k in (1, 20, 32):
    outliers.knn_mean_distance(pts, k)
outliers.remove_statistical_outliers(pts[:5], 20, 10.0)
p, c, n = mesh_handler.clean_point_cloud(pts, cols, nrm)
torch.cuda.synchronize()
print("SANITIZER_TARGET_OK", p.shape[0], pts.shape[0])
