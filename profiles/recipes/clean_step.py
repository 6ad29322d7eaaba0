#!/usr/bin/env python
"""Time --clean_pointcloud (mesh_handler.clean_point_cloud: kNN mean distances, outlier mask, compaction) on the point
clouds of bench.py's C3 (10M points from 3M Gaussians) and C5 (100M points from 6M Gaussians) scenes, each with 0.1 %
extra points scattered over 100x the scene's extent.  Warm-up, then CUDA-event timing of whole calls, then one more
pass with capi.TIMING for the split per entry point.  The GPU's name and power limit are read in the same run.

    python profiles/recipes/clean_step.py --workload c3 --reps 5 --out profiles/r03_clean_c3.json
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "3dgs-to-pc_b200"))
import torch  # noqa: E402

import bench  # noqa: E402
import gauss_handler as gh  # noqa: E402
import gauss_to_pc as g2p  # noqa: E402
import mesh_handler  # noqa: E402
from g2pc import build, capi  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--workload", default="c3", choices=["c3", "c5"])
ap.add_argument("--reps", type=int, default=5)
ap.add_argument("--warmup", type=int, default=2)
ap.add_argument("--out", required=True)
a = ap.parse_args()

build.build()
capi.load()
dev = "cuda:0"
gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                     capture_output=True, text=True).stdout.strip()
wl = bench.WORKLOADS[a.workload]
torch.set_num_threads(min(16, os.cpu_count() or 1))
sc = bench._scene_for(wl)
d = {k: v.to(dev) for k, v in sc.items()}
G = gh.Gaussians(d["xyz"], d["scales"], d["rots"], d["colours"] * 255, d["opacities"])
G.calculate_normals()
G.validate_covariances()
pts, cols, nrm = g2p.generate_pointcloud(G, wl["points"], quiet=True)
del G, d
g = torch.Generator().manual_seed(11)
ext = float((pts.max(0).values - pts.min(0).values).max())
no = pts.shape[0] // 1000
pts = torch.cat([pts, ((torch.rand(no, 3, generator=g) * 2 - 1) * 50 * ext).to(dev)]).contiguous()
cols = torch.cat([cols, torch.full((no, 3), 128.0, dtype=cols.dtype, device=dev)])
nrm = torch.cat([nrm, torch.zeros((no, 3), dtype=nrm.dtype, device=dev)])
n = pts.shape[0]
torch.cuda.synchronize()

for _ in range(a.warmup):
    out = mesh_handler.clean_point_cloud(pts, cols, nrm)
torch.cuda.synchronize()
times = []
for _ in range(a.reps):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    out = mesh_handler.clean_point_cloud(pts, cols, nrm)
    e1.record()
    torch.cuda.synchronize()
    times.append(e0.elapsed_time(e1))
capi.TIMING = {}
mesh_handler.clean_point_cloud(pts, cols, nrm)
torch.cuda.synchronize()
split = {k: sum(x.elapsed_time(y) for x, y in v) for k, v in capi.TIMING.items()}
capi.TIMING = None
res = {
    "workload": a.workload, "gpu": gpu, "points": n, "injected_outliers": no, "kept": int(out[0].shape[0]),
    "clean_ms": sorted(times), "clean_ms_median": sorted(times)[len(times) // 2],
    "split_ms": split,
    "knn_workspace_bytes_per_point": capi.load().g2pc_knn_workspace_bytes(n, 20) / n,
    "note": "whole clean_point_cloud calls (kNN + mask + compaction of points, colours, normals, one host sync), "
            "CUDA events; split_ms: one extra call with every entry point bracketed by events",
}
print(json.dumps(res, indent=1))
os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
with open(a.out, "w") as f:
    json.dump(res, f, indent=1)
