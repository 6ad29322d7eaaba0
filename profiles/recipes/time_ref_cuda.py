#!/usr/bin/env python
"""Time the UNMODIFIED reference pipeline with renderer_type=cuda (the reference CUDA rasterizer built for sm_100 by
oracle/build_ref.py) on a bench.py workload, with a colour-stage / sampling-stage split.

    python profiles/recipes/time_ref_cuda.py --workload c3 --steps 1 [--json out.json]
"""
import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "3dgs-to-pc_b200"))
import torch  # noqa: E402

import bench  # noqa: E402
from baseline import ref_run  # noqa: E402
from g2pc import synth  # noqa: E402
from oracle import ref_shim  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--workload", default="c3")
ap.add_argument("--steps", type=int, default=1)
ap.add_argument("--json", default=None)
a = ap.parse_args()
wl = bench.WORKLOADS[a.workload]
sc = bench._scene_for(wl)
cams, intr = synth.make_cameras(wl["cams"]) if wl["cams"] else ([], [])
ref = ref_shim.load()
g2p = ref.gauss_to_pc
stage = {}
orig_gen = g2p.generate_pointcloud


def timed_gen(*args, **kw):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = orig_gen(*args, **kw)
    torch.cuda.synchronize()
    stage["generate_pointcloud_s"] = time.perf_counter() - t0
    return out


g2p.generate_pointcloud = timed_gen
rows = []
for i in range(a.steps + 1):  # first pass = warm-up (CUDA context, lazy imports)
    pc, dt = ref_run.run(sc, cams, intr, device="cuda:0", renderer_type="cuda", num_points=wl["points"],
                         render_colours=wl["colours"], colour_resolution=wl["res"], max_sh_degree=wl["sh"])
    row = dict(step=i, seconds=round(dt, 3), points=int(pc.points.shape[0]),
               mpoints_per_s=round(pc.points.shape[0] / dt / 1e6, 4), **{k: round(v, 3) for k, v in stage.items()})
    print(json.dumps(row), flush=True)
    rows.append(row)
if a.json:
    json.dump(dict(workload=a.workload, rows=rows), open(a.json, "w"), indent=1)
