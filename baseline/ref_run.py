"""Run the UNMODIFIED reference pipeline (convert_3dgs_to_pc, gauss_to_pc.py:373-601) on an in-memory synthetic scene.

The reference's own code does all the work; only its two FILE LOADERS are replaced in its module namespace (the
container has no `plyfile`, and BASELINE.md §3.1 excludes file parsing from the timed region):
    load_gaussians(path, max_sh_degree)   -> the synthetic tensors, on the device the reference would put them on
    load_transform_data(path, skip_rate)  -> ({name: 4x4 nested list}, {name: [w, h, fx, fy]})

  run(scene, cams, intr, settings_kwargs, device)   device "cuda:0": stock GPU path (renderer_type "cuda" uses the
                                                     reference's CUDA rasterizer built by oracle/build_ref.py)
                                                     device "cpu": through oracle.ref_shim.cpu_redirect (the
                                                     reference hard-codes "cuda" devices)
Used by bench.py's reference legs and by GPU tests that compare against the reference itself.  Never imported by the
product.
"""
import contextlib
import os
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from oracle import ref_shim  # noqa: E402


def available():
    return ref_shim.available()


def cuda_extension_available():
    import glob
    return bool(glob.glob(os.path.join(ref_shim.STAGED_EXT_ROOT, "gaussian_pointcloud_rasterization", "_C*.so")))


def settings(ref, **kw):
    d = dict(renderer_type="cuda", num_points=10_000_000, prioritise_visible_gaussians=True,
             mahalanobis_distance_std=2.0, camera_skip_rate=0, render_colours=True, min_opacity=0.0,
             bounding_box_min=None, bounding_box_max=None, calculate_normals=True, cull_large_percentage=0.0,
             remove_unrendered_gaussians=True, colour_resolution=1280, max_sh_degree=3, exact_num_points=False,
             visibility_threshold=0.05, surface_distance_std=None, generate_mesh=False, quiet=True, device="cuda:0")
    d.update(kw)
    return ref.gauss_to_pc.GaussPointCloudSettings(**d)


def run(scene, cams, intr, device="cuda:0", pinned_tiles=(60, 60000), **settings_kw):
    """scene: dict of CPU tensors from g2pc.synth.make_scene; cams / intr: lists from g2pc.synth.make_cameras.
    Returns (PointCloudData, seconds of convert_3dgs_to_pc incl. a final device synchronise, stage seconds dict)."""
    ref = ref_shim.load()
    g2p = ref.gauss_to_pc
    on_gpu = str(device).startswith("cuda")
    dev = device if on_gpu else "cpu"
    tens = {k: v.to(dev) for k, v in scene.items()}
    transforms = {f"cam{i:04d}": c.tolist() for i, c in enumerate(cams)}
    intrinsics = {f"cam{i:04d}": list(k) for i, k in enumerate(intr)}

    def load_gaussians(path, max_sh_degree=3):
        return (tens["xyz"].clone(), tens["scales"].clone(), tens["rots"].clone(), tens["colours"].clone(),
                tens["opacities"].clone(), tens["shs"].clone())

    def load_transform_data(path, skip_rate=0):
        return dict(transforms), dict(intrinsics)

    saved = (g2p.load_gaussians, g2p.load_transform_data)
    g2p.load_gaussians, g2p.load_transform_data = load_gaussians, load_transform_data
    st = settings(ref, device=dev, **settings_kw)
    ctx = contextlib.ExitStack()
    if not on_gpu:
        ctx.enter_context(ref_shim.cpu_redirect(pinned_tiles))
    if st.renderer_type == "cuda":
        ctx.enter_context(ref_shim.reference_extension())  # the reference's own package, not the product's namesake
    try:
        with ctx:
            if on_gpu:
                torch.cuda.synchronize()
            t0 = time.perf_counter()
            pc, _ = g2p.convert_3dgs_to_pc("synthetic.ply", "synthetic" if (cams and st.render_colours) else None,
                                           None, st)
            if on_gpu:
                torch.cuda.synchronize()
            dt = time.perf_counter() - t0
    finally:
        g2p.load_gaussians, g2p.load_transform_data = saved
    return pc, dt
