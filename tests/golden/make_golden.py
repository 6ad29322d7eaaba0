"""Generate the golden vectors that pin the oracle and the kernels: outputs of the UNMODIFIED reference on small
seeded scenes.  The CPU cases run the reference's Python code through oracle/ref_shim.py:

    G2PC_REFERENCE_ROOT=<reference checkout> python tests/golden/make_golden.py [case ...]

The `ref_ext` case runs the reference's compiled CUDA rasterizer (oracle/build_ref.py) on a GPU and needs no other
part of the reference:

    python tests/golden/make_golden.py ref_ext [output directory]

Inputs are regenerated from the seeds by g2pc.synth (and the test helpers), so only outputs are stored.
"""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "3dgs-to-pc_b200"))

from oracle import philox, ref_shim  # noqa: E402
from g2pc import synth  # noqa: E402

SAMPLING_CASES = {
    # name: (n_gaussians, scene_seed, num_points, exact_num_points, attempts, rng_seed)
    "sampling_a": (1500, 1301, 12000, False, 5, 42),
    "sampling_b": (800, 1302, 9000, True, 100, 43),
}


def make_sampling(name, n, scene_seed, num_points, exact, attempts, rng_seed):
    ref = ref_shim.load()
    sc = synth.make_scene(n, seed=scene_seed)
    eps_fn = lambda g, k, a: philox.draw_eps(g, k, a, rng_seed, 0)
    with ref_shim.cpu_redirect():
        G = ref.gauss_handler.Gaussians(sc["xyz"].clone(), sc["scales"].clone(), sc["rots"].clone(),
                                        sc["colours"].clone() * 255, sc["opacities"].clone())
        G.calculate_normals()
        cov0 = G.covariances.clone()
        keep = G.validate_covariances()
        mags = G.get_gaussian_magnitudes()
        ppg = ref.gauss_to_pc.distribute_points(mags, num_points).type(torch.int)
        with ref_shim.EpsInjector(ref, G.xyz, eps_fn) as inj:
            pts, cols, nrm = ref.gauss_to_pc.generate_pointcloud(
                G, num_points, mahalanobis_distance_std=2.0, exact_num_points=exact,
                num_sample_attempts=attempts, device="cpu", quiet=True)
            calls = np.array([(k, a, len(g)) for (k, a, g) in inj.log], dtype=np.int64)
    np.savez_compressed(
        os.path.join(HERE, name + ".npz"),
        meta=np.array([n, scene_seed, num_points, int(exact), attempts, rng_seed], dtype=np.int64),
        cov0=cov0.numpy(), cov=G.covariances.numpy(), keep=keep.numpy(), normals=G.normals.numpy(),
        magnitudes=mags.numpy(), ppg=ppg.numpy(), points=pts.numpy(), colours=cols.numpy().astype(np.float32),
        point_normals=nrm.numpy().astype(np.float32), mvn_calls=calls)
    print(name, "points", tuple(pts.shape), "mvn calls", calls.shape[0])


COLOUR_CASES = {
    # name: (n_gaussians, scene_seed, n_cameras, colour_resolution)
    "colour_a": (2500, 1310, 2, 200),
    "colour_b": (1200, 1311, 3, 180),
}


def make_colour(name, n, scene_seed, ncams, res):
    """GaussPythonRenderer of the reference (gauss_render.py:210-465), tile parameters pinned to (60, 60000)."""
    ref = ref_shim.load()
    sc = synth.make_scene(n, seed=scene_seed)
    cams, intr = synth.make_cameras(ncams)
    with ref_shim.cpu_redirect(pinned_tiles=(60, 60000)):
        G = ref.gauss_handler.Gaussians(sc["xyz"].clone(), sc["scales"].clone(), sc["rots"].clone(),
                                        sc["colours"].clone(), sc["opacities"].clone())
        R = ref.gauss_render.get_renderer("python", G.xyz, torch.unsqueeze(torch.clone(G.opacities), 1), G.colours,
                                          G.covariances, visible_gaussian_threshold=0.05)
        imgs = []
        for c2w, k in zip(cams, intr):
            cam = ref.camera_handler.get_camera("python", c2w.clone(), k, colour_resolution=res)
            img, _, _, _ = R(cam)
            imgs.append(img.numpy().astype(np.float32))
        np.savez_compressed(os.path.join(HERE, name + ".npz"),
                            meta=np.array([n, scene_seed, ncams, res], dtype=np.int64),
                            max_contribution=R.gaussian_max_contribution.numpy(),
                            colours=R.gaussian_colours.numpy(), images=np.stack(imgs),
                            visible=R.get_visible_gaussians().numpy())
    print(name, "images", np.stack(imgs).shape, "seen", int((R.gaussian_max_contribution > 0).sum()))


def make_sh(name="sh_a", n=400, seed=1320):
    """eval_sh of the reference (gauss_render.py:43-99), degrees 0..3, on seeded coefficients / unit directions; the
    rendered colour is eval_sh + 0.5 clamped at 0 (forward.cu:65-72)."""
    ref = ref_shim.load()
    g = torch.Generator().manual_seed(seed)
    sh = (0.4 * torch.randn(n, 3, 16, generator=g)).float()
    d = torch.randn(n, 3, generator=g)
    d = (d / d.norm(dim=1, keepdim=True)).float()
    out = {f"deg{deg}": ref.gauss_render.eval_sh(deg, sh[..., : (deg + 1) ** 2], d).numpy() for deg in range(4)}
    np.savez_compressed(os.path.join(HERE, name + ".npz"), meta=np.array([n, seed], dtype=np.int64), **out)
    print(name, {k: v.shape for k, v in out.items()})


def make_live_small(name="live_small", n=600, scene_seed=77, num_points=5000, rng_seed=5):
    """generate_pointcloud of the reference (gauss_to_pc.py:73-371) with the product's eps, default arguments."""
    ref = ref_shim.load()
    sc = synth.make_scene(n, seed=scene_seed)
    eps_fn = lambda g, k, a: philox.draw_eps(g, k, a, rng_seed, 0)
    with ref_shim.cpu_redirect():
        G = ref.gauss_handler.Gaussians(sc["xyz"].clone(), sc["scales"].clone(), sc["rots"].clone(),
                                        sc["colours"].clone() * 255, sc["opacities"].clone())
        G.calculate_normals()
        G.validate_covariances()
        with ref_shim.EpsInjector(ref, G.xyz, eps_fn):
            pts, cols, nrm = ref.gauss_to_pc.generate_pointcloud(G, num_points, device="cpu", quiet=True)
    np.savez_compressed(os.path.join(HERE, name + ".npz"),
                        meta=np.array([n, scene_seed, num_points, rng_seed], dtype=np.int64),
                        points=pts.numpy(), colours=cols.numpy())
    print(name, "points", tuple(pts.shape), pts.dtype, cols.dtype)


TRANSFORM_KINDS = ("json", "colmap_txt", "colmap_bin")


def make_transforms(name="transforms"):
    """load_transform_data of the reference (transform_dataloader.py) on the files tests/test_io_cpu.py writes."""
    import tempfile
    sys.path.insert(0, os.path.dirname(HERE))
    import test_io_cpu as tio
    ref = ref_shim.load()
    out = {}
    with tempfile.TemporaryDirectory() as tmp:
        for kind in TRANSFORM_KINDS:
            path = tio.write_transform_files(tmp, kind)
            for skip in (0, 2):
                tr, ik = ref.transform_dataloader.load_transform_data(path, skip_rate=skip)
                out[f"{kind}_skip{skip}_names"] = np.array(list(tr.keys()))
                out[f"{kind}_skip{skip}_c2w"] = np.array([np.asarray(tr[k], dtype=np.float64) for k in tr])
                out[f"{kind}_skip{skip}_intrinsics"] = np.array([[float(v) for v in ik[k]] for k in tr])
    np.savez_compressed(os.path.join(HERE, name + ".npz"), **out)
    print(name, {k: v.shape for k, v in out.items()})


# n_gaussians, scene_seed, n_cameras, colour_resolution, sampled pixels per image, pixel-sample seed
REF_EXT_CASE = (20000, 1253, 4, 720, 12000, 7)


def load_reference_extension():
    """The reference's compiled `_C` module (oracle/build_ref.py) under a private name; its Python wrapper is not
    needed: the op's 22 arguments are assembled here exactly as the wrapper does (GaussianRasterizer.forward)."""
    import importlib.util
    from oracle import build_ref
    path = build_ref.extension_path()
    if path is None:
        raise SystemExit("reference extension not built: run oracle/build_ref.py")
    spec = importlib.util.spec_from_file_location("g2pc_reference_ext._C", path)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def make_ref_ext(out_dir, name="ref_ext_a"):
    """The reference CUDA rasterizer (renderer_type "cuda", colours precomputed, surface distance on) on REF_EXT_CASE:
    per camera the radii and a fixed pixel sample of the image and depth; per Gaussian the maximum / total
    contribution and the minimum surface distance accumulated over the cameras as the reference's wrapper does."""
    import camera_handler as ch
    from oracle import gaussians as og
    _C = load_reference_extension()
    n, scene_seed, ncams, res, n_pix, pix_seed = REF_EXT_CASE
    dev = "cuda:0"
    sc = synth.make_scene(n, seed=scene_seed, sh_degree=3)
    cov = og.build_covariance(sc["scales"], sc["rots"])
    xyz, opac = sc["xyz"].to(dev).float(), sc["opacities"].to(dev).unsqueeze(1).float()
    colours = sc["colours"].to(dev).float()
    cov6 = cov.to(dev).reshape(-1, 9)[:, [0, 1, 2, 4, 5, 8]].float()  # strip_symmetric
    empty = torch.Tensor([])
    max_c = torch.zeros(n, device=dev)
    tot_c = torch.zeros(n, device=dev)
    min_sd = torch.full((n,), torch.finfo(torch.float).max, device=dev)
    cams, intr = synth.make_cameras(ncams)
    radii_all, img_s, dep_s, pix = [], [], [], None
    for c2w, k in zip(cams, intr):
        rs = ch.get_camera("cuda", c2w.to(dev), k, colour_resolution=res)
        H, W = rs.image_height, rs.image_width
        if pix is None:
            pix = np.sort(np.random.default_rng(pix_seed).choice(H * W, n_pix, replace=False)).astype(np.int32)
        mask = torch.full((H * W,), 1, device=dev, dtype=torch.int)
        out = _C.rasterize_gaussians(rs.bg, xyz, colours, opac, empty, empty, rs.scale_modifier, cov6, rs.viewmatrix,
                                     rs.projmatrix, rs.tanfovx, rs.tanfovy, H, W, empty, rs.sh_degree, rs.campos, mask,
                                     rs.prefiltered, rs.antialiasing, True, rs.debug)
        _, colour, depth, radii, _, _, _, _, contrib, surf, _ = out
        upd = contrib > max_c
        max_c[upd] = contrib[upd]
        tot_c += contrib
        upd = surf < min_sd
        min_sd[upd] = surf[upd]
        assert int(radii.max()) < 2 ** 15
        radii_all.append(radii.cpu().numpy().astype(np.int16))
        img_s.append(colour.reshape(3, -1)[:, pix].cpu().numpy())
        dep_s.append(depth.reshape(-1)[pix].cpu().numpy())
    path = os.path.join(out_dir, name + ".npz")
    np.savez_compressed(path, meta=np.array(REF_EXT_CASE, dtype=np.int64), image_hw=np.array([H, W]), pixels=pix,
                        radii=np.stack(radii_all), image=np.stack(img_s), depth=np.stack(dep_s),
                        max_contribution=max_c.cpu().numpy(), total_contribution=tot_c.cpu().numpy(),
                        min_surface_distance=min_sd.cpu().numpy())
    print(name, path, os.path.getsize(path), "bytes")


CPU_CASES = {"sh": make_sh,
             **{k: (lambda k=k: make_sampling(k, *SAMPLING_CASES[k])) for k in SAMPLING_CASES},
             **{k: (lambda k=k: make_colour(k, *COLOUR_CASES[k])) for k in COLOUR_CASES},
             "live_small": make_live_small, "transforms": make_transforms}


if __name__ == "__main__":
    torch.manual_seed(0)
    if sys.argv[1:2] == ["ref_ext"]:
        make_ref_ext(sys.argv[2] if len(sys.argv) > 2 else HERE)
    else:
        for case in sys.argv[1:] or list(CPU_CASES):
            CPU_CASES[case]()
