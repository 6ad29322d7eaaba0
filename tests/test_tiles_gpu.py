"""GPU parity tests of the renderer_type="cuda" colour back-end (csrc/s7_tiles.cu through the C ABI):
  * against the CPU oracle oracle/render_cuda.py (restatement of the reference's CUDA rasterizer, deterministic);
  * against the stored outputs of the UNMODIFIED reference extension (tests/golden/ref_ext_a.npz; its results race, so
    tolerances + mask IoU instead of exactness, SURVEY.md §8a);
  * the op surface `_C.rasterize_gaussians` (22 arguments -> 11-tuple) and the CLI with its default flags.
"""
import numpy as np
import pytest
import torch

from util import scene_to

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _scene(n, seed):
    from g2pc import synth
    from oracle import gaussians as og
    sc = synth.make_scene(n, seed=seed, sh_degree=3)
    cov = og.build_covariance(sc["scales"], sc["rots"])
    return sc, cov


@pytest.mark.parametrize("n,res,ncams,surf,masked", [(2500, 200, 3, False, False), (4000, 330, 2, True, False),
                                                     (2500, 200, 2, True, True), (12000, 720, 1, True, False)])
def test_tiles_parity_vs_oracle(lib, n, res, ncams, surf, masked):
    import camera_handler as ch
    import gauss_render as gr
    from g2pc import synth
    from oracle import render_cuda as orc
    sc, cov = _scene(n, 1250)
    d = scene_to(sc, DEV)
    R = gr.get_renderer("cuda", d["xyz"], d["opacities"].unsqueeze(1), d["colours"], cov.to(DEV),
                        visible_gaussian_threshold=0.05, surface_distance_std=2.0 if surf else None,
                        calculate_surface_distance=surf)
    O = orc.CudaRasterizerOracle(sc["xyz"], sc["opacities"], sc["colours"].float(), cov, calculate_surface_distance=surf)
    cams, intr = synth.make_cameras(ncams)
    for c2w, k in zip(cams, intr):
        mask = None
        if masked:  # native-size mask: the image is not rescaled (camera_handler.py:55-61)
            k = [res, int(res * 9 / 16), k[2] * res / k[0], k[3] * res / k[0]]
            g = torch.Generator().manual_seed(3)
            mask = (torch.rand(k[1], k[0], generator=g) > 0.3).to(torch.int32)
        rs = ch.get_camera("cuda", c2w.to(DEV), k, colour_resolution=res, mask=None if mask is None else mask.to(DEV))
        ors = orc.RasterSettings(c2w, k, colour_resolution=res, mask=None if mask is None else mask.numpy())
        img, radii, invd, dep = R(rs)
        oimg, oradii, oinvd, odep = O(ors)
        pre = O.last["pre"]
        assert img.shape == (3, rs.image_height, rs.image_width) and dep.shape == (1, rs.image_height, rs.image_width)
        rflip = int((radii.cpu().numpy() != oradii).sum())
        assert rflip <= max(1, int(3e-4 * n)), f"{rflip} radius / cull flips"
        same = radii.cpu().numpy() == oradii
        derr = np.abs(img.cpu().numpy() - oimg)
        assert int((derr > 1e-4).sum()) <= int(1e-4 * derr.size) + 3 * rflip * 256 and derr.max() < 5e-3, \
            f"image: max {derr.max():.2e}, {(derr > 1e-4).sum()} off"
        dd = np.abs(dep.cpu().numpy() - odep)
        # (a pixel that stops one Gaussian earlier / later — T on the 1e-4 threshold — moves its depth by that Gaussian's share)
        assert int((dd > 2e-4).sum()) <= int(3e-4 * dd.size) + 3 * rflip * 256 and dd.max() < 2e-2
        di = np.abs(invd.cpu().numpy() - oinvd)
        assert int((di > 1e-4).sum()) <= int(1e-4 * di.size) + 3 * rflip * 256
    kmax, omax = R.gaussian_max_contribution.cpu().numpy(), O.gaussian_max_contribution
    ktot, otot = R.gaussian_total_contribution.cpu().numpy(), O.gaussian_total_contribution
    n_off = int((np.abs(kmax - omax) > 1e-4).sum())
    assert n_off <= max(2, int(5e-4 * n)), f"{n_off} max contributions off"
    assert int((np.abs(ktot - otot) > 1e-4 * ncams).sum()) <= max(2, int(1e-3 * n))
    kcol, ocol = R.gaussian_colours.cpu().numpy(), O.gaussian_colours
    c_off = int((np.abs(kcol - ocol).max(axis=1) > 1e-4).sum())
    assert c_off <= max(3, int(2e-3 * n)), f"{c_off} colours off (near-tied arg-max pixels)"
    flips = int(((kmax > 0.05) != (omax > 0.05)).sum())
    assert flips <= max(1, int(3e-4 * n))
    msg = f"[tiles parity] n={n} res={res}: contrib off {n_off}, colours off {c_off}, visibility flips {flips}"
    if surf:
        kd, od = R.gaussian_min_surface_distance.cpu().numpy(), O.gaussian_min_surface_distance
        fin = (kd < 1e38) & (od < 1e38)
        assert int(((kd < 1e38) != (od < 1e38)).sum()) <= max(2, int(1e-3 * n))
        # |depth_j - E_p| with E_p ~ 1..6 carrying ~1e-5 of fp32 / ex2.approx noise: absolute tolerance
        rel = np.abs(kd[fin] - od[fin])
        assert int((rel > 2e-4).sum()) <= max(3, int(5e-3 * fin.sum())), f"{(rel > 2e-4).sum()} surface distances off"
        km = R.get_gaussians_with_low_surface_distance().cpu().numpy()
        om = O.low_surface_distance_mask(2.0)
        iou = (km & om).sum() / max(1, (km | om).sum())
        assert iou > 0.995
        msg += f", surface dist off {(rel > 2e-4).sum()}/{fin.sum()}, cull mask IoU {iou:.4f}"
    print(msg)


def test_tiles_sh_layouts_and_async(lib):
    """SH colour (deg 3) through both coefficient layouts gives the python back-end's per-camera colours; async mode with
    a tiny instance buffer replays exactly."""
    import camera_handler as ch
    import gauss_render as gr
    from g2pc import synth
    from g2pc.rasterizer import GaussianRasterizer
    from oracle import render as orr
    sc, cov = _scene(3000, 1251)
    d = scene_to(sc, DEV)
    cams, intr = synth.make_cameras(3)
    R0 = gr.get_renderer("cuda", d["xyz"], d["opacities"].unsqueeze(1), d["colours"], cov.to(DEV), shs=d["shs"])
    R1 = GaussianRasterizer(d["xyz"].float(), None, d["opacities"].float(), shs=d["shs"].float().permute(0, 2, 1).contiguous(),
                            cov3D_precomp=cov.to(DEV), sh_layout=1)
    R1.async_mode = True
    R1._inst_cap = 512
    for c2w, k in zip(cams, intr):
        rs = ch.get_camera("cuda", c2w.to(DEV), k, colour_resolution=200, sh_degree=3)
        R0(rs)
        R1(rs)
    R1.flush()
    assert R1.replays >= 1
    assert torch.equal(R0.gaussian_max_contribution, R1.gaussian_max_contribution)
    assert torch.equal(R0.gaussian_colours, R1.gaussian_colours)
    # per-camera SH colours of the last camera against the (pinned) SH oracle
    ocam = orr.Camera(cams[-1], intr[-1], colour_resolution=200)
    dirs = sc["xyz"] - ocam.camera_center[None, :]
    dirs = dirs / dirs.norm(dim=1, keepdim=True)
    want = orr.sh_colour(3, sc["shs"].float(), dirs.float()).numpy()
    R0.flush()
    proj = R0._slots[R0._last_slot]["proj"].cpu().numpy()
    seen = proj[:, 11] > 0
    assert np.abs(proj[seen][:, [6, 7, 8]] - want[seen]).max() < 3e-6


def test_rasterize_gaussians_op_surface(lib):
    """The native-op stand-in: 22 positional arguments -> the reference's 11-tuple (rasterize_points.cu:36-145)."""
    import camera_handler as ch
    from g2pc import synth
    import gaussian_pointcloud_rasterization as gpr
    sc, cov = _scene(1500, 1252)
    d = scene_to(sc, DEV)
    cams, intr = synth.make_cameras(1)
    rs = ch.get_camera("cuda", cams[0].to(DEV), intr[0], colour_resolution=180)
    cov6 = cov.reshape(-1, 9)[:, [0, 1, 2, 4, 5, 8]].to(DEV)
    n = 1500
    H, W = rs.image_height, rs.image_width
    mask = torch.ones(H * W, dtype=torch.int32, device=DEV)
    empty = torch.Tensor([])
    out = gpr._C.rasterize_gaussians(rs.bg, d["xyz"], d["colours"].float(), d["opacities"].unsqueeze(1), empty, empty, 1.0,
                                     cov6, rs.viewmatrix, rs.projmatrix, rs.tanfovx, rs.tanfovy, H, W, empty, 3, rs.campos,
                                     mask, False, False, True, True)
    assert len(out) == 11
    num, colour, depth, radii, gb, bb, ib, invd, contrib, surf, pix = out
    assert isinstance(num, int) and num > 0
    assert colour.shape == (3, H, W) and depth.shape == (1, H, W) and invd.shape == (1, H, W)
    assert radii.shape == (n,) and radii.dtype == torch.int32 and pix.dtype == torch.int32
    assert contrib.shape == (n,) and surf.shape == (n,) and float(contrib.max()) <= 0.99 + 1e-6
    assert int((pix >= H * W).sum()) == 0 and torch.isfinite(colour).all()
    # same camera through the class API gives the same per-camera contributions
    R = gpr.GaussianRasterizer(d["xyz"].float(), None, d["opacities"].float(), colors_precomp=d["colours"].float(),
                               cov3D_precomp=cov6, calculate_surface_distance=True)
    c2, r2, i2, d2 = R(rs)
    assert torch.equal(c2, colour) and torch.equal(R.gaussian_max_contribution, contrib)
    assert torch.equal(R.gaussian_min_surface_distance, surf)


def test_tiles_vs_reference_extension(lib):
    """Kernels against the unmodified reference rasterizer (built for sm_100, run on a B200): its radii and a fixed
    pixel sample of every image / depth map, and the per-Gaussian contributions and surface distances accumulated over
    the cameras, as stored by tests/golden/make_golden.py (ref_ext)."""
    import os
    import camera_handler as ch
    import gauss_render as gr
    from g2pc import synth
    from util import GOLDEN
    g = np.load(os.path.join(GOLDEN, "ref_ext_a.npz"))
    n, scene_seed, ncams, res, _, _ = [int(v) for v in g["meta"]]
    pix = torch.from_numpy(g["pixels"].astype(np.int64)).to(DEV)
    sc, cov = _scene(n, scene_seed)
    d = scene_to(sc, DEV)
    cams, intr = synth.make_cameras(ncams)
    R = gr.get_renderer("cuda", d["xyz"], d["opacities"].unsqueeze(1), d["colours"], cov.to(DEV),
                        surface_distance_std=2.0, calculate_surface_distance=True)
    worst = 0.0
    for i, (c2w, k) in enumerate(zip(cams, intr)):
        rs = ch.get_camera("cuda", c2w.to(DEV), k, colour_resolution=res)
        img, radii, invd, dep = R(rs)
        assert (rs.image_height, rs.image_width) == tuple(int(v) for v in g["image_hw"])
        rradii = torch.from_numpy(g["radii"][i].astype(np.int32)).to(DEV)
        assert int((radii != rradii).sum()) <= max(1, int(3e-4 * n))
        e = (img.reshape(3, -1)[:, pix] - torch.from_numpy(g["image"][i]).to(DEV)).abs()
        assert float(e.max()) < 5e-3 and int((e > 2e-4).sum()) <= int(2e-4 * e.numel())
        worst = max(worst, float(e.max()))
        ed = (dep.reshape(-1)[pix] - torch.from_numpy(g["depth"][i]).to(DEV)).abs()
        assert int((ed > 1e-3).sum()) <= int(2e-4 * ed.numel())
    # The reference publishes a Gaussian's per-tile maximum WITHOUT a barrier between the blend loop and the read of the
    # shared maximum (forward.cu:447-456 follows :392-445 directly): a thread whose pixel has finished reads the entry
    # before slower warps have written theirs, so the reference UNDER-reports contributions run-dependently.  The
    # deterministic maximum can therefore only be compared one-sidedly: never below the reference's (up to rounding).
    km, rm = R.gaussian_max_contribution, torch.from_numpy(g["max_contribution"]).to(DEV)
    below = int((km < rm - 1e-4).sum())
    off = int(((km - rm).abs() > 1e-4).sum())
    flips = int(((km > 0.05) != (rm > 0.05)).sum())
    lost = int(((rm > 0.05) & ~(km > 0.05)).sum())
    kt, rt = R.gaussian_total_contribution, torch.from_numpy(g["total_contribution"]).to(DEV)
    tbelow = int((kt < rt - 4e-4).sum())
    toff = int(((kt - rt).abs() > 4e-4).sum())
    # the reference wrapper's selection (get_surface_gaussians_below_distance_threshold) on its stored distances
    rd = torch.from_numpy(g["min_surface_distance"]).to(DEV)
    rsel = rd < torch.std_mean(rd[rd < torch.finfo(torch.float).max])[1] * 2.0
    ksel = R.get_gaussians_with_low_surface_distance()
    iou = float((ksel & rsel).sum()) / max(1.0, float((ksel | rsel).sum()))
    print(f"[vs reference ext] image max diff {worst:.2e}; max contribution: {below} below the reference's, {off}/{n} differ "
          f"(reference under-reports, see comment); total: {tbelow} below, {toff} differ; visibility flips {flips} "
          f"({lost} visible only in the reference); surface-distance cull mask IoU {iou:.4f} (kept {int(ksel.sum())} vs "
          f"{int(rsel.sum())})")
    assert below <= max(2, int(2e-4 * n)) and tbelow <= max(2, int(5e-4 * n)) and lost <= max(1, int(1e-4 * n))
    assert iou > 0.9


def test_cli_default_flags_and_surface_distance(lib, tmp_path):
    """The CLI with its DEFAULT renderer (cuda) and with --surface_distance_std (ADVICE r1: both used to crash)."""
    import gauss_dataloader as gd
    import gauss_to_pc as g2p
    from g2pc import synth
    from test_io_cpu import write_gaussian_ply, write_transforms_json
    sc = synth.make_scene(3000, seed=22, sh_degree=3)
    cams, intr = synth.make_cameras(3)
    ply, tj, out = str(tmp_path / "scene.ply"), str(tmp_path / "transforms.json"), str(tmp_path / "pc.ply")
    write_gaussian_ply(ply, sc)
    write_transforms_json(tj, cams, intr)
    g2p.main(["--input_path", ply, "--transform_path", tj, "--output_path", out, "--num_points", "30000",
              "--colour_quality", "tiny", "--quiet"])
    v = gd.read_ply_vertices(out)
    assert abs(v.shape[0] - 30000) < 900 and v["red"].max() > 0
    g2p.main(["--input_path", ply, "--transform_path", tj, "--output_path", out, "--num_points", "30000",
              "--colour_quality", "tiny", "--surface_distance_std", "2.0", "--exact_num_points", "--quiet"])
    v2 = gd.read_ply_vertices(out)
    assert abs(v2.shape[0] - 30000) < 300
    with pytest.raises(AttributeError):
        g2p.config_parser(["--input_path", ply, "--transform_path", tj, "--generate_mesh"])
