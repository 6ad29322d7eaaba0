"""3DGS -> point cloud: CLI, pipeline driver and the sampling stage — drop-in for the reference's gauss_to_pc.py.

Reference: /root/reference/gauss_to_pc.py.  Same flags (:607-646), same settings tuple (:26-60), same public
functions and argument order (distribute_points :73, mahalanobis :92, calculate_bin_sizes :105,
sample_from_multivariate_normal :140, create_new_gaussian_points :157, generate_pointcloud :277,
convert_3dgs_to_pc :373).  The sampling stage runs as two fused sm_100a kernels (csrc/s2_sample.cu) driven by
g2pc/sampler.py; the colour stage runs through gauss_render.get_renderer.  No CPU fallback.
"""
from typing import NamedTuple

import numpy as np
import torch

from gauss_handler import Gaussians
from gauss_render import get_renderer
from camera_handler import get_camera
from g2pc import capi, config, sampler
from g2pc.trace import nvtx

LAST_SAMPLE_STATS = {}
LAST_RENDER_STATS = {}
COLOR_QUALITY_OPTIONS = {"tiny": 180, "low": 360, "medium": 720, "high": 1280, "ultra": 1920, "original": None}


class GaussPointCloudSettings(NamedTuple):
    """Same fields, same order as the reference (gauss_to_pc.py:26-60)."""
    renderer_type: str
    num_points: int
    prioritise_visible_gaussians: bool
    mahalanobis_distance_std: float
    camera_skip_rate: int
    render_colours: bool
    min_opacity: float
    bounding_box_min: list
    bounding_box_max: list
    calculate_normals: bool
    cull_large_percentage: float
    remove_unrendered_gaussians: bool
    colour_resolution: int
    max_sh_degree: int
    exact_num_points: int
    visibility_threshold: float
    surface_distance_std: float
    generate_mesh: bool
    quiet: bool
    device: str


class PointCloudData(NamedTuple):
    points: torch.Tensor
    colours: torch.Tensor
    normals: torch.Tensor


def imwrite(path, image):
    """Save a rendered image (debug helper, gauss_to_pc.py:67-71)."""
    import imageio
    imageio.imwrite(path, ((255 * np.clip(image, 0, 1)).astype(np.uint8)))


def distribute_points(gaussian_sizes, num_points):
    """Points per Gaussian proportional to its size (gauss_to_pc.py:73-90): round(size * P / sum(size)), then the
    first min(deficit, #zeros) Gaussians with zero points get one."""
    ratio = num_points / torch.sum(gaussian_sizes)
    points_per_gaussian = torch.round(gaussian_sizes * ratio)
    is_zero = points_per_gaussian == 0
    deficit = num_points - points_per_gaussian.sum()
    # (one host sync, like the reference's .item())
    take = int(min(deficit.item(), int(is_zero.sum().item())))
    zero_rank = torch.cumsum(is_zero.to(torch.int64), 0)  # 1-based rank among the zero entries
    if take >= 0:
        promote = is_zero & (zero_rank <= take)
    else:  # python slice [:negative] keeps all but the last |take| zero entries — reproduced knowingly
        promote = is_zero & (zero_rank <= int(is_zero.sum().item()) + take)
    points_per_gaussian[promote] = 1
    return points_per_gaussian


def mahalanobis(means, samples, covs):
    """sqrt(d^T Sigma^-1 d) for d = mu - x (gauss_to_pc.py:92-103).  Stand-alone helper kept for API parity; inside
    the pipeline the test is fused into g2pc_sample_count."""
    delta = (means - samples).unsqueeze(2)
    m = torch.bmm(delta.transpose(1, 2), torch.bmm(torch.inverse(covs), delta))
    return torch.sqrt(m).squeeze(1).squeeze(1)


def calculate_bin_sizes(points_per_gaussian):
    """Heuristic deciding from which point count on Gaussians are batched into wider bins (gauss_to_pc.py:105-138)."""
    hist = torch.bincount(points_per_gaussian).cpu().numpy()
    return sampler.calculate_bin_sizes_from_hist(hist[np.nonzero(hist)[0]])


def _attempt_ladder(num_attempts):
    """Stored-attempt sizes to try: most Gaussians finish within a few attempts, so the count pass first keeps
    config.ATTEMPTS_STORED_FIRST dense attempts; if some Gaussian still emits later (status word ST_OVERFLOW, e.g. a
    small --mahalanobis_distance_std with --exact_num_points) the deterministic stream is simply replayed with every
    attempt stored.  The reference has no such limit (gauss_to_pc.py:189-263)."""
    num_attempts = int(num_attempts)
    if num_attempts > 255:
        raise capi.G2pcError("num_sample_attempts must be <= 255 (8-bit attempt tag in the emit pass)")
    first = min(num_attempts, config.ATTEMPTS_STORED_FIRST)
    return [first] if first == num_attempts else [first, num_attempts]


def _single_bin_run(k, means, covariances, colours, normals, std, num_attempts, include_centres, seed, call_id,
                    out_dtype=None, cull_mode=None):
    n = means.shape[0]
    perm = torch.arange(n, dtype=torch.int32, device=means.device)
    for A in _attempt_ladder(num_attempts):
        plan = sampler.SamplePlan([(int(k), n)], A, include_centres=include_centres)
        res = sampler.run_plan(plan, means.to(torch.float32), covariances.to(torch.float32), colours, normals, perm,
                               num_attempts, std, seed, call_id, out_dtype=out_dtype, cull_mode=cull_mode,
                               want_normals=normals is not None)
        if A == num_attempts or not int(res[4][capi.ST_OVERFLOW].item()):
            break
    return res


def sample_from_multivariate_normal(means, covariances, num_points_to_sample, max_num_gen_attempts=3, epsilon=1e-6):
    """num_points_to_sample draws from every N(mean, cov) (gauss_to_pc.py:140-155) -> (k, n, 3).  Covariances that
    need it are regularised by +epsilon*I per try inside the kernel (per Gaussian, not per batch)."""
    k = int(num_points_to_sample)
    n = means.shape[0]
    dummy = torch.zeros((n, 3), dtype=torch.float32, device=means.device)
    pts, _, _, total, status, _ = _single_bin_run(k, means, covariances, dummy, None, float("inf"), 1, False,
                                                   config.SEED, sampler.next_call_id(),
                                                   cull_mode=capi.CULL_EPS_NORM)
    if int(status[capi.ST_CHOLFAIL].item()) > 0:
        return None
    return pts[: n * k].view(n, k, 3).transpose(0, 1).contiguous()


def create_new_gaussian_points(num_points_to_sample, means, covariances, colours, mahalanobis_distance_std=2,
                               num_attempts=5, normals=None, max_num_gen_attemps=3, device="cuda:0"):
    """Sample up to num_points_to_sample points per Gaussian, re-drawing for at most num_attempts rounds; per round a
    Gaussian emits the first min(remaining, #accepted) samples of its block (gauss_to_pc.py:157-275).

    Returns (new_points, new_colours, new_normals) in the reference's order (attempt-major, Gaussian-minor)."""
    k = int(num_points_to_sample)
    pts, cols, nrm, total, status, _ = _single_bin_run(k, means, covariances, colours, normals,
                                                       mahalanobis_distance_std, num_attempts, False, config.SEED,
                                                       sampler.next_call_id())
    t = int(total.item())
    _check_status(status)
    return pts[:t], cols[:t], (nrm[:t] if nrm is not None else None)


def _check_status(status):
    s = status.tolist()
    if s[capi.ST_OVERFLOW]:  # cannot happen through the drivers in this module (they replay with every attempt stored)
        raise capi.G2pcError("the count pass stored fewer attempts than some Gaussian needed; re-run with "
                             "attempts_stored = num_attempts")
    if s[capi.ST_CHOLFAIL] and not getattr(config, "QUIET_CHOL", False):
        print(f"WARNING: Could not generate points for {s[capi.ST_CHOLFAIL]} Gaussians "
              "(covariance not positive-definite even after regularisation)")


def generate_pointcloud(gaussians, num_points, contributions=None, mahalanobis_distance_std=2,
                        exact_num_points=False, calculate_normals=True, num_sample_attempts=5, device="cuda:0",
                        quiet=False, seed=None, call_id=None, gid_offset=0, return_debug=False):
    """
    Generates a pointcloud from a set of gaussians  (reference: gauss_to_pc.py:277-371)

    Args / returns as the reference: (total_points (P,3) f32, total_colours (P,3), total_normals (P,3) | None), in
    the reference's order: per bin the Gaussian centres, then the samples attempt-major / Gaussian-minor.
    Extra keyword-only knobs: seed / call_id (Philox stream), gid_offset (global id of row 0 when the Gaussian
    array is a shard).
    """
    seed = config.SEED if seed is None else seed
    call_id = sampler.next_call_id() if call_id is None else call_id

    # magnitudes (gauss_handler.py:252-279) and the point budget (distribute_points, :73-90) on the device, no host sync
    points_per_gaussian, _ = gaussians.points_per_gaussian(num_points, contributions)

    if not quiet:
        print("Distributed Points to Gaussians")
        print()

    res = sample_points_per_gaussian(gaussians.xyz, gaussians.covariances, gaussians.colours,
                                     gaussians.normals if calculate_normals else None, points_per_gaussian,
                                     mahalanobis_distance_std, exact_num_points, num_sample_attempts, seed, call_id,
                                     gid_offset=gid_offset, quiet=quiet, gids=getattr(gaussians, "ids", None))
    pts, cols, nrm, total, status, dbg = res
    t = int(total.item())  # the one sync of the stage (the reference syncs per bin and per attempt)
    _check_status(status)
    out = (pts[:t], cols[:t], (nrm[:t] if nrm is not None else None))
    if return_debug:
        return out + ({"points_per_gaussian": points_per_gaussian, **dbg},)
    return out


def sample_points_per_gaussian(xyz, covariances, colours, normals, points_per_gaussian, mahalanobis_distance_std,
                               exact_num_points, num_sample_attempts, seed, call_id, gid_offset=0, quiet=True,
                               hist=None, gids=None, global_bins=None):
    """Bin planning on the host (from the histogram, as the reference does) + the two S2 kernels.
    Everything is enqueued asynchronously; the caller syncs once on the returned total.
    gids: global Gaussian id per row (keys the RNG; survives culls / sharding).  global_bins: bins planned on the
    histogram of ALL ranks (g2pc.dist); the local member counts are taken from this rank's histogram."""
    dev = xyz.device
    ppg = points_per_gaussian.to(torch.int64)
    if hist is None:
        hist = torch.bincount(ppg).cpu().numpy()  # host needs the histogram to lay out bins (reference: :110-115)
    if global_bins is not None:
        from g2pc import dist as gdist
        bins = [b for b in gdist.local_bin_counts(global_bins, hist) if b[3] > 0]
    else:
        bins = sampler.plan_bins(hist, exact_num_points)
    if not quiet:
        print("Starting Point Cloud Generation")

    # value -> bin lookup, then a stable sort brings the Gaussians into bin order (index order inside a bin)
    lut = np.full((hist.shape[0],), len(bins), dtype=np.int64)
    for b, (start, end, n, count) in enumerate(bins):
        lo, hi = int(np.ceil(start)), int(np.ceil(end))
        lut[max(lo, 0):max(hi, 0)] = b
    bin_of = torch.from_numpy(lut).to(dev)[ppg]
    order = torch.sort(bin_of, stable=True).indices
    n_used = int(sum(c for (_, _, _, c) in bins))
    perm = order[:n_used].to(torch.int32)
    global LAST_SAMPLE_STATS
    LAST_SAMPLE_STATS = {"n_active": n_used, "bins": len(bins), "n_gaussians": int(xyz.shape[0])}

    for A in _attempt_ladder(num_sample_attempts):
        plan = sampler.SamplePlan([(n - 1, count) for (_, _, n, count) in bins], A, include_centres=True)
        pts, cols, nrm, total, status, bufs = sampler.run_plan(
            plan, xyz.to(torch.float32), covariances.to(torch.float32), colours, normals, perm, num_sample_attempts,
            mahalanobis_distance_std, seed, call_id, gid_offset=gid_offset, want_normals=normals is not None,
            gids=gids)
        # (the overflow word is read only when a replay is possible; callers sync on `total` right after anyway)
        if A == int(num_sample_attempts) or not int(status[capi.ST_OVERFLOW].item()):
            break
    dbg = {"bins": bins, "perm": perm, "plan": plan, "buffers": bufs}
    return pts, cols, nrm, total, status, dbg


def convert_3dgs_to_pc(input_path, transform_path, mask_path, pointcloud_settings):
    """
    Generates a pointcloud from a 3DGS file  (reference: gauss_to_pc.py:373-601; same stages in the same order)

    Returns (total_point_cloud, surface_point_cloud) as PointCloudData tuples.
    """
    from transform_dataloader import load_transform_data
    from mask_dataloader import load_image_masks
    from gauss_dataloader import load_gaussians

    s = pointcloud_settings
    say = (lambda *a: None) if s.quiet else print
    transforms, intrinsics, mask_images = None, None, None

    if transform_path is not None:
        say("Loading Camera Poses\n")
        transforms, intrinsics = load_transform_data(transform_path, skip_rate=s.camera_skip_rate)

    if mask_path is not None:
        say("Loading Masks\n")
        mask_images = load_image_masks(mask_path)
        for mask_name in mask_images.keys():
            if mask_name not in transforms.keys():
                print(f"WARNING: Mask with name {mask_name} not found in provided transforms")

    say("Loading Gaussians from File\n")
    xyz, scales, rots, colours, opacities, shs = load_gaussians(input_path, max_sh_degree=s.max_sh_degree)
    return convert_gaussians_to_pc(xyz, scales, rots, colours, opacities, shs, transforms, intrinsics, mask_images, s)


def convert_gaussians_to_pc(xyz, scales, rots, colours, opacities, shs, transforms, intrinsics, mask_images,
                            pointcloud_settings, render_shs=False):
    """The device-resident part of convert_3dgs_to_pc (gauss_to_pc.py:414-601): everything between the loaders and the
    PLY writer.  transforms: {name: 4x4 c2w (nested list / tensor)} or None; intrinsics: {name: [w, h, fx, fy]}.
    render_shs=True evaluates the SH colour per camera inside the colour stage (the reference's CLI never passes the SH
    coefficients to its renderer, gauss_to_pc.py:429-432; get_renderer accepts them)."""
    s = pointcloud_settings
    say = (lambda *a: None) if s.quiet else print

    with nvtx("g2pc: covariances + normals"):
        gaussians = Gaussians(xyz, scales, rots, colours, opacities, shs=shs)

        if s.calculate_normals:
            gaussians.calculate_normals()

    total_gaussian_contributions = None

    if s.render_colours:
        say("Rendering Gaussian Colours")

        want_surface = True if (s.surface_distance_std is not None or s.generate_mesh) else False
        gaussian_renderer = get_renderer(s.renderer_type, gaussians.xyz, torch.unsqueeze(torch.clone(gaussians.opacities), 1),
                                         gaussians.colours, gaussians.covariances,
                                         shs=gaussians.shs if render_shs else None,
                                         visible_gaussian_threshold=s.visibility_threshold,
                                         surface_distance_std=s.surface_distance_std,
                                         calculate_surface_distance=want_surface)
        # the driver never looks at the rendered images before the getters: let the renderer run ahead of the host
        if hasattr(gaussian_renderer, "async_mode"):
            gaussian_renderer.async_mode = True

        if transforms is None:
            raise Exception("Transforms are required to render colours")

        for img_name, transform in transforms.items():
            # the 4x4 pose stays on the host: the camera matrices are kernel arguments, not device data
            transform = torch.as_tensor(transform, dtype=torch.float32) if not torch.is_tensor(transform) else transform
            mask = None
            if mask_images is not None and img_name in mask_images.keys():
                mask = mask_images[img_name].to(s.device)
            camera = get_camera(s.renderer_type, transform, intrinsics[img_name], colour_resolution=s.colour_resolution,
                                sh_degree=s.max_sh_degree, white_bkgd=True, mask=mask)
            with nvtx(f"g2pc: camera {img_name}"):
                render, _, _, depth_map = gaussian_renderer(camera)

        say(f"\nNumber Initial Gaussians: {gaussians.xyz.shape[0]}")

        gaussians.colours = gaussian_renderer.get_gaussian_colours()

        # every cull of gauss_to_pc.py:483-496 in one fused mask + compaction (csrc/s8_cull.cu): surface distance,
        # visibility, min opacity, bounding box (+ the size-percentile cull, which needs a sort, through filter_indices)
        surface_mask = None
        if s.surface_distance_std is not None:
            surface_mask = gaussian_renderer.get_gaussians_with_low_surface_distance()
        gaussians.cull_large_gaussians(s.cull_large_percentage)
        gaussian_renderer.flush() if hasattr(gaussian_renderer, "flush") else None
        culled_indices = gaussians.fused_cull(
            max_contribution=gaussian_renderer.gaussian_max_contribution if s.remove_unrendered_gaussians else None,
            visibility_threshold=gaussian_renderer.visible_gaussian_threshold, min_opacity=s.min_opacity,
            bounding_box_min=s.bounding_box_min, bounding_box_max=s.bounding_box_max, extra_mask=surface_mask)

        say(f"\nNumber Gaussians after Culling: {gaussians.xyz.shape[0]}")

        if gaussians.xyz.shape[0] < 1:
            raise Exception("Number of Gaussians after culling is 0, meaning a point cloud cannot be generated")

        if s.generate_mesh:
            surface_gaussian_idxs = gaussian_renderer.get_predicted_surface_gaussians(predicted_surface_std=1.0)
            surface_gaussian_idxs = surface_gaussian_idxs[culled_indices]

        if s.prioritise_visible_gaussians:
            total_gaussian_contributions = gaussian_renderer.get_total_gaussian_contributions()[culled_indices]

        global LAST_RENDER_STATS
        LAST_RENDER_STATS = {"stats": getattr(gaussian_renderer, "_stats", None),
                             "replays": getattr(gaussian_renderer, "replays", 0)}
        del gaussian_renderer
    else:
        gaussians.colours = gaussians.colours * 255
        say("Skipping Rendering Gaussian Colours")

    say("\nEnsuring Gaussians are Positive Semidefinite")

    with nvtx("g2pc: validate covariances"):
        valid = gaussians.validate_covariances()

    if total_gaussian_contributions is not None:
        total_gaussian_contributions = total_gaussian_contributions[valid]

    num_sample_attempts = 5 if not s.exact_num_points else 100

    say("\nStarting Point Cloud Generation for All Gaussians\n")

    with nvtx("g2pc: point budget + sampling"):
        points, colours, normals = generate_pointcloud(gaussians, s.num_points, exact_num_points=s.exact_num_points,
                                                       mahalanobis_distance_std=s.mahalanobis_distance_std,
                                                       calculate_normals=s.calculate_normals,
                                                       num_sample_attempts=num_sample_attempts,
                                                       contributions=total_gaussian_contributions,
                                                       device=s.device, quiet=s.quiet)

    total_point_cloud = PointCloudData(points=points, colours=colours, normals=normals)
    surface_point_cloud = None

    if s.generate_mesh and s.render_colours:
        say("Starting Point Cloud Generation for Surface Gaussians\n")
        surface_gaussian_idxs = surface_gaussian_idxs[valid]
        gaussians.add_gaussians_to_cull(surface_gaussian_idxs)
        gaussians.filter_gaussians()
        avg_points_per_gauss_for_mesh = 25
        total_mesh_points = min(s.num_points // 2, int(gaussians.xyz.shape[0] * avg_points_per_gauss_for_mesh))
        points, colours, normals = generate_pointcloud(gaussians, total_mesh_points, exact_num_points=s.exact_num_points,
                                                       num_sample_attempts=num_sample_attempts,
                                                       contributions=total_gaussian_contributions[surface_gaussian_idxs],
                                                       device=s.device, quiet=s.quiet)
        surface_point_cloud = PointCloudData(points=points, colours=colours, normals=normals)

    return total_point_cloud, surface_point_cloud


def config_parser(argv=None):
    """Same flags and validation as the reference (gauss_to_pc.py:603-710).  configargparse is optional in this
    image; argparse accepts the same flag names."""
    try:
        import configargparse as ap
    except ImportError:
        import argparse as ap

    parser = ap.ArgumentParser()

    parser.add_argument("--input_path", type=str, required=True, help="Path to ply or splat file to convert to a point cloud")
    parser.add_argument("--output_path", type=str, default="3dgs_pc.ply", help="Path to output file (must be ply file)")
    parser.add_argument("--transform_path", default=None, type=str, help="Path to COLMAP or Transform file used for loading in camera positions for rendering")
    parser.add_argument("--mask_path", default=None, type=str, help="Path to directory containing associated masks for image transforms")
    parser.add_argument("--renderer_type", type=str, default="cuda", help="The type of renderer to use for determining point colours ('cuda' or 'python')")
    parser.add_argument("--num_points", type=int, default=10000000, help="Total number of points to generate for the pointcloud")
    parser.add_argument("--exact_num_points", action="store_true", help="Match num_points more closely (slower)")
    parser.add_argument("--no_prioritise_visible_gaussians", action="store_true", help="Do not give more points to Gaussians that contribute most")
    parser.add_argument("--visibility_threshold", type=float, default=0.05, help="Minimum contribution each Gaussian must have to be included")
    parser.add_argument("--surface_distance_std", type=float, default=None, help="Cull Gaussians further than X standard deviations from the scene surfaces")
    parser.add_argument("--clean_pointcloud", action="store_true", help="Remove statistical outliers after generation (on the GPU)")
    parser.add_argument("--generate_mesh", action="store_true", help="Also generate a mesh (requires Open3D)")
    parser.add_argument("--poisson_depth", default=10, type=int, help="Depth of the poisson surface reconstruction")
    parser.add_argument("--laplacian_iterations", default=10, type=int, help="Iterations of laplacian mesh smoothing")
    parser.add_argument("--mesh_output_path", type=str, default="3dgs_mesh.ply", help="Path to mesh output file (must be ply file)")
    parser.add_argument("--camera_skip_rate", type=int, default=0, help="Number of cameras to skip for each rendered camera")
    parser.add_argument("--no_render_colours", action="store_true", help="Skip rendering colours")
    parser.add_argument("--colour_quality", type=str, default="high", help="tiny, low, medium, high, ultra or original")
    parser.add_argument("--bounding_box_min", nargs=3, help="Minimum position of gaussians to include")
    parser.add_argument("--bounding_box_max", nargs=3, help="Maximum position of gaussians to include")
    parser.add_argument("--mahalanobis_distance_std", type=float, default=2.0, help="Maximum distance each point can be from the centre of its gaussian")
    parser.add_argument("--no_calculate_normals", action="store_true", help="Do not calculate normals for the points")
    parser.add_argument("--min_opacity", type=float, default=0.0, help="Minimum opacity for gaussians to be included (0-1)")
    parser.add_argument("--cull_gaussian_sizes", type=float, default=0.0, help="Percentage of gaussians to remove from largest to smallest")
    parser.add_argument("--max_sh_degree", type=int, default=3, help="Spherical-harmonics degree of the loaded point cloud")
    parser.add_argument("--quiet", action="store_true", help="Suppress output")

    args = parser.parse_args(argv)

    if args.min_opacity < 0 or args.min_opacity > 1:
        raise AttributeError("Minumum opacity must be between 0 and 1")
    if args.mahalanobis_distance_std <= 0:
        raise AttributeError("Std distance must be greater than 0")
    if args.num_points <= 0:
        raise AttributeError("Number of points must be greater than 0")
    for name in ("bounding_box_min", "bounding_box_max"):
        v = getattr(args, name)
        if v is not None:
            try:
                v = [float(x) for x in v]
            except ValueError:
                raise AttributeError(f"{name.replace('_', ' ').title()} must contain float values")
            if len(v) != 3:
                raise AttributeError(f"{name.replace('_', ' ').title()} must have exactly 3 values")
            setattr(args, name, v)
    if args.colour_quality.lower() not in COLOR_QUALITY_OPTIONS.keys():
        raise AttributeError(f"Colour quality must be in the following options {COLOR_QUALITY_OPTIONS.keys()}")
    if args.max_sh_degree < 0:
        raise AttributeError("The number of spherical harmonics must be larger than 0")
    if args.camera_skip_rate < 0:
        raise AttributeError("The camera skip rate must be larger than 0")
    if args.generate_mesh and args.no_calculate_normals:
        raise AttributeError("Normals are required for accurate meshing")
    if args.generate_mesh and args.no_render_colours:
        raise AttributeError("Colours are required for meshing")
    if args.generate_mesh and args.transform_path is None:
        raise AttributeError("Transforms are required for meshing")
    if not args.no_render_colours and args.transform_path is None:
        raise AttributeError("Transforms are required for rendering accurate point colours, set --no_render_colours to True to render with no colour")
    if args.visibility_threshold < 0.0 or args.visibility_threshold > 1.0:
        raise AttributeError("Visible Gaussian Threshold must be between 0 and 1")
    if args.surface_distance_std is not None and args.surface_distance_std <= 0.0:
        raise AttributeError("Surface std must be large than 0")
    if args.mask_path is not None and args.transform_path is None:
        raise AttributeError("Cannot use masks when no transforms have been provided")
    if args.renderer_type != "cuda" and args.surface_distance_std is not None:
        raise AttributeError("Surface distance calculations only supported in CUDA renderer")
    if args.generate_mesh:
        # Open3D meshing is outside this build (SURVEY.md §2 row 15): fail before any loading / rendering
        try:
            import open3d  # noqa: F401
        except ImportError:
            raise AttributeError("--generate_mesh needs Open3D, which is not installed")
        raise AttributeError("--generate_mesh (Open3D meshing) is not part of this build")

    return args


def main(argv=None):
    args = config_parser(argv)

    if not torch.cuda.is_available():
        raise capi.G2pcError("a CUDA device is required (the g2pc kernels have no CPU fallback)")

    pointcloud_settings = GaussPointCloudSettings(
        renderer_type=args.renderer_type,
        num_points=args.num_points,
        prioritise_visible_gaussians=not args.no_prioritise_visible_gaussians,
        mahalanobis_distance_std=args.mahalanobis_distance_std,
        camera_skip_rate=args.camera_skip_rate,
        render_colours=not args.no_render_colours,
        min_opacity=args.min_opacity,
        bounding_box_min=args.bounding_box_min,
        bounding_box_max=args.bounding_box_max,
        calculate_normals=not args.no_calculate_normals,
        cull_large_percentage=args.cull_gaussian_sizes,
        colour_resolution=COLOR_QUALITY_OPTIONS[args.colour_quality.lower()],
        max_sh_degree=args.max_sh_degree,
        exact_num_points=args.exact_num_points,
        generate_mesh=args.generate_mesh,
        visibility_threshold=args.visibility_threshold,
        surface_distance_std=args.surface_distance_std,
        quiet=args.quiet,
        remove_unrendered_gaussians=True if args.visibility_threshold > 0 else False,
        device="cuda:0",
    )

    total_point_cloud, surface_point_cloud = convert_3dgs_to_pc(args.input_path, args.transform_path, args.mask_path,
                                                                pointcloud_settings)

    if args.clean_pointcloud:
        if not args.quiet:
            print("Cleaning Point Cloud")
            print()
        from mesh_handler import clean_point_cloud
        pts, cols, nrm = clean_point_cloud(total_point_cloud.points, total_point_cloud.colours,
                                           total_point_cloud.normals, device=pointcloud_settings.device)
        total_point_cloud = PointCloudData(points=pts, colours=cols, normals=nrm)

    if not args.quiet:
        print("Saving Final Point Cloud")

    from gauss_dataloader import save_xyz_to_ply
    save_xyz_to_ply(total_point_cloud.points, args.output_path, rgb_colors=total_point_cloud.colours,
                    normals_points=total_point_cloud.normals, chunk_size=10**6, quiet=args.quiet)

    if pointcloud_settings.generate_mesh:
        from mesh_handler import generate_mesh
        generate_mesh(surface_point_cloud.points, surface_point_cloud.colours, surface_point_cloud.normals,
                      args.mesh_output_path, depth=args.poisson_depth, laplacian_iters=args.laplacian_iterations)


if __name__ == "__main__":
    main()
