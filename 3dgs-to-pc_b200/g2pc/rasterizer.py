"""renderer_type="cuda": drop-in for the reference's CUDA rasterizer package `gaussian_pointcloud_rasterization`.

Reference call surface restated here (same names, argument order, defaults, return arity):
    GaussianRasterizationSettings     gaussian_pointcloud_rasterization/__init__.py:21-35
    GaussianRasterizer                :37-220   (constructor :38-76, forward :90-140, getters :160-220)
    _C.rasterize_gaussians            ext.cpp:15-17 / rasterize_points.cu:36-145  (22 arguments -> 11-tuple)
The work is done by the sm_100a kernels of csrc/s7_tiles.cu + the shared depth sort / multisplit (csrc/s4_tree.cu) behind
the C ABI (include/g2pc.h, g2pc_tiles_*).  Differences that are deliberate and documented:
  * results are deterministic (the reference's max-contribution / surface-distance updates race, SURVEY.md §2.1);
  * one camera costs no host synchronisation (g2pc/frames.py) — the reference runs with debug=True, i.e. a
    cudaDeviceSynchronize after every stage, plus a blocking D2H of the instance count;
  * `shs` may be given channel-major (N,3,K) as the loader yields it (gauss_dataloader.py:42-44); the reference hands that
    tensor to a kernel that reads it coefficient-major (forward.cu:31) — its SH path is unfinished (SURVEY.md §2 row 10).
"""
import ctypes
import math
from typing import NamedTuple

import torch

from . import capi
from .frames import FrameQueue

FLT_MAX_BITS = 0x7F7FFFFF
TILE = 16


class GaussianRasterizationSettings(NamedTuple):
    image_height: int
    image_width: int
    tanfovx: float
    tanfovy: float
    bg: torch.Tensor
    scale_modifier: float
    viewmatrix: torch.Tensor
    projmatrix: torch.Tensor
    sh_degree: int
    campos: torch.Tensor
    mask: torch.Tensor
    prefiltered: bool
    debug: bool
    antialiasing: bool


def _host_list(t, n):
    if isinstance(t, (list, tuple)):
        v = [float(x) for x in t]
    else:
        v = t.detach().to("cpu", torch.float32).reshape(-1).tolist()
    if len(v) != n:
        raise ValueError(f"expected {n} values, got {len(v)}")
    return v


def _raster_struct(rs):
    c = capi.Raster()
    V = getattr(rs, "_viewmatrix_host", None) or _host_list(rs.viewmatrix, 16)
    P = getattr(rs, "_projmatrix_host", None) or _host_list(rs.projmatrix, 16)
    pos = getattr(rs, "_campos_host", None) or _host_list(rs.campos, 3)
    for i in range(16):
        c.viewmatrix[i] = V[i]
        c.projmatrix[i] = P[i]
    for i in range(3):
        c.campos[i] = pos[i]
    c.tan_fovx, c.tan_fovy = float(rs.tanfovx), float(rs.tanfovy)
    c.width, c.height = int(rs.image_width), int(rs.image_height)
    return c


def _cov6_to_full(cov6):
    """(P,6) [00,01,02,11,12,22] (gauss_render.py:195-204) -> (P,3,3)."""
    c = cov6.to(torch.float32)
    return torch.stack([c[:, 0], c[:, 1], c[:, 2], c[:, 1], c[:, 3], c[:, 4], c[:, 2], c[:, 4], c[:, 5]], 1).reshape(-1, 3, 3)


def _cov_from_scale_rot(scales, rotations, mod):
    """computeCov3D (forward.cu:116-150): Sigma = (S R)^T (S R), S = mod * diag(scale), q = (r,x,y,z) not normalised."""
    q = rotations.to(torch.float32)
    r, x, y, z = q[:, 0], q[:, 1], q[:, 2], q[:, 3]
    R = torch.stack([1 - 2 * (y * y + z * z), 2 * (x * y - r * z), 2 * (x * z + r * y),
                     2 * (x * y + r * z), 1 - 2 * (x * x + z * z), 2 * (y * z - r * x),
                     2 * (x * z - r * y), 2 * (y * z + r * x), 1 - 2 * (x * x + y * y)], 1).reshape(-1, 3, 3)
    L = R * (mod * scales.to(torch.float32))[:, None, :]
    return L @ L.transpose(1, 2)


class GaussianRasterizer(FrameQueue):
    """Holds the per-Gaussian accumulators and renders one camera per forward() call
    (gaussian_pointcloud_rasterization/__init__.py:37-220)."""

    def __init__(self, means3D, means2D, opacities, shs=None, colors_precomp=None, scales=None, rotations=None,
                 cov3D_precomp=None, visible_gaussian_threshold=0.0, surface_distance_std=None,
                 calculate_surface_distance=False, sh_layout=0):
        if (shs is None and colors_precomp is None) or (shs is not None and colors_precomp is not None):
            raise Exception('Please provide excatly one of either SHs or precomputed colors!')
        if ((scales is None or rotations is None) and cov3D_precomp is None) or \
                ((scales is not None or rotations is not None) and cov3D_precomp is not None):
            raise Exception('Please provide exactly one of either scale/rotation pair or precomputed 3D covariance!')
        capi.require_cuda(means3D, opacities, shs, colors_precomp, scales, rotations, cov3D_precomp)
        self.lib = capi.load()
        self.means3D = means3D.to(torch.float32).contiguous()
        self.means2D = means2D
        self.opacities = opacities
        self.shs = shs if shs is not None else torch.Tensor([])
        self.colors_precomp = colors_precomp if colors_precomp is not None else torch.Tensor([])
        self.scales = scales if scales is not None else torch.Tensor([])
        self.rotations = rotations if rotations is not None else torch.Tensor([])
        self.cov3D_precomp = cov3D_precomp if cov3D_precomp is not None else torch.Tensor([])
        self.device = self.means3D.device
        dev = self.device
        n = self.means3D.shape[0]
        self._n = n

        self.gaussian_max_contribution = torch.zeros(n, device=dev, dtype=torch.float)
        self.gaussian_min_surface_distance = torch.full((n,), torch.finfo(torch.float).max, device=dev, dtype=torch.float)
        self.gaussian_total_contribution = torch.zeros(n, device=dev, dtype=torch.float)
        self.gaussian_colours = torch.zeros((n, 3), device=dev, dtype=torch.float)
        self.visible_gaussian_threshold = visible_gaussian_threshold
        self.surface_distance_std = surface_distance_std
        self.calculate_surface_distance = calculate_surface_distance
        self.first_frame = None

        # ---- device-resident inputs in the kernels' layout -------------------------------------------------------------
        self._scale_modifier = None
        self._geom = torch.empty((max(n, 1), 12), dtype=torch.float32, device=dev)
        self._packed = False
        self._colour_f32 = colors_precomp.to(torch.float32).contiguous() if colors_precomp is not None else None
        self._shs_f32 = None
        self._sh_layout = int(sh_layout)
        if shs is not None:
            self._shs_f32 = shs.to(torch.float32).contiguous()
            self._sh_stride = int(self._shs_f32.shape[2] if self._sh_layout == 0 else self._shs_f32.shape[1])
        self._init_frames(n)
        m = max(n, 1)
        for sl in self._slots:
            sl["radii"] = torch.zeros((m,), dtype=torch.int32, device=dev)
        self._cam_dist = None
        if calculate_surface_distance:
            self._cam_dist = torch.empty((m,), dtype=torch.int32, device=dev)
            capi.call("g2pc_fill_u32", capi.ptr(self._cam_dist), FLT_MAX_BITS, m, capi.stream_ptr(dev))

    # ---- nn.Module-like call surface -----------------------------------------------------------------------------------
    def __call__(self, raster_settings, **kw):
        return self.forward(raster_settings, **kw)

    def _pack(self, scale_modifier):
        if self._packed and self._scale_modifier == scale_modifier:
            return
        if self.cov3D_precomp.numel():
            cov = _cov6_to_full(self.cov3D_precomp) if self.cov3D_precomp.dim() == 2 else self.cov3D_precomp.to(torch.float32)
        else:
            cov = _cov_from_scale_rot(self.scales, self.rotations, float(scale_modifier))
        op = self.opacities.to(torch.float32).reshape(-1).contiguous()
        capi.call("g2pc_pack_geometry", capi.ptr(self.means3D), capi.ptr(cov.contiguous()), capi.ptr(op), self._n,
                  capi.ptr(self._geom), capi.stream_ptr(self.device))
        self._packed, self._scale_modifier = True, scale_modifier

    def _res_tables(self, W, H):
        t = self._tables.get((W, H))
        if t is None:
            dev = self.device
            # the depth-ordered lists are built per super-tile of 2x2 tiles (csrc/s7_tiles.cu)
            gx, gy = ((W + TILE - 1) // TILE + 1) // 2, ((H + TILE - 1) // TILE + 1) // 2
            ntiles = gx * gy
            chunk = int(self.lib.g2pc_multisplit_chunk(ntiles))
            if chunk <= 0:
                raise capi.G2pcError(f"{ntiles} tiles: image too large for the multisplit tables")
            t = dict(gx=gx, gy=gy, ntiles=ntiles, rows=int(self.lib.g2pc_multisplit_rows(self._n, ntiles)),
                     slots=[dict(node_cnt=torch.zeros((ntiles,), dtype=torch.int32, device=dev),
                                 leaves=torch.zeros((ntiles, capi.LEAF_WORDS), dtype=torch.int32, device=dev),
                                 leaf_order=torch.zeros((ntiles,), dtype=torch.int32, device=dev))
                            for _ in range(self.num_slots)],
                     colour=torch.zeros((3, H, W), dtype=torch.float32, device=dev),
                     depth=torch.zeros((1, H, W), dtype=torch.float32, device=dev),
                     invdepth=torch.zeros((1, H, W), dtype=torch.float32, device=dev))
            self._tables[(W, H)] = t
        return t

    def _mask_of(self, rs, W, H):
        mask = rs.mask
        if mask is None:
            return None
        if not mask.is_cuda:
            raise capi.G2pcError("mask must be a CUDA tensor")
        if mask.numel() != W * H:
            raise capi.G2pcError("mask must have image_height * image_width entries")
        return mask.to(torch.int32).contiguous()

    def _ensure_buffers(self, rs, slot):
        self._pack(float(rs.scale_modifier))
        t = self._res_tables(int(rs.image_width), int(rs.image_height))
        self._grow_lists(self._slots[slot], t["ntiles"], t["rows"])
        # (kept per slot: the tensor must outlive the frame's kernels, the slot is reused only after they have run)
        self._slots[slot]["mask"] = self._mask_of(rs, int(rs.image_width), int(rs.image_height))

    def _enqueue_front(self, rs, frame, slot):
        st = capi.stream_ptr(self.device)
        W, H = int(rs.image_width), int(rs.image_height)
        n = self._n
        t = self._res_tables(W, H)
        sl, ts = self._slots[slot], t["slots"][slot]
        c = _raster_struct(rs)
        deg = int(rs.sh_degree) if self._shs_f32 is not None else 0
        capi.call("g2pc_tiles_preprocess", capi.ptr(self._geom), capi.ptr(self._colour_f32), capi.ptr(self._shs_f32),
                  self._sh_stride if self._shs_f32 is not None else 0, min(deg, 3), self._sh_layout, n, ctypes.byref(c),
                  capi.ptr(sl["proj"]), capi.ptr(ts["node_cnt"]), capi.ptr(sl["depth_key"]), capi.ptr(sl["val"]),
                  capi.ptr(sl["radii"]), st)
        capi.call("g2pc_depth_sort", capi.ptr(sl["depth_key"]), capi.ptr(sl["val"]), n, capi.ptr(sl["val_sorted"]),
                  capi.ptr(sl["depth_ws"]), sl["depth_ws"].numel(), st)
        capi.call("g2pc_tiles_build", capi.ptr(ts["node_cnt"]), W, H, capi.ptr(ts["leaves"]), capi.ptr(ts["leaf_order"]),
                  t["ntiles"], self._inst_cap, sl["matrix"].numel(), t["rows"], frame, capi.ptr(sl["hdr"]),
                  capi.ptr(self._fail), capi.ptr(sl["work"]), st)
        capi.call("g2pc_multisplit_grid", capi.ptr(sl["val_sorted"]), n, t["gx"], t["gy"], capi.ptr(ts["leaves"]),
                  capi.ptr(sl["hdr"]), capi.ptr(self._fail), frame, t["ntiles"], capi.ptr(sl["matrix"]),
                  capi.ptr(sl["inst_gid"]), st)
        self._last, self._last_slot = t, slot
        return sl["hdr"]

    def _enqueue_back(self, rs, frame, camera_index, slot):
        st = capi.stream_ptr(self.device)
        W, H = int(rs.image_width), int(rs.image_height)
        n = self._n
        t = self._res_tables(W, H)
        sl, ts = self._slots[slot], t["slots"][slot]
        mask = sl.get("mask")
        # pixels that are masked out are never written by the blend (forward.cu:485): they keep the zeros of the fresh
        # output tensors the reference allocates per call (rasterize_points.cu:72-90)
        if mask is not None:
            t["colour"].zero_(); t["depth"].zero_(); t["invdepth"].zero_()
        bg = (ctypes.c_float * 3)(*(getattr(rs, "_bg_host", None) or _host_list(rs.bg, 3)))
        capi.call("g2pc_tiles_blend", capi.ptr(ts["leaves"]), capi.ptr(ts["leaf_order"]), capi.ptr(sl["hdr"]),
                  capi.ptr(self._fail), frame, capi.ptr(sl["inst_gid"]), capi.ptr(sl["proj"]), capi.ptr(self._cam_best),
                  capi.ptr(self._cam_dist), capi.ptr(mask), capi.ptr(t["colour"]), capi.ptr(t["depth"]),
                  capi.ptr(t["invdepth"]), W, H, bg, capi.ptr(sl["work"]), capi.ptr(self._stats), st)
        pc = getattr(self, "_per_camera", None) or (None, None, None)
        capi.call("g2pc_tiles_accumulate", capi.ptr(self._cam_best), capi.ptr(self._cam_dist), capi.ptr(t["colour"]), W, H,
                  n, capi.ptr(self.gaussian_max_contribution), capi.ptr(self.gaussian_total_contribution),
                  capi.ptr(self.gaussian_colours), capi.ptr(self.gaussian_min_surface_distance),
                  capi.ptr(self.first_frame), int(camera_index), capi.ptr(pc[0]), capi.ptr(pc[1]), capi.ptr(pc[2]), st)

    def forward(self, raster_settings, camera_index=None):
        """Render one camera and update the accumulators (__init__.py:90-140).
        Returns (colour (3,H,W), radii (P) int32, invdepths (1,H,W), depths (1,H,W))."""
        self._submit(raster_settings, camera_index)
        t, radii = self._last, self._slots[self._last_slot]["radii"]
        if self.async_mode:  # shared buffers: final after flush(), overwritten by the next camera(s)
            return t["colour"], radii, t["invdepth"], t["depth"]
        return t["colour"].clone(), radii.clone(), t["invdepth"].clone(), t["depth"].clone()

    # ---- FrameQueue hooks ---------------------------------------------------------------------------------------------
    def _confirm(self, h):
        self.last_stats = dict(num_tiles=h[capi.HDR_NUM_LEAVES], frame=h[capi.HDR_FRAME],
                               total_instances=h[capi.HDR_TOTAL_INST] + (h[capi.HDR_TOTAL_INST_HI] << 32))

    def _fix(self, h):
        if h[capi.HDR_CAP_OVERFLOW]:
            self._grow_inst_cap(h)
        else:
            raise capi.G2pcError("failed frame header without a recoverable cause")

    # ---- accumulator updates kept for API parity (the kernels fuse them) -------------------------------------------------
    def update_max_contributions(self, new_gauss_contributions, new_gauss_colours):
        self.flush()
        upd = new_gauss_contributions > self.gaussian_max_contribution
        self.gaussian_max_contribution[upd] = new_gauss_contributions[upd]
        self.gaussian_colours[upd] = new_gauss_colours[upd]
        self.gaussian_total_contribution += new_gauss_contributions

    def update_min_surface_distances(self, new_gauss_surface_distances):
        self.flush()
        upd = new_gauss_surface_distances < self.gaussian_min_surface_distance
        self.gaussian_min_surface_distance[upd] = new_gauss_surface_distances[upd]

    # ---- getters (__init__.py:160-220) ------------------------------------------------------------------------------------
    def get_gaussian_colours(self):
        self.flush()
        return self.gaussian_colours * 255

    def get_max_gaussian_contributions(self):
        self.flush()
        return self.gaussian_max_contribution

    def get_total_gaussian_contributions(self):
        self.flush()
        return self.gaussian_total_contribution

    def get_gaussians_above_contribution_threshold(self, contribution_threshold):
        return self.get_max_gaussian_contributions() > contribution_threshold

    def get_gaussians_above_total_contribution_threshold(self, contribution_threshold):
        return self.get_total_gaussian_contributions() > contribution_threshold

    def get_surface_gaussians_below_distance_threshold(self, surface_distance_threshold):
        """dist < mean(finite dists) * threshold — the reference takes element [1] (the MEAN) of torch.std_mean
        (__init__.py:190-201); kept."""
        if not self.calculate_surface_distance:
            raise Exception("Cannot determine Gaussian surface distance as this feature was not set at the start of rendering")
        self.flush()
        finite = self.gaussian_min_surface_distance < torch.finfo(torch.float).max
        mean_and_std = torch.std_mean(self.gaussian_min_surface_distance[finite])
        return self.gaussian_min_surface_distance < mean_and_std[1] * surface_distance_threshold

    def get_visible_gaussians(self):
        return self.get_gaussians_above_contribution_threshold(self.visible_gaussian_threshold)

    def get_gaussians_with_low_surface_distance(self):
        return self.get_surface_gaussians_below_distance_threshold(self.surface_distance_std)

    def get_predicted_surface_gaussians(self, predicted_surface_std=0.5):
        return self.get_surface_gaussians_below_distance_threshold(predicted_surface_std)


# ------------------------------------------------------------------------------------------------------------------------
def rasterize_gaussians(background, means3D, colors, opacity, scales, rotations, scale_modifier, cov3D_precomp,
                        viewmatrix, projmatrix, tan_fovx, tan_fovy, image_height, image_width, sh, degree, campos, mask,
                        prefiltered, antialiasing, calculate_surface_distance, debug):
    """The native op of the reference (`_C.rasterize_gaussians`, rasterize_points.cu:36-145): 22 arguments -> 11-tuple
    (num_rendered, color (3,H,W), depth (1,H,W), radii (P) i32, geomBuffer, binningBuffer, imgBuffer, invdepth (1,H,W),
    gauss_contributions (P), gauss_surface_distances (P), gauss_pixels (P) i32), one stateless call per camera.
    `sh` is (P,M,3) coefficient-major as the reference kernel reads it; the three byte buffers are returned empty (the
    scratch lives in caller-owned tensors behind the C ABI).  antialiasing must be False (the CLI never enables it)."""
    if antialiasing:
        raise NotImplementedError("antialiasing=True is not part of the path (camera_handler.py:107 always passes False)")
    has_sh = sh is not None and sh.numel() > 0
    R = GaussianRasterizer(means3D, None, opacity, shs=sh if has_sh else None,
                           colors_precomp=None if has_sh else colors,
                           scales=scales if (cov3D_precomp is None or cov3D_precomp.numel() == 0) else None,
                           rotations=rotations if (cov3D_precomp is None or cov3D_precomp.numel() == 0) else None,
                           cov3D_precomp=cov3D_precomp if (cov3D_precomp is not None and cov3D_precomp.numel()) else None,
                           calculate_surface_distance=bool(calculate_surface_distance), sh_layout=1)
    n = means3D.shape[0]
    dev = means3D.device
    rs = GaussianRasterizationSettings(image_height=int(image_height), image_width=int(image_width), tanfovx=tan_fovx,
                                       tanfovy=tan_fovy, bg=background, scale_modifier=scale_modifier,
                                       viewmatrix=viewmatrix, projmatrix=projmatrix, sh_degree=int(degree), campos=campos,
                                       mask=mask, prefiltered=prefiltered, debug=debug, antialiasing=False)
    contrib = torch.zeros((n,), dtype=torch.float32, device=dev)
    pixels = torch.zeros((n,), dtype=torch.int32, device=dev)
    surf = torch.full((n,), torch.finfo(torch.float).max, dtype=torch.float32, device=dev)
    R._per_camera = (contrib, pixels, surf if calculate_surface_distance else None)
    R._submit(rs)
    R.flush()
    t = R._last
    empty = torch.empty((0,), dtype=torch.uint8, device=dev)
    return (int(R.last_stats["total_instances"]), t["colour"], t["depth"], R._slots[R._last_slot]["radii"], empty,
            empty.clone(), empty.clone(), t["invdepth"], contrib, surf, pixels)


def mark_visible(means3D, viewmatrix, projmatrix):
    """`_C.mark_visible` (rasterizer_impl.cu:53-65,140-152): z_view > 0.2 — unused by the tool (the Python caller is
    commented out, __init__.py:79-88); kept for surface completeness as a one-line torch expression."""
    V = viewmatrix.to(torch.float32)
    z = means3D.to(torch.float32) @ V[:3, 2] + V[3, 2]
    return z > 0.2
