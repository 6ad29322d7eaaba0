"""Colour stage — drop-in for the reference's gauss_render.py.

Reference: /root/reference/gauss_render.py.  `get_renderer` (:467-493) is the plugin boundary: it returns a callable
`renderer(camera) -> (image, radii|None, invdepth|None, depth|None)` that, as a side effect, keeps for every Gaussian
the largest contribution alpha*T it made to any pixel of any camera and the blended colour of that pixel, plus the
getters used by the pipeline (gauss_to_pc.py:481-513).

`renderer_type="python"` reproduces GaussPythonRenderer (:210-465): quadtree tiles, every Gaussian of a tile blended
into every pixel of the tile — but as sm_100a kernels behind the C ABI (csrc/s3_preprocess.cu, s4_tree.cu,
s5_blend.cu), one camera = 8 asynchronous entry-point calls and no host wait.  The tile parameters the reference derives
from free GPU memory at call time (:440-444) are pinned (g2pc.config.MAX_TILE_SIZE / MAX_GAUSSIANS_PER_TILE).
"""
import ctypes
import math

import numpy as np
import torch

from g2pc import capi, config, quadtree
from g2pc.frames import FrameQueue

# SH constants kept for API parity with the reference module (gauss_render.py:9-38)
C0 = 0.28209479177387814
C1 = 0.4886025119029199

homogeneous = lambda points: torch.cat([points, torch.ones_like(points[..., :1])], dim=-1)


def strip_lowerdiag(L):
    idx = torch.tensor([0, 1, 2, 4, 5, 8], device=L.device)
    return L.reshape(L.shape[0], 9).index_select(1, idx).to(torch.float)


def strip_symmetric(sym):
    return strip_lowerdiag(sym)


class GaussPythonRenderer(FrameQueue):
    """B200 implementation of the reference's pure-torch tile renderer (same constructor arguments, attributes and
    getters as gauss_render.py:210-264).

    One camera ("frame") = 8 asynchronous entry-point calls and NO host wait: every size the later kernels need lives
    in a device-side frame header.  The host sizes its buffers optimistically; a frame that does not fit (or needs a
    deeper quadtree table) poisons the header on the device, every later kernel becomes a no-op, and the host — which
    reads the 64-byte headers back asynchronously — grows the buffers and replays from the failed frame, so the
    accumulators are updated in exactly the reference's camera order.  `async_mode = False` (default) confirms every
    frame before returning (the returned image is final); the pipeline driver sets `async_mode = True` and confirms
    lazily (getters call flush())."""

    def __init__(self, means3D, opacity, colour, cov3d, white_bkgd=True, visible_gaussian_threshold=0.0, shs=None,
                 sh_degree=None):
        capi.require_cuda(means3D, opacity, colour, cov3d, shs)
        self.lib = capi.load()
        self.white_bkgd = white_bkgd
        self.device = means3D.device
        n = means3D.shape[0]
        dev = self.device

        self.gaussian_max_contribution = torch.zeros(n, device=dev, dtype=torch.float32)
        self.gaussian_total_contribution = torch.zeros(n, device=dev, dtype=torch.float32)
        # blended colour of each Gaussian's best pixel (f32; the reference keeps f64)
        self.gaussian_colours = torch.zeros((n, 3), device=dev, dtype=torch.float32)
        self.visible_gaussian_threshold = visible_gaussian_threshold

        self.means3D = means3D.to(torch.float32).contiguous()
        self.opacity = opacity.to(torch.float32).reshape(-1).contiguous()
        self.cov3d = cov3d.to(torch.float32).contiguous()
        self.colour = colour
        self._colour_f32 = None if colour is None else colour.to(torch.float32).contiguous()
        self.shs = None
        self.sh_degree = 0
        if shs is not None:
            self.shs = shs.to(torch.float32).contiguous()
            ncoef = self.shs.shape[-1]
            deg = int(round(math.sqrt(ncoef))) - 1 if sh_degree is None else int(sh_degree)
            self.sh_degree = min(deg, 3)

        self.max_tile_size = config.MAX_TILE_SIZE
        self.max_gaussians_per_tile = config.MAX_GAUSSIANS_PER_TILE
        self.t_stop = config.BLEND_T_STOP
        self.compose_image = True
        self.async_mode = False
        self.first_frame = None  # optional (n) int32: index of the camera that raised each maximum (g2pc/dist.py)
        self._extra_levels = 0
        self._n = n
        st = capi.stream_ptr(dev)
        # packed geometry, read by every camera with 16-byte loads (once per renderer)
        self._geom = torch.empty((max(n, 1), 12), dtype=torch.float32, device=dev)
        capi.call("g2pc_pack_geometry", capi.ptr(self.means3D), capi.ptr(self.cov3d), capi.ptr(self.opacity), n,
                  capi.ptr(self._geom), st)
        self._init_frames(n)
        self._leaf_colour = None

    # ---- getters (gauss_render.py:237-264) -----------------------------------------------------------------
    def get_gaussian_colours(self):
        self.flush()
        return self.gaussian_colours * 255

    def get_gaussians_above_contribution_threshold(self, contribution_threshold):
        self.flush()
        return self.gaussian_max_contribution > contribution_threshold

    def get_visible_gaussians(self):
        return self.get_gaussians_above_contribution_threshold(self.visible_gaussian_threshold)

    def get_surface_gaussians(self):
        self.flush()
        return self.get_gaussians_above_contribution_threshold(torch.mean(self.gaussian_max_contribution))

    def get_total_gaussian_contributions(self):
        # the python back-end of the reference reports the MAX contribution here (gauss_render.py:261-264)
        self.flush()
        return self.gaussian_max_contribution

    # ---- per-resolution tables ---------------------------------------------------------------------------------
    def _get_tables(self, W, H):
        key = (W, H, self.max_tile_size, self.max_gaussians_per_tile, self._extra_levels)
        t = self._tables.get(key)
        if t is None:
            qt = quadtree.QuadtreeTables(W, H, self.max_tile_size, self.max_gaussians_per_tile,
                                         extra_levels=self._extra_levels)
            flat = np.concatenate(qt.flat()).astype(np.int32)
            dev = self.device
            mask = qt.candidate_level_mask()
            base = (mask & -mask).bit_length() - 1
            if base > 8:
                raise capi.G2pcError("image too large for the packed node range (first leaf level deeper than 8)")
            luts = qt.pixel_luts()
            if luts.shape[0] % 2:
                luts = np.concatenate([luts, np.zeros(1, np.uint16)])
            t = dict(qt=qt, tables=torch.from_numpy(flat).to(dev), level_mask=mask, base_level=base,
                     clean_mask=qt.clean_level_mask(),
                     luts=torch.from_numpy(luts.view(np.int16).copy()).to(dev),
                     slots=[dict(node_cnt=torch.zeros((qt.nodes_2d,), dtype=torch.int32, device=dev),
                                 node_state=torch.zeros((qt.nodes_2d,), dtype=torch.uint8, device=dev),
                                 node_leaf=torch.full((qt.nodes_2d,), -1, dtype=torch.int32, device=dev),
                                 leaves=None, leaf_order=None) for _ in range(self.num_slots)],
                     owner=torch.zeros((W * H,), dtype=torch.int32, device=dev),
                     image=torch.ones((H, W, 3), dtype=torch.float32, device=dev),
                     leaf_cap=0, pix_cap=int(1.25 * W * H) + 4096,
                     max_quads=int(((min(self.max_tile_size, W) + 3) // 4) * min(self.max_tile_size, H)))
            self._set_leaf_cap(t, min(qt.nodes_2d, 2 * (4 ** base)))
            self._tables[key] = t
        return t

    def _set_leaf_cap(self, t, cap):
        cap = int(min(max(cap, 1), t["qt"].nodes_2d))
        chunk = int(self.lib.g2pc_multisplit_chunk(cap))
        if chunk <= 0:
            raise capi.G2pcError(f"the quadtree has more than {cap} leaves: too many for the multisplit tables")
        t["leaf_cap"], t["chunk"] = cap, chunk
        t["chunks"] = int(self.lib.g2pc_multisplit_rows(self._n, cap))  # matrix rows: chunks + persistent CTAs
        for ts in t["slots"]:
            ts["leaves"] = torch.zeros((cap, capi.LEAF_WORDS), dtype=torch.int32, device=self.device)
            ts["leaf_order"] = torch.zeros((cap,), dtype=torch.int32, device=self.device)

    @staticmethod
    def _camera_struct(camera):
        c = capi.Camera()
        if hasattr(camera, "host"):  # matrices already on the host (camera_handler.Camera)
            get = camera.host
        else:
            get = lambda k: getattr(camera, k).detach().to("cpu", torch.float32)
        V = get("world_view_transform").contiguous().reshape(-1).tolist()
        P = get("projection_matrix").contiguous().reshape(-1).tolist()
        pos = get("camera_center").reshape(-1).tolist()
        for i in range(16):
            c.view[i] = V[i]
            c.proj[i] = P[i]
        for i in range(3):
            c.campos[i] = pos[i]
        c.tan_fovx = math.tan(camera.FoVx * 0.5)
        c.tan_fovy = math.tan(camera.FoVy * 0.5)
        c.focal_x = camera.focal_x
        c.focal_y = camera.focal_y
        c.width = camera.image_width
        c.height = camera.image_height
        return c

    def _ensure_buffers(self, camera, slot):
        """(Re)allocate the slot's frame buffers for the current capacities."""
        t = self._get_tables(int(camera.image_width), int(camera.image_height))
        self._grow_lists(self._slots[slot], t["leaf_cap"], t["chunks"])
        if self._leaf_colour is None or self._leaf_colour.numel() < 3 * t["pix_cap"]:
            self._leaf_colour = torch.empty((3 * t["pix_cap"],), dtype=torch.float32, device=self.device)

    def _enqueue_front(self, camera, frame, slot):
        """Projection, depth sort, tile table and per-tile lists of one camera, asynchronously on the current stream."""
        st = capi.stream_ptr(self.device)
        W, H = int(camera.image_width), int(camera.image_height)
        cam = self._camera_struct(camera)
        n = self._n
        t = self._get_tables(W, H)
        qt = t["qt"]
        sl, ts = self._slots[slot], t["slots"][slot]
        capi.call("g2pc_preprocess", capi.ptr(self._geom), capi.ptr(self._colour_f32) if self.shs is None else None,
                  capi.ptr(self.shs), int(self.shs.shape[-1]) if self.shs is not None else 0, self.sh_degree, n,
                  ctypes.byref(cam), capi.ptr(t["tables"]), capi.ptr(t["luts"]), qt.num_levels, t["level_mask"],
                  t["clean_mask"], capi.ptr(sl["proj"]),
                  capi.ptr(ts["node_cnt"]), capi.ptr(sl["depth_key"]), capi.ptr(sl["val"]), st)
        capi.call("g2pc_depth_sort", capi.ptr(sl["depth_key"]), capi.ptr(sl["val"]), n, capi.ptr(sl["val_sorted"]),
                  capi.ptr(sl["depth_ws"]), sl["depth_ws"].numel(), st)
        capi.call("g2pc_build_tree", capi.ptr(t["tables"]), qt.num_levels, qt.max_gaussians_per_tile,
                  capi.ptr(ts["node_cnt"]), capi.ptr(ts["node_state"]), capi.ptr(ts["node_leaf"]), capi.ptr(ts["leaves"]),
                  capi.ptr(ts["leaf_order"]), t["leaf_cap"], self._inst_cap, t["pix_cap"], sl["matrix"].numel(),
                  t["chunks"], frame, capi.ptr(sl["hdr"]), capi.ptr(self._fail), capi.ptr(sl["work"]), st)
        capi.call("g2pc_multisplit", capi.ptr(sl["val_sorted"]), n, capi.ptr(sl["proj"]), W, H, capi.ptr(t["tables"]),
                  qt.num_levels, t["level_mask"], t["clean_mask"], capi.ptr(ts["node_leaf"]), capi.ptr(ts["leaves"]),
                  capi.ptr(sl["hdr"]),
                  capi.ptr(self._fail), frame, t["leaf_cap"], capi.ptr(sl["matrix"]), capi.ptr(sl["inst_gid"]), st)
        self._last_tables, self._last_slot = t, slot
        return sl["hdr"]

    def _enqueue_back(self, camera, frame, camera_index, slot):
        """Blend + accumulator update (+ image) of one camera; runs after the previous camera's accumulator update."""
        st = capi.stream_ptr(self.device)
        W, H = int(camera.image_width), int(camera.image_height)
        n = self._n
        t = self._get_tables(W, H)
        sl, ts = self._slots[slot], t["slots"][slot]
        bg = 1.0 if self.white_bkgd else 0.0
        capi.call("g2pc_blend", capi.ptr(ts["leaves"]), capi.ptr(ts["leaf_order"]), capi.ptr(sl["hdr"]),
                  capi.ptr(self._fail), frame, t["max_quads"], capi.ptr(sl["inst_gid"]), capi.ptr(sl["proj"]),
                  capi.ptr(self._cam_best), capi.ptr(self.gaussian_max_contribution), capi.ptr(self._leaf_colour),
                  capi.ptr(t["owner"]), W, H, bg, float(self.t_stop), capi.ptr(sl["work"]), capi.ptr(self._stats), st)
        capi.call("g2pc_accumulate", capi.ptr(self._cam_best), capi.ptr(self._leaf_colour), n,
                  capi.ptr(self.gaussian_max_contribution), capi.ptr(self.gaussian_colours),
                  capi.ptr(self.first_frame), int(camera_index), st)
        if self.compose_image:
            capi.call("g2pc_compose_image", capi.ptr(t["owner"]), capi.ptr(self._leaf_colour), W, H, bg,
                      capi.ptr(t["image"]), st)
        else:
            t["owner"].zero_()

    def __call__(self, camera, camera_index=None, **kwargs):
        """Render one camera and update the per-Gaussian accumulators (gauss_render.py:404-465).
        Returns (image (H,W,3) f32 flipped left-right | None, None, None, None)."""
        self._submit(camera, camera_index)
        if not self.compose_image:
            return None, None, None, None
        t = self._last_tables  # (a replay may have switched to a deeper table set)
        # confirmed frames get their own tensor, like the reference; in async mode the shared buffer is handed out (it is
        # final once flush() has run and is overwritten by the next camera)
        return (t["image"] if self.async_mode else t["image"].clone()), None, None, None

    # ---- FrameQueue hooks ---------------------------------------------------------------------------------------------
    def _confirm(self, h):
        t = self._last_tables
        self.last_stats = dict(num_leaves=h[capi.HDR_NUM_LEAVES],
                               total_instances=h[capi.HDR_TOTAL_INST] + (h[capi.HDR_TOTAL_INST_HI] << 32),
                               total_leaf_pixels=h[capi.HDR_TOTAL_PIX], levels=t["qt"].num_levels, frame=h[capi.HDR_FRAME])

    def _fix(self, h):
        """A frame did not fit: grow what was too small (everything from that frame on was skipped on the device)."""
        t = self._last_tables
        W, H = t["qt"].width, t["qt"].height
        if h[capi.HDR_NEED_DEEPER]:
            # a tile at the deepest tabulated level holds more than max_gaussians_per_tile Gaussians: tabulate one more
            # level (rare; the reference keeps splitting in its host BFS)
            levels = t["qt"].num_levels
            self._extra_levels += 1
            if self._get_tables(W, H)["qt"].num_levels <= levels:
                raise capi.G2pcError(
                    f"a tile still holds more than max_gaussians_per_tile={self.max_gaussians_per_tile} Gaussians at "
                    f"quadtree level {levels - 1} (tiles of a few pixels): deeper than the tabulated levels")
        elif h[capi.HDR_LEAF_OVERFLOW]:
            if t["leaf_cap"] >= t["qt"].nodes_2d:
                raise capi.G2pcError("leaf table overflow")
            self._set_leaf_cap(t, max(2 * t["leaf_cap"], int(1.25 * h[capi.HDR_NUM_LEAVES])))
        elif h[capi.HDR_CAP_OVERFLOW]:
            self._grow_inst_cap(h)
            t["pix_cap"] = max(t["pix_cap"], int(1.25 * h[capi.HDR_TOTAL_PIX]) + 1024)
        else:
            raise capi.G2pcError("poisoned frame header without a cause")

    # ---- introspection for the parity tests ---------------------------------------------------------------------
    def debug_last_camera(self):
        """Per-Gaussian projection records and per-leaf sorted Gaussian ids of the most recent camera (host copies)."""
        self.flush()
        t, sl = self._last_tables, self._slots[self._last_slot]
        nl = self.last_stats["num_leaves"]
        leaves = t["slots"][self._last_slot]["leaves"][:nl].cpu().numpy()
        gids = sl["inst_gid"].cpu().numpy().astype(np.int64) if nl else np.zeros(0, np.int64)
        out = []
        for (r0, c0, w, h, beg, cnt, pix, node) in leaves:
            out.append((int(r0), int(c0), int(w), int(h), gids[beg:beg + cnt]))
        return sl["proj"].cpu().numpy(), out


def get_renderer(renderer_type: str, xyz, opacities, colours, covariances, shs=None, visible_gaussian_threshold=0.0,
                 surface_distance_std=None, calculate_surface_distance=False):
    """Factory with the reference's signature (gauss_render.py:467-493)."""
    if renderer_type == "python":
        return GaussPythonRenderer(xyz, opacities.type(torch.float), colours if shs is None else None, covariances,
                                   visible_gaussian_threshold=visible_gaussian_threshold, shs=shs)
    if renderer_type == "cuda":
        # the reference's CUDA back-end semantics (16x16 tiles, alpha / transmittance cut-offs, depth maps, surface
        # distances) on the sm_100a kernels of csrc/s7_tiles.cu — gauss_render.py:469-488
        from g2pc.rasterizer import GaussianRasterizer as GaussianPCRasterizer
        means2D = None  # (the reference allocates a zero tensor nobody reads, :476)
        common = dict(cov3D_precomp=covariances.to(torch.float), visible_gaussian_threshold=visible_gaussian_threshold,
                      surface_distance_std=surface_distance_std, calculate_surface_distance=calculate_surface_distance)
        if shs is None:
            return GaussianPCRasterizer(xyz.to(torch.float), means2D, opacities.type(torch.float),
                                        colors_precomp=colours.to(torch.float), **common)
        return GaussianPCRasterizer(xyz.to(torch.float), means2D, opacities.type(torch.float), shs=shs.to(torch.float),
                                    sh_layout=0, **common)
    raise Exception(f"Renderer of type {renderer_type} is not supported")
