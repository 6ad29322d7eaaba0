"""Host side of the device-driven frame pipeline shared by both colour back-ends (gauss_render.GaussPythonRenderer,
g2pc.rasterizer.GaussianRasterizer).

A "frame" is one camera.  All kernels of a frame are enqueued without waiting; the sizes later kernels need live in a
device-side header (include/g2pc.h, G2PC_HDR_*).  Frames alternate between two slots (scratch buffers + a CUDA stream
each): the front-end of frame f + 1 (projection, depth sort, tile table, multisplit) overlaps the blend of frame f, whose
tail would otherwise idle most SMs; the blend of frame f + 1 waits (event) for the accumulator update of frame f, so
the per-Gaussian accumulators see the cameras in exactly the reference's order (gauss_to_pc.py:437-454).

A frame that does not fit the host's buffers lowers the shared failure word on the device: every kernel of that and of
all later frames is a no-op, earlier frames still complete.  The host copies the 64-byte header of every frame to pinned
memory asynchronously and looks at it when the frame's end event has fired (or when a getter calls flush()): on failure it
grows what was too small, resets the word and replays the skipped frames in order.  No call ever waits for a count; the
reference synchronises the device several times per camera (rasterizer_impl.cu:289 blocking D2H, auxiliary.h:178-185
CHECK_CUDA after every stage).
"""
import torch

from . import capi, config


_HDR_POOLS = {}  # device -> free pinned frame headers (cudaHostAlloc is slow: never once per renderer)


class FrameQueue:
    """Mixin.  The owner provides: self.device, self.lib, self._ensure_buffers(camera, slot) (allocate / grow the slot's
    scratch on the current stream), self._enqueue_front(camera, frame, slot) -> device header tensor,
    self._enqueue_back(camera, frame, camera_index, slot), self._fix(header_list) and self._confirm(header_list).
    self._tables maps a resolution to its tables, each with a "slots" list of per-slot dicts holding "node_cnt"."""

    def _init_frames(self, n):
        self._frame = 0
        self._pending = []   # (frame, camera, camera_index, pinned header, end-of-frame event)
        self._hdr_pool = _HDR_POOLS.setdefault(str(self.device), [])  # pinned headers are shared by all renderers
        self.replays = 0
        self.async_mode = False
        self.num_slots = max(1, int(config.FRAME_SLOTS))
        self._streams = [torch.cuda.Stream(device=self.device) for _ in range(self.num_slots)]
        self._fail = torch.full((1,), -1, dtype=torch.int32, device=self.device)  # 0xFFFFFFFF: no frame has failed
        self._prev_done = None
        # per-frame scratch: one set per slot (frames alternate between the slots)
        dev = self.device
        m = max(n, 1)
        nbytes = self.lib.g2pc_depth_sort_workspace_bytes(m)
        self._slots = [dict(proj=torch.empty((m, 12), dtype=torch.float32, device=dev),
                            depth_key=torch.empty((m,), dtype=torch.int32, device=dev),
                            val=torch.empty((m,), dtype=torch.int64, device=dev),
                            val_sorted=torch.empty((m,), dtype=torch.int64, device=dev),
                            depth_ws=torch.empty((max(int(nbytes), 1),), dtype=torch.uint8, device=dev),
                            hdr=torch.zeros((capi.HDR_WORDS,), dtype=torch.int32, device=dev),
                            work=torch.zeros((capi.WORK_COUNTERS,), dtype=torch.int32, device=dev),
                            inst_gid=None, matrix=None) for _ in range(self.num_slots)]
        self._cam_best = torch.zeros((m,), dtype=torch.int64, device=dev)
        self._stats = torch.zeros((capi.STAT_WORDS,), dtype=torch.int64, device=dev)
        self._inst_cap = max(8 * n, 1 << 16)  # (Gaussian, list) instances; grown when a frame overflows
        self._tables = {}
        self._last_slot = 0
        self.last_stats = {}

    def _grow_lists(self, sl, lists, matrix_rows):
        """Grow the slot's list buffer (inst_gid) to _inst_cap instances in `lists` lists and its multisplit matrix to
        matrix_rows x lists."""
        need = self._inst_cap + 4 * lists + 64  # lists are padded to 16 bytes; slack for the last TMA unit
        if sl["inst_gid"] is None or sl["inst_gid"].numel() < need:
            sl["inst_gid"] = torch.empty((need,), dtype=torch.int32, device=self.device)
        mneed = matrix_rows * lists
        if sl["matrix"] is None or sl["matrix"].numel() < mneed:
            sl["matrix"] = torch.empty((max(mneed, 1),), dtype=torch.int32, device=self.device)

    def _grow_inst_cap(self, h):
        """The frame of header h had more (Gaussian, tile) instances than _inst_cap: grow it."""
        total = h[capi.HDR_TOTAL_INST] + (h[capi.HDR_TOTAL_INST_HI] << 32)
        if total > 0x7FFFFFFF:
            raise capi.G2pcError(f"{total} (Gaussian, tile) instances in one camera: more than 2^31 - 1")
        self._inst_cap = max(self._inst_cap, int(1.25 * total) + 1024)

    def _reset_counts(self):
        """Zero the per-slot tile counters (a failed frame left them half counted)."""
        for t in self._tables.values():
            for ts in t["slots"]:
                ts["node_cnt"].zero_()

    def executed_pairs(self):
        """(pixel, Gaussian) pairs the blend evaluated since construction: 32 threads x 4 pixels per warp and Gaussian
        (device counter)."""
        self.flush()
        return int(self._stats[capi.STAT_WARP_GAUSSIANS].item()) * 128

    def _launch(self, frame, camera, camera_index):
        slot = frame % self.num_slots
        st = self._streams[slot]
        # every buffer is allocated on the CALLER's stream (never inside the side-stream context): torch's caching
        # allocator keeps per-stream pools, and a block allocated under a pooled side stream cannot be reused by the next
        # renderer (different stream objects) — the allocator then falls back to cudaMalloc / cudaFree every step
        self._ensure_buffers(camera, slot)
        ready = torch.cuda.Event()
        ready.record(torch.cuda.current_stream(self.device))  # inputs prepared on the caller's stream
        st.wait_event(ready)
        with torch.cuda.stream(st):
            dev_hdr = self._enqueue_front(camera, frame, slot)
            hdr = self._hdr_pool.pop() if self._hdr_pool else torch.zeros((capi.HDR_WORDS,), dtype=torch.int32).pin_memory()
            hdr.copy_(dev_hdr, non_blocking=True)
            if self._prev_done is not None:
                st.wait_event(self._prev_done)  # the accumulators must have seen the previous camera
            self._enqueue_back(camera, frame, camera_index, slot)
            done = torch.cuda.Event()
            done.record(st)
        self._prev_done = done
        self._pending.append((frame, camera, camera_index, hdr, done))

    def _submit(self, camera, camera_index=None):
        frame = self._frame
        self._frame += 1
        camera_index = frame if camera_index is None else camera_index
        self._launch(frame, camera, camera_index)
        if not self.async_mode:
            self.flush()
        else:
            self._poll(block_if_more_than=8)

    def _poll(self, block_if_more_than=None):
        while self._pending:
            frame, camera, cidx, hdr, ev = self._pending[0]
            if not ev.query():
                if block_if_more_than is None or len(self._pending) <= block_if_more_than:
                    return
                ev.synchronize()
            h = hdr.tolist()
            if h[capi.HDR_POISON] and h[capi.HDR_POISON] - 1 <= frame:
                self._recover(h)
                continue
            self._confirm(h)
            self._hdr_pool.append(hdr)
            self._pending.pop(0)

    def flush(self):
        """Wait for every enqueued frame and replay the ones a failed frame skipped."""
        while self._pending:
            self._pending[-1][4].synchronize()
            self._poll(block_if_more_than=0)
        if self._prev_done is not None:
            torch.cuda.current_stream(self.device).wait_event(self._prev_done)

    def _recover(self, h):
        for st in self._streams:
            st.synchronize()
        failed = h[capi.HDR_POISON] - 1
        todo = [p for p in self._pending if p[0] >= failed]
        self._pending = [p for p in self._pending if p[0] < failed]
        self._fix(h)  # capacities only; the buffers are re-allocated by the next _launch, on the caller's stream
        self._fail.fill_(-1)
        self._reset_counts()
        torch.cuda.current_stream(self.device).synchronize()
        self.replays += 1
        for (frame, camera, cidx, hdr, ev) in todo:
            self._hdr_pool.append(hdr)
            self._launch(frame, camera, cidx)

    def __del__(self):
        try:
            for st in getattr(self, "_streams", []):
                st.synchronize()
        except Exception:
            pass
