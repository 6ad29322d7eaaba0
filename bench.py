#!/usr/bin/env python
"""bench.py — Mpoints/s (sample + colour) of the 3DGS-to-PC hot path on B200.

    python bench.py --gpus N --steps K --warmup W            (N > 1: launched by torch.distributed.run, one rank per GPU)
    python bench.py --impl reference ...                      (the reference's own code on the host cores)

One "step" = one pass of the hot path over the whole synthetic scene: covariance build (S1) -> colour stage over all
cameras (S3-S6, SH evaluated per camera) -> culls -> validate covariances -> magnitudes / points-per-Gaussian / bins ->
sampling + Mahalanobis cull (S2).  `value` is measured with the scene already resident in HBM; `e2e` goes through the
same public call (gauss_to_pc.convert_gaussians_to_pc) with pinned HOST buffers, host->device copies of the scene and
the device->host read of the point cloud inside the timed region.

Workloads (BASELINE.json configs): c3 = 3M Gaussians / 200 cameras / 10M points / 1280x720 / SH deg 3 / visibility
0.05 (headline, default); c2 = 1M / 50 / 10M / 720x405 / SH deg 2; c1 = 10k Gaussians, 100k points, no colour stage;
c4 = c3's scene, 50M points, surface_distance_std 2.0, exact_num_points (renderer_type cuda); c5 = 6M / 500 / 100M /
1920x1080.

Extra objects in the JSON line (all measured in this run, on this box):
  roofline        the dominant kernel of the step (by summed CUDA-event time) against the roof that bounds it
  rooflines       every hand-written kernel: algorithmic bytes / event time vs the measured HBM peak
  ref_cuda        the UNMODIFIED reference pipeline with its CUDA rasterizer (oracle/_ref, built for sm_100) on the same
                  workload and GPU — the ">= 10x" comparator of BASELINE.md §3.5
  c1              config C1 like for like: this build (GPU) next to the reference's own code on the host cores, in full
  cpu_baseline    the reference's own python path on a bounded sample of the workload (host cores)
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(ROOT, "3dgs-to-pc_b200")
for p in (ROOT, PKG):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np  # noqa: E402
import torch  # noqa: E402

WORKLOADS = {
    # name: n_gaussians, n_cameras, num_points, colour_quality width, sh_degree, render colours
    "c3": dict(n=3_000_000, cams=200, points=10_000_000, res=1280, sh=3, colours=True, seed=1234 + 2),
    "c2": dict(n=1_000_000, cams=50, points=10_000_000, res=720, sh=2, colours=True, seed=1234 + 1),
    "c1": dict(n=10_000, cams=0, points=100_000, res=None, sh=0, colours=False, seed=1234 + 0),
    "c4": dict(n=3_000_000, cams=200, points=50_000_000, res=1280, sh=3, colours=True, seed=1234 + 3,
               renderer="cuda", surface_distance_std=2.0, exact=True),
    "c5": dict(n=6_000_000, cams=500, points=100_000_000, res=1920, sh=3, colours=True, seed=1234 + 4),
    "tiny": dict(n=100_000, cams=4, points=400_000, res=720, sh=3, colours=True, seed=1234 + 9),
}
METRIC = "Mpoints/sec (sample+colour) at 3M Gaussians/200 cams, 1/2/4/8 B200 vs CPU ref"
UNIT = "Mpoints/s"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c3", choices=list(WORKLOADS))
    ap.add_argument("--renderer", default=None, choices=["python", "cuda"],
                    help="colour back-end semantics (default: the workload's, python unless stated)")
    ap.add_argument("--strict-blend", action="store_true", help="t_stop = FLT_MIN (strict-parity blend)")
    ap.add_argument("--blend-strips", action="store_true", help="row-strip pixel mapping in the blend (default: compact blocks)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-ref-cuda", action="store_true")
    ap.add_argument("--no-c1", action="store_true")
    ap.add_argument("--cpu-sample-gaussians", type=int, default=30000)
    ap.add_argument("--cpu-sample-cams", type=int, default=2)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the point cloud of the last timed step to DIR/<name>.npy (a fixed row sample if large)")
    return ap.parse_args()


DUMP_MAX_ROWS = 700_000  # rows kept per array: 3 arrays x 700 k rows x 3 x 8 B = 50.4 MB even if all are float64


def dump_outputs(pc, out_dir, suffix=""):
    """points / colours / normals of a PointCloudData as float32 (float64 kept) .npy files; more than DUMP_MAX_ROWS rows
    are reduced to the same seeded, sorted row sample in every array, so two builds that agree on the cloud agree here."""
    os.makedirs(out_dir, exist_ok=True)
    n = int(pc.points.shape[0])
    rows = None
    if n > DUMP_MAX_ROWS:
        g = torch.Generator().manual_seed(0)
        rows = torch.randperm(n, generator=g)[:DUMP_MAX_ROWS].sort().values
    for name in ("points", "colours", "normals"):
        t = getattr(pc, name)
        if t is None:
            continue
        if rows is not None:
            t = t[rows.to(t.device)]
        a = t.detach().cpu().numpy()
        np.save(os.path.join(out_dir, name + suffix + ".npy"), a if a.dtype == np.float64 else a.astype(np.float32))


def settings_for(wl, g2p, device, renderer=None):
    return g2p.GaussPointCloudSettings(
        renderer_type=renderer or wl.get("renderer", "python"), num_points=wl["points"],
        prioritise_visible_gaussians=True,
        mahalanobis_distance_std=2.0, camera_skip_rate=0, render_colours=wl["colours"], min_opacity=0.0,
        bounding_box_min=None, bounding_box_max=None, calculate_normals=True, cull_large_percentage=0.0,
        remove_unrendered_gaussians=True, colour_resolution=wl["res"], max_sh_degree=wl["sh"],
        exact_num_points=bool(wl.get("exact", False)),
        visibility_threshold=0.05, surface_distance_std=wl.get("surface_distance_std"), generate_mesh=False, quiet=True,
        device=device)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons, one sample every 200 ms.  ONE process per node (local rank 0) watches the
    GPUs of all local ranks; it is started before the warm-up so that its start-up (NVML initialisation, hundreds of ms
    of driver traffic) stays out of the timed region, and only the samples taken between mark_begin() and mark_end() are
    reported."""

    def __init__(self, indices=(0,), enabled=True):
        self.indices = list(indices)
        self.enabled = enabled
        self.rows = []
        self.proc = None
        self.t0 = self.t1 = None

    def __enter__(self):
        if not self.enabled:
            return self
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "--id=" + ",".join(str(i) for i in self.indices),
                                          f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
            # NVML start-up stalls every GPU of the node for tens of ms (seen as one 220 ms step among 150 ms ones at
            # N=2): wait for the first sample, i.e. until the tool is in its steady 200 ms polling loop
            t_end = time.time() + 10.0
            while not self.rows and time.time() < t_end and self.proc.poll() is None:
                time.sleep(0.02)
        except Exception:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [c.strip() for c in line.strip().split(",")]))

    def mark_begin(self):
        self.t0 = time.time()

    def mark_end(self):
        self.t1 = time.time()

    def __exit__(self, *exc):
        if self.proc is not None:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()
        return False

    def summary(self):
        rows = [r for t, r in self.rows if self.t0 is None or (self.t0 <= t <= (self.t1 or t) + 0.25)]
        sm = [float(r[0]) for r in rows if r and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) > 2 + i and r[2 + i].lower().startswith("active") for r in rows)]
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm), "gpus_watched": self.indices}


def _peaks():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        return {}


def _calibration():
    """Per-kernel constants taken from the committed ncu captures (profiles/): executed warp instructions per
    (warp, Gaussian) iteration of the blend kernel, dram bytes per launch of each kernel on C3."""
    try:
        return json.load(open(os.path.join(ROOT, "profiles", "r02_calibration.json")))
    except Exception:
        return {}


# --------------------------------------------------------------------------------------------------------------------
def run_ours(args):
    import torch.distributed as dist
    from g2pc import build, capi, config, sampler, synth
    build.build()
    capi.load()
    import gauss_to_pc as g2p

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    # torchrun pins OMP_NUM_THREADS=1: give every rank its share of the host cores for the (untimed) scene synthesis
    torch.set_num_threads(max(1, min(16, (os.cpu_count() or 1) // world)))
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local}"))
    torch.cuda.set_device(local)
    dev = f"cuda:{local}"
    wl = WORKLOADS[args.workload]
    if args.strict_blend:
        config.BLEND_T_STOP = 0.0
    if args.blend_strips:
        capi.load().g2pc_blend_set_compact(0)
    st = settings_for(wl, g2p, dev, args.renderer)

    sc = _scene_for(wl)
    cams, intr = synth.make_cameras(wl["cams"]) if wl["cams"] else ([], [])
    transforms = {f"cam{i:04d}": c for i, c in enumerate(cams)}
    intrinsics = {f"cam{i:04d}": k for i, k in enumerate(intr)}
    host = {k: v.pin_memory() for k, v in sc.items()}
    h2d_bytes = sum(v.numel() * v.element_size() for v in host.values()) + len(cams) * 64

    def upload():
        if world > 1:  # every rank uploads its row range, the shards are exchanged over NVLink (g2pc/dist.py)
            return gdist.upload_sharded(host, dev)
        return {k: v.to(dev, non_blocking=True) for k, v in host.items()}

    if world > 1:
        from g2pc import dist as gdist
        h2d_bytes = (h2d_bytes + world - 1) // world  # per rank, per step
        runner = lambda d: gdist.convert_gaussians_to_pc_sharded(d, transforms, intrinsics, st, render_shs=wl["sh"] > 0)
    else:
        def runner(d):
            pc, _ = g2p.convert_gaussians_to_pc(d["xyz"], d["scales"], d["rots"], d["colours"].clone(), d["opacities"],
                                                d["shs"], transforms if wl["colours"] else None, intrinsics, None, st,
                                                render_shs=wl["colours"] and wl["sh"] > 0)
            return pc

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    resident = upload()
    torch.cuda.synchronize()

    def step_resident():
        sampler.reset_call_counter(0)
        return runner(resident)

    out_host = {}

    def step_e2e():
        sampler.reset_call_counter(0)
        d = upload()
        pc = runner(d)
        for name, t in (("points", pc.points), ("colours", pc.colours), ("normals", pc.normals)):
            if t is None:
                continue
            buf = out_host.get(name)
            if buf is None or buf.shape[0] < t.shape[0]:
                buf = torch.empty((int(t.shape[0] * 1.05) + 16, 3), dtype=t.dtype).pin_memory()
                out_host[name] = buf
            buf[: t.shape[0]].copy_(t, non_blocking=True)
        torch.cuda.synchronize()
        return pc

    def timed(fn, steps):
        """CUDA-event timing of `steps` calls, barrier + synchronize on both sides, max over ranks."""
        barrier()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        pc = None
        dbg = os.environ.get("G2PC_BENCH_DEBUG")
        for _ in range(steps):
            t0 = time.perf_counter()
            pc = fn()
            if dbg:
                t1 = time.perf_counter()
                torch.cuda.synchronize()
                ph = getattr(sys.modules.get("g2pc.dist"), "LAST_PHASES", None) if world > 1 else None
                ms_ = torch.cuda.memory_stats(dev)
                print(f"[rank {rank}] {fn.__name__}: host {1e3 * (t1 - t0):.1f} ms, +drain {1e3 * (time.perf_counter() - t1):.1f} ms"
                      f" cudaMalloc {ms_.get('num_device_alloc')} cudaFree {ms_.get('num_device_free')}"
                      f" reserved {ms_.get('reserved_bytes.all.current', 0) >> 20} MiB"
                      + (f" phases {({k: round(v, 1) for k, v in ph.items()})}" if ph else ""), file=sys.stderr, flush=True)
        b.record()
        barrier()
        ms = torch.tensor([a.elapsed_time(b)], device=dev, dtype=torch.float64)
        npts = torch.tensor([pc.points.shape[0]], device=dev, dtype=torch.int64)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
            dist.all_reduce(npts, op=dist.ReduceOp.SUM)
        return float(ms.item()), int(npts.item()), pc

    # (torchrun: LOCAL_WORLD_SIZE ranks on this node; their GPUs are 0..LOCAL_WORLD_SIZE-1)
    local_world = int(os.environ.get("LOCAL_WORLD_SIZE", world))
    with ClockSampler(range(local_world), enabled=(local == 0)) as clk:
        # the warm-up has the shape of the timed loop (the previous step's cloud is still referenced while the next one is
        # computed): otherwise the second timed step is the first to need a second set of output buffers and pays three
        # cudaMalloc calls (seen as one 138 ms step among 59 ms ones on C2)
        pc_warm = None
        for _ in range(max(args.warmup, 3)):
            pc_warm = step_resident()
        del pc_warm
        capi.LAUNCHES = 0
        clk.mark_begin()
        ms, npts, pc = timed(step_resident, args.steps)
        clk.mark_end()
    launches = capi.LAUNCHES
    if args.dump_outputs:
        dump_outputs(pc, args.dump_outputs, f"_rank{rank}" if world > 1 else "")
    ms_step = ms / args.steps
    value = npts / (ms_step * 1e-3) / 1e6

    step_e2e()
    e2e_ms, e2e_pts, pc2 = timed(step_e2e, args.steps)
    e2e_step = e2e_ms / args.steps
    d2h_bytes = sum(t.numel() * t.element_size() for t in (pc2.points, pc2.colours, pc2.normals) if t is not None)

    # ---- per-kernel CUDA-event times: ONE extra step with every launch bracketed (kept out of the timed regions: the
    # ~5 k event records per step perturb the host-side enqueue) ------------------------------------------------------
    capi.TIMING = {}
    slots = config.FRAME_SLOTS
    config.FRAME_SLOTS = 1  # per-kernel times are only meaningful when the frames do not overlap
    step_resident()
    torch.cuda.synchronize()
    config.FRAME_SLOTS = slots
    timing = {k: [a.elapsed_time(b) for (a, b) in v] for k, v in capi.TIMING.items()}
    capi.TIMING = None
    rs = getattr(g2p, "LAST_RENDER_STATS", {}).get("stats")
    warp_gaussians = int(rs[0].item()) if rs is not None else 0  # the renderer of the profiled step only
    kernel_ms = {k.replace("g2pc_", ""): round(float(np.sum(v)), 3) for k, v in timing.items() if v}
    roof, roofs = rooflines(wl, timing, warp_gaussians, g2p, pc, world, clk.summary())
    rank_phases = None
    if world > 1:
        # per-rank timeline of one extra step (device-synchronised at every phase boundary: not a timed step)
        sampler.reset_call_counter(0)
        gdist.convert_gaussians_to_pc_sharded(resident, transforms, intrinsics, st, render_shs=wl["sh"] > 0,
                                              phase_timing=True)
        mine = {k: round(v, 2) for k, v in gdist.LAST_PHASES.items()}
        rank_phases = [None] * world
        dist.all_gather_object(rank_phases, mine)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    extras = {}
    if world == 1:
        if not args.no_ref_cuda and wl["colours"]:
            extras["ref_cuda"] = ref_cuda_leg(wl, e2e_pts / (e2e_step * 1e-3) / 1e6)
        if not args.no_c1:
            extras["c1"] = c1_leg(g2p, capi, sampler, dev)
        if not args.no_cpu_baseline:
            extras["cpu_baseline"] = cpu_baseline(wl, args.cpu_sample_gaussians, args.cpu_sample_cams)
    rtype = st.renderer_type
    line = {
        "metric": METRIC, "value": round(value, 3), "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": max(args.warmup, 3), "ms_per_step": round(ms_step, 3), "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"{args.workload}: {wl['n']} Gaussians, {wl['cams']} cameras, {wl['points']} points, "
                               f"width {wl['res']}, SH deg {wl['sh']}, visibility_threshold 0.05, renderer_type={rtype} "
                               "semantics", "points_out": npts,
                   "blend_t_stop": config.BLEND_T_STOP, "frame_slots": config.FRAME_SLOTS,
                   "l2": ("inputs larger than L2 (per-step working set >> 126 MB)" if h2d_bytes * world > 4 * 126e6 else
                          "working set below L2 and not flushed (non-headline workload)"),
                   "parallelism": "1 GPU" if world == 1 else f"cameras sharded x{world} (colour), Gaussians sharded x{world} (sampling)"},
        "e2e": {"value": round(e2e_pts / (e2e_step * 1e-3) / 1e6, 3), "unit": UNIT, "ms_per_step": round(e2e_step, 3),
                "h2d_bytes_per_step": h2d_bytes, "d2h_bytes_per_step": d2h_bytes},
        "gpu_launches": launches,
        "clocks": clk.summary(),
        "roofline": roof,
        "rooflines": roofs,
        "kernel_ms_per_step": kernel_ms,
        "frame_replays": getattr(g2p, "LAST_RENDER_STATS", {}).get("replays", 0),
    }
    if rank_phases is not None:
        line["rank_phases_ms"] = rank_phases
    line.update(extras)
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def rooflines(wl, timing, warp_gaussians, g2p, pc, world, clocks):
    """Roofline entries for every hand-written kernel from the per-launch CUDA-event times of the profiled step.
    HBM kernels: algorithmic bytes (SURVEY §8d / DESIGN.md §4) / time vs MEASURED_PEAKS.json hbm_gbs.
    Blend: not HBM and not tensor cores (no dense contraction) — executed warp instructions / time vs the issue roof
    (SMs x 4 schedulers x SM clock), with the instruction count per (warp, Gaussian) iteration taken from the committed
    ncu capture (profiles/r02_calibration.json)."""
    peaks = _peaks()
    cal = _calibration()
    peak_gbs = float(peaks.get("hbm_gbs", 6650.0))
    src = "measured" if peaks else "fallback"
    cams_rank = max(1, (wl["cams"] + world - 1) // world) if wl["cams"] else 0
    n = wl["n"]
    ncoef = (wl["sh"] + 1) ** 2
    n_active = int(getattr(g2p, "LAST_SAMPLE_STATS", {}).get("n_active", 0))
    p_rank = int(pc.points.shape[0])
    alg = {
        # per launch
        "g2pc_preprocess": n * (48 + (12 * ncoef if wl["sh"] > 0 else 12)) + n * (48 + 4 + 8),
        "g2pc_sample_emit": n_active * 44 + p_rank * 36,
        "g2pc_sample_count": n_active * (44 + 64),
        "g2pc_accumulate": n * 8,
        "g2pc_cov_build": n * (56 + 36),
    }
    out = []
    for name, v in timing.items():
        if not v or name not in alg:
            continue
        ms = float(np.mean(v))
        ach = alg[name] / (ms * 1e-3) / 1e9
        out.append({"kernel": name.replace("g2pc_", ""), "bound": "hbm", "achieved": round(ach, 1), "peak": peak_gbs,
                    "unit": "GB/s", "frac": round(ach / peak_gbs, 4), "alg_bytes_per_launch": int(alg[name]),
                    "avg_launch_ms": round(ms, 4), "launches": len(v), "peak_source": src,
                    "traffic": cal.get("dram_bytes_per_launch", {}).get(name.replace("g2pc_", ""))})
    blend = timing.get("g2pc_blend") or timing.get("g2pc_blend_tiles")
    dominant = None
    if blend:
        tot_ms = float(np.sum(blend))
        ipi = cal.get("blend_inst_per_warp_gaussian")
        sm_mhz = clocks.get("sm_mhz") or peaks.get("sm_max_mhz") or 1965.0
        sms = torch.cuda.get_device_properties(0).multi_processor_count
        peak_issue = sms * 4 * sm_mhz * 1e6 / 1e9  # G warp-instructions / s
        entry = {"kernel": "blend_kernel", "bound": "issue", "unit": "Gwarp-inst/s", "peak": round(peak_issue, 1),
                 "peak_source": "SMs x 4 schedulers x SM clock under load",
                 "pairs_per_s": round(warp_gaussians * 128 / (tot_ms * 1e-3), 1) if warp_gaussians else None,
                 "executed_pairs_per_step": warp_gaussians * 128, "ms_per_step": round(tot_ms, 3),
                 "inst_per_warp_gaussian": ipi, "traffic": cal.get("dram_bytes_per_launch", {}).get("blend")}
        if ipi and warp_gaussians:
            ach = warp_gaussians * ipi / (tot_ms * 1e-3) / 1e9
            entry.update(achieved=round(ach, 1), frac=round(ach / peak_issue, 4))
        else:
            entry.update(achieved=None, frac=None)
        out.append(entry)
    # dominant kernel = largest summed time among the entries
    tot = {e["kernel"]: (e.get("ms_per_step") or e["avg_launch_ms"] * e["launches"]) for e in out}
    if tot:
        k = max(tot, key=tot.get)
        dominant = next(e for e in out if e["kernel"] == k)
    return dominant, out


# --------------------------------------------------------------------------------------------------------------------
_SCENE_CACHE = {}


def _scene_for(wl):
    """The synthetic scene is a pure function of the workload: generate it once per process."""
    from g2pc import synth
    key = (wl["n"], wl["seed"], wl["sh"])
    if key not in _SCENE_CACHE:
        _SCENE_CACHE[key] = synth.make_scene(wl["n"], seed=wl["seed"], sh_degree=wl["sh"])
    return _SCENE_CACHE[key]


def host_threads():
    """Threads for the CPU arm: all cores up to 32 (beyond that the torch-CPU ops of this workload — thousands of
    small tile tensors — get slower, not faster: measured 240 s at 128 threads vs seconds at 8-32)."""
    return min(os.cpu_count() or 1, 32)


def ref_cuda_leg(wl, our_e2e):
    """The unmodified reference pipeline, renderer_type=cuda (its own CUDA rasterizer recompiled for sm_100), same
    workload, same GPU, one warm-up pass + one timed pass (BASELINE.md §3.5)."""
    try:
        from baseline import ref_run
        from g2pc import synth
        if not (ref_run.available() and ref_run.cuda_extension_available()):
            return {"unavailable": "reference not available (G2PC_REFERENCE_ROOT unset or oracle/build_ref.py not run)"}
        sc = _scene_for(wl)
        cams, intr = synth.make_cameras(wl["cams"])
        kw = dict(renderer_type="cuda", num_points=wl["points"], colour_resolution=wl["res"], max_sh_degree=wl["sh"],
                  exact_num_points=bool(wl.get("exact", False)), surface_distance_std=wl.get("surface_distance_std"))
        ref_run.run(sc, cams[:2], intr[:2], device="cuda:0", **dict(kw, num_points=min(wl["points"], 200_000)))  # warm-up
        torch.cuda.empty_cache()
        pc, dt = ref_run.run(sc, cams, intr, device="cuda:0", **kw)
        v = pc.points.shape[0] / dt / 1e6
        out = {"value": round(v, 4), "unit": UNIT, "seconds": round(dt, 2), "points_out": int(pc.points.shape[0]),
               "what": "unmodified reference convert_3dgs_to_pc, renderer_type=cuda (DC colours: the reference CLI never "
                       "passes SH to its renderer), debug=True syncs kept, file loaders replaced by in-memory tensors",
               "speedup_e2e": round(our_e2e / v, 2) if v > 0 else None}
        del pc
        torch.cuda.empty_cache()
        return out
    except Exception as e:  # the comparator must never take the bench line down
        return {"unavailable": f"{type(e).__name__}: {e}"[:300]}


def c1_leg(g2p, capi, sampler, dev):
    """BASELINE config C1 (10 k Gaussians, 100 k points, --no_render_colours) like for like: this build on the GPU (value
    = resident, e2e = pinned host in / host out) and the reference's own code on the host cores, both in full."""
    from g2pc import synth
    wl = WORKLOADS["c1"]
    st = settings_for(wl, g2p, dev)
    sc = _scene_for(wl)
    host = {k: v.pin_memory() for k, v in sc.items()}

    def run(d):
        sampler.reset_call_counter(0)
        pc, _ = g2p.convert_gaussians_to_pc(d["xyz"], d["scales"], d["rots"], d["colours"].clone(), d["opacities"],
                                            d["shs"], None, None, None, st)
        return pc

    res = {k: v.to(dev) for k, v in host.items()}
    for _ in range(3):
        run(res)
    torch.cuda.synchronize()
    K = 20
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(K):
        pc = run(res)
    b.record()
    torch.cuda.synchronize()
    ms = a.elapsed_time(b) / K
    t0 = time.perf_counter()
    for _ in range(K):
        d = {k: v.to(dev, non_blocking=True) for k, v in host.items()}
        pc = run(d)
        outs = [t.cpu() for t in (pc.points, pc.colours, pc.normals)]
    torch.cuda.synchronize()
    e2e_ms = (time.perf_counter() - t0) / K * 1e3
    npts = int(pc.points.shape[0])
    out = {"workload": "c1: 10000 Gaussians, 100000 points, --no_render_colours",
           "ours": {"value": round(npts / ms / 1e3, 3), "e2e": round(npts / e2e_ms / 1e3, 3), "unit": UNIT,
                    "ms_per_step": round(ms, 3), "e2e_ms_per_step": round(e2e_ms, 3), "points_out": npts}}
    out["reference_cpu"] = reference_c1()
    rv = out["reference_cpu"].get("value")
    if rv:
        out["speedup_e2e"] = round(out["ours"]["e2e"] / rv, 1)
    return out


def reference_c1(steps=5):
    """The reference's OWN code (unmodified, the checkout named by $G2PC_REFERENCE_ROOT) on C1 in full, CPU."""
    try:
        from baseline import ref_run
        if not ref_run.available():
            return {"unavailable": "reference sources not staged"}
        wl = WORKLOADS["c1"]
        threads = host_threads()
        torch.set_num_threads(threads)
        sc = _scene_for(wl)
        ref_run.run(sc, [], [], device="cpu", render_colours=False, num_points=wl["points"])  # warm-up (lazy imports)
        ts, npts = [], 0
        for _ in range(steps):
            pc, dt = ref_run.run(sc, [], [], device="cpu", render_colours=False, num_points=wl["points"])
            ts.append(dt)
            npts = int(pc.points.shape[0])
        dt = float(np.median(ts))
        return {"value": round(npts / dt / 1e6, 4), "unit": UNIT, "seconds": round(dt, 3), "points_out": npts,
                "cores": threads, "kind": "reference", "same_config": True}
    except Exception as e:
        return {"unavailable": f"{type(e).__name__}: {e}"[:300]}


def cpu_sample_run(wl, n_s, cams_s, threads):
    """The reference's python path (renderer_type=python + sampling) on a BOUNDED SAMPLE of the workload: the first n_s
    Gaussians, the first cams_s cameras at full resolution, num_points scaled by (n_s / n) * (cams_s / cams).  The
    reference's own code when it is staged (kind "reference"), else the oracle port (kind "port")."""
    from g2pc import synth
    torch.set_num_threads(threads)
    n_s = min(n_s, wl["n"])
    sc = {k: v[:n_s].clone() for k, v in _scene_for(wl).items()}
    cams, intr = synth.make_cameras(wl["cams"]) if wl["cams"] else ([], [])
    cams, intr = cams[:cams_s], intr[:cams_s]
    frac = (n_s / wl["n"]) * ((len(cams) / wl["cams"]) if wl["cams"] else 1.0)
    points = max(200, int(round(wl["points"] * frac)))
    desc = dict(gaussians=n_s, cameras=len(cams), points_requested=points)
    try:
        from baseline import ref_run
        if ref_run.available():
            pc, dt = ref_run.run(sc, cams, intr, device="cpu", renderer_type="python", num_points=points,
                                 render_colours=wl["colours"] and bool(cams), colour_resolution=wl["res"],
                                 max_sh_degree=wl["sh"])
            return int(pc.points.shape[0]), dt, desc, "reference"
    except Exception:
        pass
    from oracle import gaussians as og, render as orr, sampling as osamp
    t0 = time.perf_counter()
    cov = og.build_covariance(sc["scales"], sc["rots"])
    nrm = og.calculate_normals(sc["scales"], sc["rots"])
    contrib = sc["opacities"]
    colours = sc["colours"] * 255
    keep = torch.ones(n_s, dtype=torch.bool)
    if wl["colours"] and cams:
        O = orr.PythonRendererOracle(sc["xyz"], sc["opacities"], sc["colours"], cov, dense=True)
        for c2w, k in zip(cams, intr):
            O(orr.Camera(c2w, k, colour_resolution=wl["res"]))
        colours = torch.as_tensor(O.get_gaussian_colours())
        mc = torch.as_tensor(O.gaussian_max_contribution)
        keep = mc > 0.05
        contrib = mc
    if int(keep.sum()) < 2:
        keep[:] = True
    cov_k, vkeep = og.validate_covariances(cov[keep])
    mags = og.gaussian_magnitudes(cov_k, contrib[keep])
    o = osamp.generate_pointcloud(sc["xyz"][keep], cov_k, colours[keep], nrm[keep], mags, points, std=2.0,
                                  num_sample_attempts=5, seed=42)
    return o["points"].shape[0], time.perf_counter() - t0, desc, "port"


def _sample_text(desc, kind):
    who = "the reference's own code, unmodified" if kind == "reference" else "oracle port of the reference's python path"
    return (f"bounded sample, NOT the full workload: first {desc['gaussians']} Gaussians, first {desc['cameras']} cameras at "
            f"full resolution, {desc['points_requested']} points requested ({who}, renderer_type=python, torch-CPU)")


def cpu_baseline(wl, n_s, cams_s):
    threads = host_threads()
    npts, dt, desc, kind = cpu_sample_run(wl, n_s, cams_s, threads)
    return {"value": round(npts / dt / 1e6, 5), "unit": UNIT + " of the sample", "cores": threads, "kind": kind,
            "seconds": round(dt, 2), "sample": _sample_text(desc, kind)}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    wl = WORKLOADS[args.workload]
    threads = host_threads()
    for _ in range(min(args.warmup, 1)):
        cpu_sample_run(wl, max(2000, args.cpu_sample_gaussians // 10), 1, threads)
    tot_pts, tot_t = 0, 0.0
    desc, kind = None, "port"
    for _ in range(args.steps):
        npts, dt, desc, kind = cpu_sample_run(wl, args.cpu_sample_gaussians, args.cpu_sample_cams, threads)
        tot_pts += npts
        tot_t += dt
    value = tot_pts / tot_t / 1e6
    sample = _sample_text(desc, kind)
    line = {
        "impl": "reference", "metric": METRIC, "value": round(value, 5), "unit": UNIT,
        "n_gpus": int(os.environ.get("WORLD_SIZE", "1")), "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": round(tot_t / args.steps * 1e3, 1), "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"{args.workload} (bounded sample)", "sample": sample},
        "cpu_baseline": {"value": round(value, 5), "unit": UNIT, "cores": threads, "kind": kind, "sample": sample},
        "e2e": {"value": round(value, 5), "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
        # the one configuration the CPU can run in full, like for like with the GPU arm's `c1` object
        "c1_full": reference_c1(),
    }
    print(json.dumps(line))


if __name__ == "__main__":
    a = parse()
    if a.impl == "reference":
        run_reference(a)
    else:
        if not torch.cuda.is_available():
            raise SystemExit("bench.py needs a CUDA device (no CPU fallback); use --impl reference for the CPU arm")
        run_ours(a)
