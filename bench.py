#!/usr/bin/env python
"""bench.py -- BASELINE.json's metric on BASELINE.json's config.

  metric   Mpixel-sweeps/s (and ms/solve) of the reference's full fixed-schedule pyramid solve
  workload configs[2]: 3840x2160 synthetic image + ~10 % brush scribbles, 6 levels,
           1000/500/250/125/62/31 sweeps = 1968 sweeps = 507.1 M pixel-sweeps per solve
  step     one whole solve frame (main.cpp:232-295: annotation restriction, Dirichlet injection,
           per level edge-weight pass + sweeps + copy back, depth prolongation, 8-bit quantise)
  value    device-resident (annotations already in HBM), CUDA events, max over ranks
  e2e      the same frame through rtdd_frame_solve_host_annotation with HOST buffers: the annotation
           plane (1 B/px, main.cpp:160-170's format) uploaded from pinned memory and the 8-bit depth
           map delivered into pinned memory inside the timed region (the last sweep pass stores it
           there itself); e2e.three_plane_upload = rtdd_frame_solve_host with main.cpp's own
           scribble + 3-channel edited planes
  N > 1    batch data parallelism: every rank solves its own 4K image, no collective on the data
           path => weak scaling; plus, at every N, the records batch256_1080p (configs[3] as written)
           and strips16k (configs[4]: one 16384^2 image in row strips, strong scaling)

--impl reference runs the reference's OWN kernels (oracle/_ref/libref.so, compiled unmodified from
/root/reference/src/*.cu) through the reference's own functions on the same workload.  The
reference has no CPU implementation (SURVEY.md fact 8), so its own path IS a GPU path; the CPU
figure (`cpu_baseline`, kind "port") is the oracle's OpenMP restatement on the host cores.

--dump-outputs DIR (native path, rank 0) writes what the last timed step handed its caller, the frame's fp32 depth map and
its 8-bit depth map, as DIR/depth.npy and DIR/depth_u8.npy in float32.  The inputs are seeded, so two builds run with the
same arguments can be compared output for output.  Where both planes together exceed 64 MB (4K and up), both keep the same
fixed, seeded sample of pixels; DIR/pixel_index.npy (float64) holds their row-major indices.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

WORKLOADS = {"8k": (4320, 7680, 1004), "4k": (2160, 3840, 1003), "1080p": (1080, 1920, 1002), "720p": (720, 1280, 1001), "tiny": (203, 317, 77)}
# dram__bytes_read.sum + dram__bytes_write.sum of ONE level-0 launch (ncu --set full, profiles/r02_ncu_L0_cluster_T7_default.txt:
# 93.5 MB read + 37.9 MB written); workloads without a capture report null
NCU_TRAFFIC_BYTES_PER_LAUNCH = {"4k": 131.5e6}
BYTES_PER_PIXEL_SWEEP = 17.0     # SURVEY.md section 8(d): x_k 4 + x_{k-1} 4 + x_{k+1} 4 + 4 link indices 4 + mask 1
DUMP_BYTES = 64 * 10 ** 6


def dump_outputs(outdir, planes):
    """planes: [(name, 2-D array)] of one shape -> outdir/<name>.npy in float32, sampled as the module docstring says."""
    os.makedirs(outdir, exist_ok=True)
    n = planes[0][1].size
    if 4 * n * len(planes) > DUMP_BYTES:
        keep = (DUMP_BYTES - (1 << 16)) // (4 * len(planes) + 8)           # float32 per plane + one float64 index, headers aside
        idx = np.sort(np.random.default_rng(0).choice(n, keep, replace=False))
        np.save(os.path.join(outdir, "pixel_index.npy"), idx.astype(np.float64))
        planes = [(name, a.reshape(-1)[idx]) for name, a in planes]
    for name, a in planes:
        np.save(os.path.join(outdir, name + ".npy"), a.astype(np.float32))


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                          "-lms", "25"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons), "samples": len(sm)}


def bind_to_gpu_numa_node(local):
    """Best effort: run this rank (and first-touch its pinned buffers) on the CPUs of the NUMA node its GPU hangs off, so that
    eight ranks' host<->device copies do not all cross the same socket link.  Silently does nothing where sysfs says nothing."""
    try:
        props = torch.cuda.get_device_properties(local)
        bus = "%04x:%02x:%02x.0" % (props.pci_domain_id, props.pci_bus_id, props.pci_device_id)
        node = int(open("/sys/bus/pci/devices/%s/numa_node" % bus).read().strip())
        if node < 0:
            return None
        cpus = set()
        for part in open("/sys/devices/system/node/node%d/cpulist" % node).read().strip().split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
            return node
    except Exception:
        pass
    return None


def dist_setup(n_gpus):
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        bind_to_gpu_numa_node(local)
    if world > 1:
        import torch.distributed as dist
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        return dist, rank, world, local
    torch.cuda.set_device(0)
    return None, 0, 1, 0


def barrier(dist):
    if dist is not None:
        dist.barrier()
    torch.cuda.synchronize()


def max_over_ranks(dist, v):
    if dist is None:
        return v
    t = torch.tensor([v], dtype=torch.float64, device="cuda")
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def pyramid_levels(rows, cols):
    """ref: src/main.cpp:95"""
    import math
    return int(math.log2(max(min(cols, rows) // 45, 1))) + 1


def pixel_sweeps(rows, cols, levels, max_iterations=1000):
    """Level sizes (ref: src/main.cpp:103 floor), sweeps per level (ref: src/main.cpp:263) and their product -- plain
    arithmetic, shared by both arms (the reference arm must not import the product package)."""
    total, per = 0, []
    for l in range(levels):
        r, c = int(rows / 2.0 ** l), int(cols / 2.0 ** l)
        it = int(np.float32(max_iterations) / np.float32(2.0 ** ((levels - 1) - l)))
        per.append((r, c, it))
        total += r * c * it
    return total, per


def workload_string(rows, cols, seed, levels, per_level, total_ps):
    return ("configs[2]: %dx%d synthetic image (seed %d+rank) + ~10%% brush scribbles, full %d-level pyramid solve, "
            "reference schedule %s sweeps = %.1f M pixel-sweeps per solve; N>1 = configs[3] batch data parallelism "
            "(one image per rank, no collective)" % (cols, rows, seed, levels, "/".join(str(p[2]) for p in reversed(per_level)), total_ps / 1e6))


def cpu_baseline(rows, cols, levels, budget_s=12.0):
    """The oracle port (OpenMP) on the host cores: level-0 sweeps of the same workload, bounded."""
    from oracle import binding as ob
    synth = ob.pkg_file("synth")
    bgr, scribble, edited = synth.synth_case(rows, cols, 1003)
    gray = ob.bgr2gray(bgr)
    depth = np.full((rows, cols), 255.0, np.float32)
    depth = ob.convert_to_float(edited, depth, scribble)
    lut = ob.load_weights(0.4)
    try:
        ob.set_num_threads(len(os.sched_getaffinity(0)))       # torchrun exports OMP_NUM_THREADS=1: use every core we may run on
    except AttributeError:
        ob.set_num_threads(os.cpu_count() or 1)
    iters = pixel_sweeps(rows, cols, levels)[1][0][2]
    ob.solve_level(depth[:64], scribble[:64], gray[:64], 2, 0, levels - 1, lut)     # warm the OpenMP pool
    t0 = time.perf_counter()
    done = 0
    while True:
        ob.solve_level(depth, scribble, gray, iters, 0, levels - 1, lut)
        done += iters
        el = time.perf_counter() - t0
        if el > budget_s:
            break
    v = rows * cols * done / el / 1e6
    return {"value": v, "unit": "Mpixel-sweeps/s", "cores": ob.num_threads(), "kind": "port",
            "sample": "%dx%d level 0, %d Chebyshev-Jacobi sweeps incl. edge-weight pass, OpenMP static rows, %.1f s" % (cols, rows, done, el)}


def batch256_1080p(rtdd, dist, rank, world, stream_main):
    """BASELINE configs[3] as written (SURVEY.md 8d, config 4): 256 synthetic 1080p images, seeds 2000..2255, ~10 % scribbles,
    image i -> rank i mod N; every image is a full job through the public API from pinned HOST buffers -- BGR upload + gray
    pyramid (rtdd_frame_set_image), annotation upload + ingest + 5-level solve (rtdd_frame_solve_host_annotation) and the
    8-bit map back (rtdd_frame_read_depth_u8) -- with K independent contexts in flight per GPU (one stream each, one host
    thread).  Images are synthesised on the device beforehand (outside the timed region) and parked in pinned memory."""
    from realtimedepthdiffusion_b200 import synth_device
    rows, cols, total_images, K = 1080, 1920, 256, 8            # K: tools/tune_batch.py -- 0.89 / 0.79 / 0.70 / 0.66 / 0.67 ms per image at 3 / 4 / 6 / 8 / 12
    mine = list(range(rank, total_images, world))
    gen = rtdd.DepthDiffusion(rows, cols)
    gen.set_stream(stream_main)
    h_bgr, h_ann = [], []
    with torch.cuda.stream(stream_main):
        for i in mine:
            bgr, scribble, edited = synth_device.synth_case_device(rows, cols, 2000 + i, gen)
            hb = torch.empty((rows, cols, 3), dtype=torch.uint8).pin_memory()
            hb.view(rows, cols * 3).copy_(bgr)
            ha = torch.empty((rows, cols), dtype=torch.uint8).pin_memory()
            ha.copy_(synth_device.annotation_plane_device(scribble, edited))
            h_bgr.append(hb)
            h_ann.append(ha)
        torch.cuda.synchronize()
    levels = gen.levels
    gen.close()
    per_image_ps, _ = pixel_sweeps(rows, cols, levels)
    ctxs = []
    for k in range(K):
        c = rtdd.DepthDiffusion(rows, cols)
        st = torch.cuda.Stream()
        c.set_stream(st)
        if not os.environ.get("RTDD_BATCH_LATENCY_PLAN"):        # (the environment switch exists for the A/B in profiles/)
            c.set_tuning("plan_throughput", 1)                   # K images share the GPU: pass plans for least SM time, not least latency
        ctxs.append((c, st, torch.empty((rows, cols), dtype=torch.uint8).pin_memory()))
    for k, (c, st, ho) in enumerate(ctxs):                       # warm-up: graphs, allocations -- the same calls as the timed loop
        c.frame_set_image(h_bgr[k % len(mine)])
        c.frame_solve_host_annotation(h_ann[k % len(mine)], 1000, None)
        c.frame_read_depth_u8(ho, sync=True)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier(dist)
    ev0.record()
    for _, st, _ in ctxs:
        st.wait_event(ev0)
    launches0 = sum(c.launch_count for c, _, _ in ctxs)
    for j in range(len(mine)):
        c, st, ho = ctxs[j % K]
        c.frame_set_image(h_bgr[j], sync=False)
        c.frame_solve_host_annotation(h_ann[j], 1000, None)
        c.frame_read_depth_u8(ho, sync=False)
    for _, st, _ in ctxs:
        torch.cuda.current_stream().wait_stream(st)
    ev1.record()
    torch.cuda.synchronize()
    launches = sum(c.launch_count for c, _, _ in ctxs) - launches0
    ms = max_over_ranks(dist, ev0.elapsed_time(ev1))
    for c, _, _ in ctxs:
        c.close()
    return {"images": total_images, "images_per_gpu": len(mine), "contexts_in_flight_per_gpu": K, "ms_total": ms, "ms_per_image": ms / total_images,
            "value": per_image_ps * total_images / (ms * 1e-3) / 1e6, "unit": "Mpixel-sweeps/s", "gpu_launches_rank0": int(launches),
            "h2d_bytes_per_image": rows * cols * 4, "d2h_bytes_per_image": rows * cols,
            "note": "256 x (1920x1080, %d levels, %.1f M pixel-sweeps) from pinned host buffers through rtdd_frame_set_image + "
                    "rtdd_frame_solve_host_annotation + rtdd_frame_read_depth_u8; uploads, gray pyramid and downloads inside the timed region"
                    % (levels, per_image_ps / 1e6)}


def run_native(args, dist, rank, world, local):
    import realtimedepthdiffusion_b200 as rtdd
    from realtimedepthdiffusion_b200 import synth
    rows, cols, seed = WORKLOADS[args.workload]
    # N > 1: image i -> rank i mod N; every rank gets its own seed
    bgr, scribble, edited = synth.synth_case(rows, cols, seed + rank + args.seed_offset)
    ctx = rtdd.DepthDiffusion(rows, cols)
    stream = torch.cuda.Stream()
    ctx.set_stream(stream)
    total_ps, per_level = pixel_sweeps(rows, cols, ctx.levels)
    ctx.frame_set_image(bgr)
    h_ann = torch.from_numpy(synth.annotation_plane(scribble, edited)).pin_memory()
    h_scr = torch.from_numpy(scribble).pin_memory()
    h_edt = torch.from_numpy(edited).pin_memory()
    h_out = torch.zeros((rows, cols), dtype=torch.uint8).pin_memory()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    with torch.cuda.stream(stream):
        # ---- device-resident arm ---------------------------------------------------------------
        ctx.frame_solve_host_annotation(h_ann, 1000, h_out)      # uploads the annotation once, builds graphs
        for _ in range(args.warmup):
            ctx.frame_solve(1000)
        ctx.sync()
        sampler = ClockSampler(local)
        sampler.start()
        barrier(dist)
        launches0 = ctx.launch_count
        ev0.record(stream)
        for _ in range(args.steps):
            ctx.frame_solve(1000)
        ev1.record(stream)
        ctx.sync()
        barrier(dist)
        launches = ctx.launch_count - launches0
        ms_dev = max_over_ranks(dist, ev0.elapsed_time(ev1) / args.steps)
        if args.dump_outputs and rank == 0:
            # copied now: every later frame starts its coarsest level from this one's depth (main.cpp:257)
            dumped = [("depth", ctx.frame_plane(ctx.PLANE_DEPTH, 0).cpu().numpy()),
                      ("depth_u8", ctx.frame_plane(ctx.PLANE_DEPTH_U8, 0).cpu().numpy())]
        lvl_ms = [ctx.level_sweep_ms(l) for l in range(ctx.levels)]
        # level 0 of the same device-resident frame once more, one frame at a time, for the roofline's launch average (the level
        # events can only be read between frames)
        l0_ms = []
        for _ in range(args.steps):
            ctx.frame_solve(1000)
            ctx.sync()
            l0_ms.append(ctx.level_sweep_ms(0)[0])

        # ---- end-to-end arm: the public call with HOST buffers, copies inside the timed region -----------------------
        def time_e2e(call):
            for _ in range(max(args.warmup // 2, 1)):
                call()
            barrier(dist)
            t, l0 = [], []
            for _ in range(args.steps):
                ev0.record(stream)
                call()                                            # synchronous: returns after the download
                ev1.record(stream)
                ev1.synchronize()
                t.append(ev0.elapsed_time(ev1))
                l0.append(ctx.level_sweep_ms(0)[0])
            barrier(dist)
            return max_over_ranks(dist, float(np.mean(t))), l0
        # the reference's persistent annotation format: ONE plane, 32 = not annotated (main.cpp:160-170), expanded on the device
        ms_e2e, l0_e2e = time_e2e(lambda: ctx.frame_solve_host_annotation(h_ann, 1000, h_out))
        plan_e2e = rtdd.DepthDiffusion.plan_passes(rows, cols, per_level[0][2], host_map=True)[0] if rows * cols >= (1 << 18) else None
        # main.cpp's own per-frame traffic (scribble + 3-channel edited, main.cpp:236-237), kept for drop-in parity
        ms_e2e3, _ = time_e2e(lambda: ctx.frame_solve_host(h_scr, h_edt, 1000, h_out))
        clocks = sampler.stop()

        # ---- effects on the solved depth (configs[2]'s second half), reported beside the solve ----
        eff = {}
        if rank == 0:
            from realtimedepthdiffusion_b200.api import pitched_empty
            import ctypes as C
            outs = [pitched_empty(rows, cols, torch.uint8, "cuda", channels=3, fill=0) for _ in range(3)]
            planes = {}
            for nm, which in (("bgr", ctx.PLANE_BGR), ("gray", ctx.PLANE_GRAY), ("depth", ctx.PLANE_DEPTH)):
                p, pi, r, c = C.c_void_p(), C.c_size_t(), C.c_int(), C.c_int()
                rtdd._native.lib.rtdd_frame_plane(ctx._h, which, 0, C.byref(p), C.byref(pi), C.byref(r), C.byref(c))
                planes[nm] = (p, pi.value)
            L = rtdd._native.lib

            def t_eff(fn, reps=5):
                fn()
                ctx.sync()
                ev0.record(stream)
                for _ in range(reps):
                    fn()
                ev1.record(stream)
                ev1.synchronize()
                return ev0.elapsed_time(ev1) / reps
            o = [(C.c_void_p(t.data_ptr()), t.stride(0)) for t in outs]
            b, g, d = planes["bgr"], planes["gray"], planes["depth"]
            px = rows * cols
            ms = t_eff(lambda: L.rtdd_desaturate(ctx._h, b[0], b[1], g[0], g[1], d[0], d[1], o[0][0], o[0][1], rows, cols))
            eff["desaturation"] = {"ms": ms, "GB/s": 11.0 * px / ms / 1e6}
            ms = t_eff(lambda: L.rtdd_haze(ctx._h, b[0], b[1], d[0], d[1], o[1][0], o[1][1], rows, cols))
            eff["haze"] = {"ms": ms, "GB/s": 10.0 * px / ms / 1e6}
            ms = t_eff(lambda: L.rtdd_defocus(ctx._h, b[0], b[1], d[0], d[1], o[2][0], o[2][1], rows, cols))
            eff["defocus"] = {"ms": ms, "GB/s": 10.0 * px / ms / 1e6}
            ms = t_eff(lambda: L.rtdd_effects_fused(ctx._h, b[0], b[1], g[0], g[1], d[0], d[1], o[0][0], o[0][1], o[1][0], o[1][1],
                                                    o[2][0], o[2][1], rows, cols))
            eff["fused_all_three"] = {"ms": ms, "GB/s": 17.0 * px / ms / 1e6}
            # the frame context knows its image is unchanged between frames: summed-area table built once per image
            ms = t_eff(lambda: L.rtdd_frame_effects(ctx._h, o[0][0], o[0][1], o[1][0], o[1][1], o[2][0], o[2][1]))
            eff["frame_effects_cached_table"] = {"ms": ms, "GB/s": 17.0 * px / ms / 1e6}
            # configs[2] as one per-frame step: solve + the three effects, device-resident
            ms = t_eff(lambda: (ctx.frame_solve(1000), L.rtdd_frame_effects(ctx._h, o[0][0], o[0][1], o[1][0], o[1][1], o[2][0], o[2][1])), reps=10)
            eff["solve_plus_effects_frame"] = {"ms": ms}

    batch = None if args.no_batch else batch256_1080p(rtdd, dist, rank, world, stream)
    strips = None if args.no_strips else strips16k_record(rtdd, dist, rank, world, stream, args)

    peak, peak_src = peaks()
    r0, c0, it0 = per_level[0]
    l0 = float(np.mean(l0_ms))
    k0 = lvl_ms[0][2]
    achieved = BYTES_PER_PIXEL_SWEEP * r0 * c0 * it0 / (l0 * 1e-3) / 1e9
    line = {
        "metric": "Mpixel-sweeps/s", "value": total_ps * world / (ms_dev * 1e-3) / 1e6, "unit": "Mpixel-sweeps/s",
        "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_dev, "ms_per_solve": ms_dev,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_string(rows, cols, seed, ctx.levels, per_level, total_ps),
                   "l2": "no explicit flush: the solve streams a %.0f MB working set (> 126 MB L2) and every level's planes are rewritten each step"
                         % (sum(r * c for r, c, _ in per_level) * 19 / 1e6),
                   "parallelism": "dp%d" % world},
        "e2e": {"value": total_ps * world / (ms_e2e * 1e-3) / 1e6, "unit": "Mpixel-sweeps/s", "ms_per_solve": ms_e2e,
                "h2d_bytes_per_step": int(h_ann.numel()), "d2h_bytes_per_step": int(h_out.numel()),
                "call": "rtdd_frame_solve_host_annotation: the annotation as ONE u8 plane (32 = not annotated, main.cpp:160-170) from pinned host "
                        "memory, expanded on the device; 8-bit depth map back to pinned host memory",
                "download": "the last level-0 pass stores the 8-bit map into the pinned host plane itself, over PCIe while it computes "
                            "(rtdd.h zero_copy_out); for that the level runs its passes as %s and takes %.3f ms instead of %.3f"
                            % (plan_e2e, float(np.mean(l0_e2e)), float(np.mean(l0_ms))),
                "three_plane_upload": {"ms_per_solve": ms_e2e3, "value": total_ps * world / (ms_e2e3 * 1e-3) / 1e6,
                                       "h2d_bytes_per_step": int(h_scr.numel() + h_edt.numel()),
                                       "call": "rtdd_frame_solve_host: scribble + 3-channel edited planes, main.cpp:236-237's own traffic"}},
        "gpu_launches": int(launches),
        "roofline": {"bound": "hbm", "limiter": "instruction issue (see note)",
                     "kernel": "level-0 sweep kernel (%dx%d, %d sweeps in %d launches)" % (c0, r0, it0, k0),
                     "achieved": achieved, "peak": peak, "peak_source": peak_src, "unit": "GB/s", "frac": achieved / peak,
                     "traffic": NCU_TRAFFIC_BYTES_PER_LAUNCH.get(args.workload), "algorithmic_bytes_per_launch": BYTES_PER_PIXEL_SWEEP * r0 * c0 * it0 / k0,
                     "avg_launch_ms": l0 / k0,
                     "note": "achieved = 17 B x pixel-sweeps / time is the EFFECTIVE sweep bandwidth (SURVEY.md 8d): the kernel is temporally "
                             "blocked (several sweeps per HBM round trip), so its real DRAM traffic (`traffic`, ncu, per launch; null when no "
                             "capture exists for this workload) is far below the algorithmic bytes and frac may exceed 1; the kernel is "
                             "issue-bound, not HBM-bound (profiles/)"},
        "levels": [{"level": l, "size": "%dx%d" % (per_level[l][1], per_level[l][0]), "sweeps": per_level[l][2], "ms": lvl_ms[l][0],
                    "launches": lvl_ms[l][2], "us_per_sweep": 1e3 * lvl_ms[l][0] / max(per_level[l][2], 1),
                    "Gpixel-sweeps/s": per_level[l][0] * per_level[l][1] * per_level[l][2] / (lvl_ms[l][0] * 1e-3) / 1e9}
                   for l in range(ctx.levels)],
        "effects": eff,
        "batch256_1080p": batch,
        "strips16k": strips,
        "clocks": clocks,
    }
    ctx.close()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, dumped)
    return line


def strips16k_record(rtdd, dist, rank, world, stream, args):
    """BASELINE configs[4] (SURVEY.md 8d config 5): ONE 16384 x 16384 synthetic image (seed 1005, synthesised on every device), cut
    into row strips over the N ranks by the native strip frame (rtdd_strip_frame_*: C++ frame loop, H = 16 ghost rows, passes of
    8 sweeps, staged peer-memory halo exchange over NVLink -- no NCCL on the data path).  Two measurements, each against the
    one-GPU time of the same run: (i) the finest level alone, 64 sweeps incl. its edge-weight pass, (ii) the full 9-level pyramid
    (1993 sweeps; its 1.5 ms of coarse levels cannot be split and are solved by every rank).  Strong scaling:
    efficiency = t(1 GPU) / (N x t(N GPUs)).  Every rank also solves the whole image alone and compares its own rows bit for bit."""
    from realtimedepthdiffusion_b200 import stripframe, synth_device
    size, halo, pass_sweeps, l0_sweeps = args.strips_size, 16, 8, 64
    sf = stripframe.StripFrameRank(size, size, rank, world, halo, pass_sweeps, 1 << 22)
    ctx = sf.ctx
    ctx.set_stream(stream)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with torch.cuda.stream(stream):
        bgr, scribble, edited = synth_device.synth_case_device(size, size, 1005, ctx)
        sf.set_image_device(bgr)
        sf.set_annotation_device(scribble, edited)
        if world > 1:
            sf.connect(dist)
        solo = rtdd.DepthDiffusion(size, size)
        solo.set_stream(stream)
        one = stripframe.StripFrameRank.__new__(stripframe.StripFrameRank)
        one.ctx, one.rank, one.world, one.rows, one.cols = solo, 0, 1, size, size
        solo._ck(rtdd._native.lib.rtdd_strip_frame_setup(solo._h, 0, 1, halo, pass_sweeps, 1 << 22))
        one.set_image_device(bgr)
        one.set_annotation_device(scribble, edited)

        def timed(who, l0, sync_ranks):
            def frame():
                who.reset_first_frame_guess()                      # outside the timed region
                torch.cuda.synchronize()
                if sync_ranks:
                    barrier(dist)
                ev0.record(stream)
                if l0:
                    who.level0(l0)
                elif who.world == 1:
                    who.ctx.frame_solve(1000)                      # one GPU: the whole frame as ONE graph, the fastest single-GPU path
                else:
                    who.solve(1000)
                ev1.record(stream)
                who.ctx.sync()
                return ev0.elapsed_time(ev1)
            for _ in range(2):
                frame()
            return max_over_ranks(dist, float(np.median([frame() for _ in range(5)])))

        res = {}
        split, a, b, w0, w1 = sf.rows_of(0)
        for tag, l0 in (("level0_x64", l0_sweeps), ("full_pyramid", 0)):
            t_n = timed(sf, l0, True)
            t_1 = timed(one, l0, False)                            # every rank alone on its own GPU (no exchange): the 1-GPU time
            mine = sf.plane(ctx.PLANE_DEPTH)[a:b]
            ref = one.plane(solo.PLANE_DEPTH)[a:b]
            same = torch.equal(mine.contiguous().view(torch.int32), ref.contiguous().view(torch.int32))
            if not l0:
                same = same and torch.equal(sf.plane(ctx.PLANE_DEPTH_U8)[a:b], one.plane(solo.PLANE_DEPTH_U8)[a:b])
            f = torch.tensor([1.0 if same else 0.0], dtype=torch.float64, device="cuda")
            if dist is not None:
                dist.all_reduce(f, op=dist.ReduceOp.MIN)
            total, per = pixel_sweeps(size, size, ctx.levels)
            ps = size * size * l0_sweeps if l0 else total
            res[tag] = {"ms_n_gpus": t_n, "ms_1_gpu": t_1, "speedup": t_1 / t_n, "efficiency": t_1 / (world * t_n),
                        "Mpixel-sweeps/s": ps / (t_n * 1e-3) / 1e6, "pixel_sweeps": ps, "bit_identical_to_single_gpu": bool(f.item() > 0.5)}
        res.update({"image": "%dx%d, seed 1005, %d levels" % (size, size, ctx.levels), "n_gpus": world, "scaling": "strong",
                    "split_levels": [sf.rows_of(l)[0] for l in range(ctx.levels)], "halo_rows": halo, "sweeps_per_pass": pass_sweeps,
                    "exchange": "staged peer memory (rtdd_strip_push / rtdd_strip_pull over NVLink, CUDA IPC between the ranks' processes)"
                                if world > 1 else "none (one rank)",
                    "driver": "rtdd_strip_frame_* (C++ frame loop inside librtdd.so)"})
        solo.close()
    sf.close()
    return res


def run_reference(args, dist, rank, world, local):
    """The reference's own kernels through the reference's own functions (libref.so).  Nothing of the product is imported
    here: synth / planes / refnames are loaded by path (oracle.binding.pkg_file), so librtdd.so is not in this process."""
    from oracle import binding as ob
    from oracle.mainloop import MainLoop, pitch, ptr
    synth = ob.pkg_file("synth")
    if rank != 0:
        return None
    if not os.path.exists(ob.LIBREF):
        return {"impl": "reference", "unavailable": "oracle/_ref/libref.so was not built (needs /root/reference at build time)"}
    rows, cols, seed = WORKLOADS[args.workload]
    bgr, scribble, edited = synth.synth_case(rows, cols, seed)
    api = ob.ref_api()
    loop = MainLoop(api, bgr)
    total_ps, per_level = pixel_sweeps(rows, cols, loop.levels)
    # staging = one true reference frame (CPU pyrUp like main.cpp's fallback); keeps each level's input guess
    loop.frame(scribble, edited, 1000, keep_levels=True)
    staged = {l: torch.from_numpy(d["in"]).cuda() for l, d in loop.per_level.items()}
    h_scr = torch.from_numpy(scribble).pin_memory()
    h_edt = torch.from_numpy(edited.reshape(rows, -1)).pin_memory()
    h_out = torch.zeros((rows, cols), dtype=torch.uint8).pin_memory()
    L = loop.levels
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def gpu_frame(host):
        # the GPU* calls of main.cpp:236-283; depth prolongation (OpenCV, outside the reference's own code)
        # is replaced by a device copy of the staged guess, which favours this arm
        if host:
            loop.scribble[0].copy_(h_scr, non_blocking=True)
            loop.edited[0].copy_(h_edt, non_blocking=True)
        for l in range(1, L):
            pr, pc = loop.sizes[l - 1]
            r, c = loop.sizes[l]
            api["GPUPyrDownAnnotation"](ptr(loop.scribble[l - 1]), pitch(loop.scribble[l - 1]), ptr(loop.edited[l - 1]),
                                        pitch(loop.edited[l - 1]), pr, pc, ptr(loop.scribble[l]), pitch(loop.scribble[l]),
                                        ptr(loop.edited[l]), pitch(loop.edited[l]), r, c)
        loop.convert(L - 1)
        for l in range(L - 1, -1, -1):
            r, c = loop.sizes[l]
            api["GPUMatrixFreeSolver"](ptr(loop.depth[l]), pitch(loop.depth[l]), ptr(loop.scribble[l]), pitch(loop.scribble[l]),
                                       ptr(loop.gray[l]), pitch(loop.gray[l]), r, c, 0.4, per_level[l][2], 1e-5, l)
            if l > 0:
                loop.depth[l - 1].copy_(staged[l - 1])
                loop.convert(l - 1)
        if host:
            q = loop.depth[0].round().clamp_(0, 255).to(torch.uint8)     # GpuMat::convertTo stand-in
            h_out.copy_(q, non_blocking=True)
            torch.cuda.synchronize()

    steps, warm = args.steps, args.warmup
    for _ in range(warm):
        gpu_frame(False)
    torch.cuda.synchronize()
    sampler = ClockSampler(local)
    sampler.start()
    ev0.record()
    for _ in range(steps):
        gpu_frame(False)
    ev1.record()
    torch.cuda.synchronize()
    ms_dev = ev0.elapsed_time(ev1) / steps
    for _ in range(max(warm // 2, 1)):
        gpu_frame(True)
    t = []
    for _ in range(steps):
        ev0.record()
        gpu_frame(True)
        ev1.record()
        ev1.synchronize()
        t.append(ev0.elapsed_time(ev1))
    clocks = sampler.stop()
    ms_e2e = float(np.mean(t))
    # effects, once each (the reference's defocus gathers up to 110^2 taps per pixel at 4K)
    eff = {}
    r, c = rows, cols
    out = torch.zeros_like(loop.orig)
    for name in ("GPUSimulateDesaturation", "GPUSimulateHaze", "GPUSimulateDefocus"):
        torch.cuda.synchronize()
        ev0.record()
        if name == "GPUSimulateDesaturation":
            api[name](ptr(loop.orig), pitch(loop.orig), ptr(loop.gray[0]), pitch(loop.gray[0]), ptr(loop.depth[0]), pitch(loop.depth[0]),
                      ptr(out), pitch(out), r, c)
        else:
            api[name](ptr(loop.orig), pitch(loop.orig), ptr(loop.depth[0]), pitch(loop.depth[0]), ptr(out), pitch(out), r, c)
        ev1.record()
        ev1.synchronize()
        eff[name] = {"ms": ev0.elapsed_time(ev1)}
    launches = sum(p[2] + 5 for p in per_level) + 2 * L - 1
    loop.close()
    value = total_ps / (ms_dev * 1e-3) / 1e6
    return {
        "impl": "reference", "metric": "Mpixel-sweeps/s", "value": value, "unit": "Mpixel-sweeps/s", "n_gpus": 1, "steps": steps, "warmup": warm,
        "ms_per_step": ms_dev, "ms_per_solve": ms_dev, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic",
        "config": {"workload": workload_string(rows, cols, seed, L, per_level, total_ps),
                   "l2": "no explicit flush: the solve streams a %.0f MB working set (> 126 MB L2) and every level's planes are rewritten each step"
                         % (sum(r * c for r, c, _ in per_level) * 24 / 1e6),
                   "parallelism": "dp1",
                   "how": "the reference's own GPU* functions (oracle/_ref/libref.so = /root/reference/src/*.cu unmodified, nvcc -O3 sm_100a) driven by "
                          "main.cpp's restated loop; OpenCV pyrUp replaced by a device copy of the staged guess (favours this arm); one GPU whatever "
                          "--gpus says (the reference has no multi-GPU path)"},
        "e2e": {"value": total_ps / (ms_e2e * 1e-3) / 1e6, "unit": "Mpixel-sweeps/s", "ms_per_solve": ms_e2e,
                "h2d_bytes_per_step": int(h_scr.numel() + h_edt.numel()), "d2h_bytes_per_step": int(h_out.numel()),
                "note": "reference kernels run on the GPU; main.cpp's own per-frame uploads/downloads (:236-237, :291) are inside the timed region"},
        "gpu_launches": launches, "effects": eff, "clocks": clocks,
        "reference_device": "1x B200 (the reference has no CPU path; its own implementation is CUDA)",
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--workload", default="4k", choices=sorted(WORKLOADS))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-batch", action="store_true", help="skip the configs[3] record (256 x 1080p)")
    ap.add_argument("--no-strips", action="store_true", help="skip the configs[4] record (16384^2 row strips)")
    ap.add_argument("--strips-size", type=int, default=16384, help="side of the configs[4] image")
    ap.add_argument("--seed-offset", type=int, default=0, help="extra offset on the synthetic image seed (diagnostics)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's depth maps to DIR (see the module docstring)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "native":
        ap.error("--dump-outputs covers the native path")
    args.warmup = max(args.warmup, 3)
    # stdout carries exactly ONE line, the JSON result: anything libraries print there meanwhile (NCCL's version banner
    # under NCCL_DEBUG=VERSION, for one) is sent to stderr instead
    sys.stdout.flush()
    result_fd = os.dup(1)
    os.dup2(2, 1)

    def emit(obj):
        sys.stdout.flush()
        os.write(result_fd, (json.dumps(obj) + "\n").encode())

    if not torch.cuda.is_available():
        emit({"error": "no CUDA device: bench.py measures the CUDA path only (no CPU fallback)"})
        sys.exit(2)
    if args.impl == "reference":
        # rank 0 alone runs the reference arm; the other ranks exit 0 without work (no process group needed)
        rank = int(os.environ.get("RANK", "0"))
        if rank != 0:
            return
        torch.cuda.set_device(int(os.environ.get("LOCAL_RANK", "0")))
        dist, world, local = None, 1, int(os.environ.get("LOCAL_RANK", "0"))
        line = run_reference(args, dist, rank, world, local)
    else:
        dist, rank, world, local = dist_setup(args.gpus)
        line = run_native(args, dist, rank, world, local)
    if rank == 0 and line is not None:
        if "unavailable" not in line and not args.no_cpu_baseline and (world == 1 or args.impl == "reference"):
            rows, cols, _ = WORKLOADS[args.workload]
            line["cpu_baseline"] = cpu_baseline(rows, cols, pyramid_levels(rows, cols))
        emit(line)
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
