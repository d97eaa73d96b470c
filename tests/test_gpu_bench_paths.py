"""The frame paths bench.py times, at the sizes it times them, against the CPU oracle (run on a B200).

bench.py's numbers rest on one claim: every pass plan gives the same bits, so the planner changes only speed.  These tests run
the kernels that carry out those plans where the plans occur and compare every result with oracle.binding.FrameState:
- the e2e frame sequence of run_native (720p, 1080p, 4K, 8K): the 8-bit map stored by the last level-0 pass into pinned host
  memory (at 8K that pass is also the level's first), frames that start the coarsest level from the previous frame's depth,
  the three-plane upload, and the effects on the frame's own pitched planes;
- contexts planned for throughput (plan_throughput = 1) and the batch256_1080p schedule: eight of them on their own streams,
  three images queued on each, driven round-robin from one host thread;
- the process-wide knobs pass_planner = 0 and pdl = 0, which include/rtdd.h documents as leaving results unchanged.

Bars (those of tests/test_gpu_parity.py): fp32 depth planes bit-exact at every level, 8-bit maps and effects byte-identical,
haze within 1 grey level on < 0.1 % of values (glibc expf vs libdevice expf).  After every frame the launches of each level's
sweeps are checked against the plan rtdd_plan_passes reports for it, so a frame that silently took another path (the staged
copy instead of the host map, the latency plan instead of the throughput plan) fails even where the bytes would agree.

Runtime: about 40 oracle frames plus the host synthesis of the 8K image, most of it CPU time.  The whole file took 28 s on an
NVIDIA B200 at a 1000 W power limit, with 16 host cores."""
import ctypes as C
import math

import numpy as np
import pytest
import torch

from oracle import binding as ob
from realtimedepthdiffusion_b200 import synth
from tests import refocus_reference
from tests.harness import to_host

pytestmark = pytest.mark.gpu

# bench.py WORKLOADS: rows, cols and the synth.synth_case seed of each --workload
WORKLOADS = {"720p": (720, 1280, 1001), "1080p": (1080, 1920, 1002), "4k": (2160, 3840, 1003), "8k": (4320, 7680, 1004)}
# bench.py batch256_1080p: image i is synth_device.synth_case_device(1080, 1920, 2000 + i), K contexts in flight.  24 images
# put three behind one another on every context's stream.
BATCH_SEED, BATCH_CONTEXTS, BATCH_IMAGES = 2000, 8, 24
MAX_ITERATIONS = 1000
# pick_variant (rtdd_abi.cu): a level of at most this many pixels (and >= 8 sweeps) is solved by the cluster-resident kernel, in one launch
RESIDENT_MAX_PIXELS = 49152
SENTINEL = 0xA5                # fills every host map before a call: a store that never happened cannot pass


@pytest.fixture(scope="module")
def rtdd():
    import realtimedepthdiffusion_b200 as pkg
    return pkg


@pytest.fixture(scope="module")
def sm_count():
    return torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count


def ingest(annotation, bgr):
    """main.cpp:160-170: scribble = 255 and edited = the annotated value where annotation != 32, else scribble = 0, edited = bgr."""
    on = annotation != 32
    scribble = np.where(on, 255, 0).astype(np.uint8)
    edited = np.where(on[..., None], annotation[..., None], bgr).astype(np.uint8)
    return scribble, edited


class OracleFrames:
    """One bench workload's inputs and its oracle frames.  Frame k (from 1) is the k-th solve of ONE FrameState with the same
    annotation: every later frame starts the coarsest level from the one before (main.cpp:257), as the library does."""

    def __init__(self, rows, cols, seed):
        self.bgr, self.scribble, self.edited = synth.synth_case(rows, cols, seed)
        self.ann = synth.annotation_plane(self.scribble, self.edited)
        s, e = ingest(self.ann, self.bgr)
        # frame 1 uploads the annotation, frame 4 the two planes: both must describe the same frame
        assert np.array_equal(s, self.scribble) and np.array_equal(e, self.edited)
        self.state = ob.FrameState(self.bgr)
        self.frames = []

    def frame(self, k):
        """-> (8-bit map, [fp32 depth of every level]) of frame k."""
        while len(self.frames) < k:
            u8 = self.state.solve(self.scribble, self.edited, MAX_ITERATIONS)
            self.frames.append((u8, list(self.state.depth)))
        return self.frames[k - 1]


@pytest.fixture(scope="module")
def oracle():
    cache = {}

    class Cases:
        def get(self, workload):
            if workload not in cache:
                cache[workload] = OracleFrames(*WORKLOADS[workload])
            return cache[workload]

        def drop(self, workload):
            cache.pop(workload, None)

    return Cases()


def expected_launches(rows, cols, iters, sms, host_map, throughput, planner):
    """Sweep launches of one level: the resident kernel's one, the planner's passes, or (pass_planner = 0) passes of one
    length T -- rtdd_plan_blocked's from 2^18 pixels on and in throughput contexts, 11 below (pick_variant, rtdd_abi.cu)."""
    from realtimedepthdiffusion_b200 import _native
    from realtimedepthdiffusion_b200.api import DepthDiffusion
    if rows * cols <= RESIDENT_MAX_PIXELS and iters >= 8:
        return 1
    if planner:
        return len(DepthDiffusion.plan_passes(rows, cols, iters, sm_count=sms, host_map=host_map, throughput=throughput)[0])
    T = 11
    if rows * cols >= (1 << 18) or throughput:
        t, form = C.c_int(), C.c_int()
        assert _native.lib.rtdd_plan_blocked(rows, cols, iters, sms, C.byref(t), C.byref(form)) == 0
        T = t.value
    return math.ceil(iters / min(T, 16, iters))


def assert_plans_ran(ctx, sms, host_map=False, throughput=False, planner=True):
    """The kernels each level's last solve launched are those of the plan the planner reports (host_map: level 0 only)."""
    from realtimedepthdiffusion_b200.api import level_iterations
    for level, (rows, cols) in enumerate(ctx.sizes):
        iters = level_iterations(MAX_ITERATIONS, ctx.levels, level)
        _, sweeps, launches = ctx.level_sweep_ms(level)
        want = expected_launches(rows, cols, iters, sms, host_map and level == 0, throughput, planner)
        assert (sweeps, launches) == (iters, want), \
            "level %d (%dx%d): %d sweeps in %d launches, the plan has %d in %d" % (level, cols, rows, sweeps, launches, iters, want)


def assert_frame(ctx, want, u8_maps, what):
    """Every level's fp32 plane (coarsest first: the first one named is where a difference began) and the 8-bit maps."""
    want_u8, want_depth = want
    for level in range(ctx.levels - 1, -1, -1):
        got = ctx.frame_plane(ctx.PLANE_DEPTH, level).cpu().numpy()
        bad = got.view(np.uint32) != want_depth[level].view(np.uint32)
        assert not bad.any(), "%s: level %d fp32 differs on %d px, first at %s" % (what, level, int(bad.sum()), np.argwhere(bad)[0])
    for name, got in [("device map", ctx.frame_plane(ctx.PLANE_DEPTH_U8, 0).cpu().numpy())] + u8_maps:
        bad = got != want_u8
        assert not bad.any(), "%s: %s differs on %d px, rows %s" % (what, name, int(bad.sum()), np.unique(np.nonzero(bad)[0])[:8])


def pinned_like(a, fill=None):
    """A pinned host copy of the u8 array `a`, or a pinned plane of its shape filled with `fill`."""
    t = torch.empty(a.shape, dtype=torch.uint8).pin_memory()
    if fill is None:
        t.copy_(torch.from_numpy(a))
    else:
        t.fill_(fill)
    return t


# ---- bench.py run_native: the e2e frame sequence and the effects --------------------------------------------------------------

def oracle_defocus_at(bgr, depth, y, x, K):
    """oracle_defocus (oracle/depth_oracle.c) at one pixel: box [y-h, y+h) x [x-h, x+h), h = (int)((double)((float)K * d) / 255) / 2,
    fp32 sums in raster order, fp32 mean truncated; an empty box keeps the pixel."""
    q = float(np.float32(K) * depth[y, x]) / 255.0
    an = 0 if q != q else 2147483647 if q >= 2147483647.0 else -2147483648 if q <= -2147483648.0 else int(q)
    h = int(an / 2)                                              # C division: toward zero
    rows, cols = depth.shape
    box = bgr[max(y - h, 0):max(min(y + h, rows), 0), max(x - h, 0):max(min(x + h, cols), 0)].reshape(-1, 3)
    if len(box) == 0:
        return bgr[y, x]
    sums = np.cumsum(box.astype(np.float32), axis=0, dtype=np.float32)[-1]
    return (sums / np.float32(len(box))).astype(np.uint8)


def reference_effects(bgr, gray, depth):
    """desaturation and haze from the oracle; defocus = the refocus reference at focus 0, band 0, aperture K, which is the
    reference defocus for every depth <= 255 while K <= 257 (include/rtdd.h), and oracle_defocus per pixel elsewhere."""
    rows, cols = depth.shape
    K = ob.defocus_kernel_size(rows, cols)
    assert K <= 257
    # the boxes reach the size of the deepest paintable value (254): the summed-area path runs at about its full size (K = 220 at 8K)
    deepest = refocus_reference.half_sides(np.float32([[254.0]]), 0.0, 0.0, K)[0, 0]
    assert refocus_reference.half_sides(depth, 0.0, 0.0, K).max() >= deepest
    defocus = refocus_reference.refocus(bgr, depth, 0.0, 0.0, -1)
    outside = np.argwhere(~((depth >= 0) & (depth <= 255)))
    assert len(outside) < 20000, "%d solved depths outside [0, 255]" % len(outside)
    for y, x in outside:
        defocus[y, x] = oracle_defocus_at(bgr, depth, y, x, K)
    return ob.desaturate(bgr, gray, depth), ob.haze(bgr, depth), defocus, len(outside)


def check_effects(rtdd, ctx, bgr, gray, depth, separate):
    """bench.py's effects: rtdd_effects_fused (and, with `separate`, the three single calls) through raw pointers to the frame's
    own pitched BGR, gray and depth planes, against the references; fused equals separate byte for byte."""
    from realtimedepthdiffusion_b200.api import pitched_empty
    lib = rtdd._native.lib
    rows, cols = depth.shape
    planes = {}
    for name, which in (("bgr", ctx.PLANE_BGR), ("gray", ctx.PLANE_GRAY), ("depth", ctx.PLANE_DEPTH)):
        p, pi, r, c = C.c_void_p(), C.c_size_t(), C.c_int(), C.c_int()
        ctx._ck(lib.rtdd_frame_plane(ctx._h, which, 0, C.byref(p), C.byref(pi), C.byref(r), C.byref(c)))
        planes[name] = (p, pi.value)
    b, g, d = planes["bgr"], planes["gray"], planes["depth"]
    outs = [pitched_empty(rows, cols, torch.uint8, "cuda", channels=3, fill=SENTINEL) for _ in range(6)]
    o = [(C.c_void_p(t.data_ptr()), t.stride(0)) for t in outs]
    if separate:
        ctx._ck(lib.rtdd_desaturate(ctx._h, b[0], b[1], g[0], g[1], d[0], d[1], o[0][0], o[0][1], rows, cols))
        ctx._ck(lib.rtdd_haze(ctx._h, b[0], b[1], d[0], d[1], o[1][0], o[1][1], rows, cols))
        ctx._ck(lib.rtdd_defocus(ctx._h, b[0], b[1], d[0], d[1], o[2][0], o[2][1], rows, cols))
    ctx._ck(lib.rtdd_effects_fused(ctx._h, b[0], b[1], g[0], g[1], d[0], d[1], o[3][0], o[3][1], o[4][0], o[4][1], o[5][0], o[5][1],
                                   rows, cols))
    ctx.sync()
    got = [to_host(t, 3) for t in outs]
    desat, haze, defocus, outside = reference_effects(bgr, gray, depth)
    fused = got[3:]
    assert np.array_equal(fused[0], desat), "desaturation differs on %d values" % int((fused[0] != desat).sum())
    h = fused[1].astype(np.int16) - haze.astype(np.int16)
    assert np.abs(h).max() <= 1 and (h != 0).mean() < 1e-3, (int(np.abs(h).max()), float((h != 0).mean()))
    assert np.array_equal(fused[2], defocus), "defocus differs on %d values (%d depths outside [0, 255])" % (int((fused[2] != defocus).sum()), outside)
    if separate:
        for name, a, f in zip(("desaturation", "haze", "defocus"), got[:3], fused):
            assert np.array_equal(a, f), "%s: fused and separate calls differ" % name


@pytest.mark.parametrize("workload", ["720p", "1080p", "4k", "8k"])
def test_bench_frame_sequence_and_effects(rtdd, oracle, sm_count, workload):
    """run_native's order on one context with pinned host planes: frame_solve_host_annotation into a pinned map (the host-map
    plan at level 0), frame_solve twice (state carried), frame_solve_host with the two planes, then the effects at 4K and 8K."""
    rows, cols, _ = WORKLOADS[workload]
    case = oracle.get(workload)
    ctx = rtdd.DepthDiffusion(rows, cols)
    stream = torch.cuda.Stream()
    ctx.set_stream(stream)
    try:
        ctx.frame_set_image(case.bgr)
        h_ann, h_scr, h_edt = pinned_like(case.ann), pinned_like(case.scribble), pinned_like(case.edited)
        h_out = pinned_like(case.ann, SENTINEL)
        with torch.cuda.stream(stream):
            ctx.frame_solve_host_annotation(h_ann, MAX_ITERATIONS, h_out)
            assert_frame(ctx, case.frame(1), [("pinned host map", h_out.numpy())], "frame 1 (annotation, pinned map)")
            assert_plans_ran(ctx, sm_count, host_map=True)
            for k in (2, 3):
                ctx.frame_solve(MAX_ITERATIONS)
                ctx.sync()
                assert_frame(ctx, case.frame(k), [], "frame %d (device-resident)" % k)
                assert_plans_ran(ctx, sm_count)
            h_out.fill_(SENTINEL)
            ctx.frame_solve_host(h_scr, h_edt, MAX_ITERATIONS, h_out)
            assert_frame(ctx, case.frame(4), [("pinned host map", h_out.numpy())], "frame 4 (two planes, pinned map)")
            assert_plans_ran(ctx, sm_count, host_map=True)
            if workload in ("4k", "8k"):
                check_effects(rtdd, ctx, case.bgr, case.state.gray[0], case.frame(4)[1][0], separate=workload == "8k")
    finally:
        ctx.close()
        if workload == "8k":
            oracle.drop(workload)


# ---- contexts planned for throughput, and the process-wide knobs ----------------------------------------------------------------

@pytest.mark.parametrize("workload", ["720p", "1080p", "4k"])
def test_throughput_planned_context(rtdd, oracle, sm_count, workload):
    """plan_throughput = 1 (per context): other pass plans and tile forms, same frames 1 and 2."""
    rows, cols, _ = WORKLOADS[workload]
    case = oracle.get(workload)
    ctx = rtdd.DepthDiffusion(rows, cols)
    try:
        ctx.set_tuning("plan_throughput", 1)
        ctx.frame_set_image(case.bgr)
        h_out = pinned_like(case.ann, SENTINEL)
        ctx.frame_solve_host_annotation(pinned_like(case.ann), MAX_ITERATIONS, h_out)
        assert_frame(ctx, case.frame(1), [("pinned host map", h_out.numpy())], "frame 1")
        assert_plans_ran(ctx, sm_count, host_map=True, throughput=True)
        ctx.frame_solve(MAX_ITERATIONS)
        ctx.sync()
        assert_frame(ctx, case.frame(2), [], "frame 2")
        assert_plans_ran(ctx, sm_count, throughput=True)
    finally:
        ctx.close()


@pytest.mark.parametrize("workload,knob", [("4k", "pass_planner"), ("1080p", "pdl")])
def test_process_wide_knobs_leave_the_frame_unchanged(rtdd, oracle, sm_count, workload, knob):
    """pass_planner = 0: one pass length per level (4K level 0 runs 7, 7, 7, 7, 3); pdl = 0: passes in plain stream order."""
    rows, cols, _ = WORKLOADS[workload]
    case = oracle.get(workload)
    ctx = rtdd.DepthDiffusion(rows, cols)
    try:
        ctx.set_tuning(knob, 0)
        ctx.frame_set_image(case.bgr)
        h_out = pinned_like(case.ann, SENTINEL)
        ctx.frame_solve_host_annotation(pinned_like(case.ann), MAX_ITERATIONS, h_out)
        assert_frame(ctx, case.frame(1), [("pinned host map", h_out.numpy())], "frame 1 with %s = 0" % knob)
        assert_plans_ran(ctx, sm_count, host_map=True, planner=knob != "pass_planner")
    finally:
        ctx.set_tuning(knob, 1)                  # process-wide: the other test modules rely on the defaults
        ctx.close()


# ---- bench.py batch256_1080p ------------------------------------------------------------------------------------------------------

def test_batch_schedule_of_throughput_contexts(rtdd, sm_count):
    """batch256_1080p's loop with 24 images: device-synthesised images parked in pinned memory, eight plan_throughput contexts on
    their own streams, the warm-up round, then set_image / solve_host_annotation / read_depth_u8 without synchronising, round
    robin from one host thread.  Every image has its own pinned output; each is compared with that image's oracle frame."""
    from realtimedepthdiffusion_b200 import synth_device
    rows, cols = 1080, 1920
    stream_main = torch.cuda.Stream()
    gen = rtdd.DepthDiffusion(rows, cols)
    gen.set_stream(stream_main)
    h_bgr, h_ann = [], []
    try:
        with torch.cuda.stream(stream_main):
            for i in range(BATCH_IMAGES):
                bgr, scribble, edited = synth_device.synth_case_device(rows, cols, BATCH_SEED + i, gen)
                hb = torch.empty((rows, cols, 3), dtype=torch.uint8).pin_memory()
                hb.view(rows, cols * 3).copy_(bgr)
                ha = torch.empty((rows, cols), dtype=torch.uint8).pin_memory()
                ha.copy_(synth_device.annotation_plane_device(scribble, edited))
                h_bgr.append(hb)
                h_ann.append(ha)
            torch.cuda.synchronize()
    finally:
        gen.close()
    ctxs = []
    warm = [pinned_like(np.zeros((rows, cols), np.uint8), SENTINEL) for _ in range(BATCH_CONTEXTS)]
    outs = [pinned_like(np.zeros((rows, cols), np.uint8), SENTINEL) for _ in range(BATCH_IMAGES)]
    try:
        for k in range(BATCH_CONTEXTS):
            c = rtdd.DepthDiffusion(rows, cols)
            st = torch.cuda.Stream()
            c.set_stream(st)
            c.set_tuning("plan_throughput", 1)
            ctxs.append((c, st))
        for k, (c, st) in enumerate(ctxs):                       # warm-up: the same calls as the timed loop
            c.frame_set_image(h_bgr[k])
            c.frame_solve_host_annotation(h_ann[k], MAX_ITERATIONS, None)
            c.frame_read_depth_u8(warm[k], sync=True)
        ev0 = torch.cuda.Event()
        ev0.record()
        for _, st in ctxs:
            st.wait_event(ev0)
        for j in range(BATCH_IMAGES):
            c, st = ctxs[j % BATCH_CONTEXTS]
            c.frame_set_image(h_bgr[j], sync=False)
            c.frame_solve_host_annotation(h_ann[j], MAX_ITERATIONS, None)
            c.frame_read_depth_u8(outs[j], sync=False)
        for _, st in ctxs:
            torch.cuda.current_stream().wait_stream(st)
        torch.cuda.synchronize()
        assert_plans_ran(ctxs[0][0], sm_count, throughput=True)
    finally:
        for c, _ in ctxs:
            c.close()
    for j in range(BATCH_IMAGES):
        bgr = h_bgr[j].numpy()
        scribble, edited = ingest(h_ann[j].numpy(), bgr)
        want = ob.FrameState(bgr).solve(scribble, edited, MAX_ITERATIONS)
        for name, got in [("batch", outs[j])] + ([("warm-up", warm[j])] if j < BATCH_CONTEXTS else []):
            bad = got.numpy() != want
            assert not bad.any(), "image %d (%s, context %d): %d px differ" % (j, name, j % BATCH_CONTEXTS, int(bad.sum()))
