"""The solver at edge-weight tables other than beta = 0.4, bit for bit against the oracle at the same beta (run on a B200).

Every golden vector, the bench and the other GPU tests load beta = 0.4, whose table has no zero entry and a denormal tail from
w[219].  Other tables send free pixels inside the image down paths that table never reaches: weight sums of exactly +0 (0 / 0 in
the kernels, `count == 0 -> 0` in the oracle) from beta = 0.45 on, sums below div_fast's 2^-100 and below pow2_scale's 2^-21,
all-ones tables (integer sums), and w[0] alone.  tests/weight_tables.py holds the grid and the inputs, and
tests/test_weight_tables_cpu.py shows that the inputs reach each regime.  Here every result is compared with
oracle.binding.solve_level / FrameState given the table of the same beta:
- level solves in every sweep form (one sweep per launch, the flat 128x32 form, the 128x64 TMA / LDG / cluster forms, the three
  builds of the cluster-resident kernel, and the automatic choice), with the residual of the last sweep;
- the planner's three forms under variant 0, the strip passes of the tolerance-driven solve, and a two-rank strip frame;
- whole frames into pinned host maps (the host-map plan at level 0), including one 3840x2160 frame;
- a table reloaded inside one context, after its CUDA graphs were captured, and through the reference-named shim;
- rtdd_load_weights refusing negative and non-finite beta (a documented deviation), with the previous table left in force.

Runtime: mostly oracle time on the host.  The whole file took 14 to 15 s of wall time on an NVIDIA B200 at a 1000 W power
limit, with 16 host cores."""
import ctypes as C

import numpy as np
import pytest
import torch

from oracle import binding as ob
from realtimedepthdiffusion_b200 import synth
from tests import weight_tables as wt
from tests.harness import MainLoop, to_dev, to_host
from tests.test_gpu_bench_paths import MAX_ITERATIONS, assert_frame, assert_plans_ran, ingest, pinned_like

pytestmark = pytest.mark.gpu
ITERS = 41
DEFAULT_TUNING = {"blocked_tile": 0, "blocked_tma": 2, "blocked_cluster": 2}

# name -> (variant, sweeps per pass, tunings): the sweep forms a level solve can take
FORMS = {
    "single-sweep": (1, 0, {}),
    "flat-128x32": (2, 7, {}),
    "tile64-tma3-cluster2": (2, 13, {"blocked_tile": 64, "blocked_tma": 3, "blocked_cluster": 2}),
    "tile64-tma3-cluster1": (2, 13, {"blocked_tile": 64, "blocked_tma": 3, "blocked_cluster": 1}),
    "tile64-tma1-cluster1": (2, 13, {"blocked_tile": 64, "blocked_tma": 1, "blocked_cluster": 1}),
    "tile64-tma1-cluster2": (2, 13, {"blocked_tile": 64, "blocked_tma": 1, "blocked_cluster": 2}),
    "tile64-ldg-cluster1": (2, 13, {"blocked_tile": 64, "blocked_tma": 0, "blocked_cluster": 1}),
    "tile64-ldg-cluster2": (2, 13, {"blocked_tile": 64, "blocked_tma": 0, "blocked_cluster": 2}),
    "automatic": (0, 0, {}),
}
# the cluster-resident kernel's three builds, by level shape: R = 1 up to 640 threads, R = 1 with 1024 threads, R = 2
RESIDENT = {"resident-r1-640": (135, 240), "resident-r1-1024": (256, 256), "resident-r2": (600, 100)}


@pytest.fixture(scope="module")
def rtdd():
    import realtimedepthdiffusion_b200 as pkg
    return pkg


@pytest.fixture(scope="module")
def sm_count():
    return torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count


def assert_bits(got, want, what, gray, depth, level, levels, lut):
    """Bit equality; on failure names the first differing pixel, its four link indices and its weight sum."""
    bad = got.view(np.uint32) != want.view(np.uint32)
    if bad.any():
        y, x = np.argwhere(bad)[0]
        idx = ob.index_to_weight(gray, depth, level, levels - 1)[y, x]
        w = lut[idx]
        s = np.float32(np.float32(np.float32(w[0] + w[1]) + w[2]) + w[3])
        pytest.fail("%s: %d px differ, first (y %d, x %d): got %r want %r, links (l, r, u, d) %s, weight sum %r"
                    % (what, int(bad.sum()), y, x, float(got[y, x]), float(want[y, x]), idx.tolist(), float(s)))


def solve_and_compare(rtdd, beta, variant, T, tuning, shape, level, levels, kinds=tuple(wt.INPUTS), residual=True, launches=None):
    """Every input of `kinds` at one level shape through one context at `beta`, against the oracle with beta's table
    (`launches`: the sweep kernels each solve must have taken)."""
    iters = ITERS
    rows, cols = shape
    lut = wt.table(beta)
    ctx = rtdd.DepthDiffusion(rows << level, cols << level, levels, beta=beta)
    assert tuple(ctx.sizes[level]) == (rows, cols)
    try:
        for k, v in tuning.items():
            ctx.set_tuning(k, v)
        ctx.set_sweep_variant(variant, T)
        for kind in kinds:
            gray, depth, scribble = wt.level_input(kind, rows, cols, level)
            want = ob.solve_level(depth, scribble, gray, iters, level, levels - 1, lut)
            d, s, g = to_dev(depth), to_dev(scribble), to_dev(gray)
            ctx.matrix_free_solver(d, s, g, iters, level)
            ctx.sync()
            what = "beta %r, %s, %dx%d level %d of %d" % (beta, kind, cols, rows, level, levels)
            assert_bits(to_host(d), want, what, gray, depth, level, levels, lut)
            if residual:
                prev = ob.solve_level(depth, scribble, gray, iters - 1, level, levels - 1, lut)
                res = ctx.level_residual(level)
                assert res == np.float32(np.abs(want - prev).max()), "%s: residual %r" % (what, res)
            if launches is not None:
                assert ctx.level_sweep_ms(level)[1:] == (iters, launches), what
    finally:
        for k in tuning:
            ctx.set_tuning(k, DEFAULT_TUNING[k])
        ctx.close()


# ---- level solves: sweep forms x beta x inputs --------------------------------------------------------------------------------

@pytest.mark.parametrize("beta", wt.BETAS, ids=wt.beta_id)
@pytest.mark.parametrize("form", list(FORMS))
def test_level_solves_in_every_sweep_form(rtdd, form, beta):
    variant, T, tuning = FORMS[form]
    for shape, level, levels in wt.LEVEL_CASES:
        solve_and_compare(rtdd, beta, variant, T, tuning, shape, level, levels)


@pytest.mark.parametrize("beta", wt.BETAS, ids=wt.beta_id)
@pytest.mark.parametrize("build", list(RESIDENT))
def test_resident_kernel_builds(rtdd, build, beta):
    """Level 0 of 2 (depth-gated) and level 1 of 2 (the ungated coarsest level) at each build's shape."""
    for level in (0, 1):
        solve_and_compare(rtdd, beta, 3, 0, {}, RESIDENT[build], level, 2)


# ---- the planner's forms, strip passes, strip frames ---------------------------------------------------------------------------

# level shapes where the pass planner reports form 0 (single CTAs, 128x64 regions), 1 (clusters of two CTAs, 128x128) and
# 2 (single CTAs, 128x32) at ITERS sweeps on 148 SMs.  The flat form is planned only below 2^18 pixels.
PLANNED = {0: (515, 517), 1: (541, 963), 2: (301, 450)}


@pytest.mark.parametrize("beta", [0.45, 8.0], ids=wt.beta_id)
def test_planner_chosen_forms(rtdd, sm_count, beta):
    from realtimedepthdiffusion_b200.api import DepthDiffusion
    hit = set()
    for form, (rows, cols) in PLANNED.items():
        plan, got_form = DepthDiffusion.plan_passes(rows, cols, ITERS, sm_count=sm_count)
        assert got_form == form, (rows, cols, got_form)
        assert (rows * cols >= 1 << 18) == (form != 2)
        solve_and_compare(rtdd, beta, 0, 0, {}, (rows, cols), 0, 2, kinds=("random", "gray-steps"), residual=False, launches=len(plan))
        hit.add(got_form)
    assert hit == {0, 1, 2}


@pytest.mark.parametrize("beta", [0.0, 0.45, 1.0, 8.0, 1e4], ids=wt.beta_id)
@pytest.mark.parametrize("shape,level,levels", [((135, 241), 0, 2), ((270, 480), 0, 1)])
def test_strip_passes_of_the_tolerance_driven_solve(rtdd, beta, shape, level, levels):
    """rtdd_solve_level_converge at tolerance 0 runs every sweep through rtdd_strip_pass (its only caller on one context)."""
    rows, cols = shape
    lut = wt.table(beta)
    ctx = rtdd.DepthDiffusion(rows << level, cols << level, levels, beta=beta)
    try:
        for kind in wt.INPUTS:
            gray, depth, scribble = wt.level_input(kind, rows, cols, level)
            d, s, g = to_dev(depth), to_dev(scribble), to_dev(gray)
            n, _ = ctx.matrix_free_solver_converge(d, s, g, 64, 0.0, level, check_every=16)
            assert n == 64
            want = ob.solve_level(depth, scribble, gray, 64, level, levels - 1, lut)
            assert_bits(to_host(d), want, "beta %r, %s, converge" % (beta, kind), gray, depth, level, levels, lut)
    finally:
        ctx.close()


@pytest.mark.parametrize("beta", [0.0, 1.0, 8.0], ids=wt.beta_id)
def test_two_rank_strip_frame_equals_the_one_gpu_frame(rtdd, beta):
    from realtimedepthdiffusion_b200 import strips
    rows, cols, iters = 512, 640, 150
    bgr, scribble, edited = synth.synth_case(rows, cols, 4242)
    st = ob.FrameState(bgr)
    st.lut = wt.table(beta)
    want_u8 = st.solve(scribble, edited, iters)
    ref = rtdd.DepthDiffusion(rows, cols, beta=beta)
    ref.frame_set_image(bgr)
    one_u8 = ref.frame_solve_host(scribble, edited, iters, np.zeros((rows, cols), np.uint8)).numpy()
    one = ref.frame_plane(ref.PLANE_DEPTH, 0).cpu().numpy()
    ref.close()
    assert np.array_equal(one.view(np.uint32), st.depth[0].view(np.uint32)) and np.array_equal(one_u8, want_u8)
    engines = []
    for r in range(2):
        ctx = rtdd.DepthDiffusion(rows, cols, beta=beta)
        engines.append(strips.GpuStripEngine(ctx, to_dev(bgr, 3), to_dev(scribble), to_dev(edited, 3)))
    try:
        results, exchanges = strips.run_local(engines, iters, halo=8, min_strip_pixels=1)
        torch.cuda.synchronize()
        assert exchanges > 0
        got = np.zeros_like(one)
        got_u8 = np.zeros_like(one_u8)
        for r, (plan, own) in enumerate(results):
            assert plan[0] is not None and plan[0][r] == own
            got[own[0]:own[1]] = to_host(engines[r].depth[0])[own[0]:own[1]]
            got_u8[own[0]:own[1]] = to_host(engines[r].depth_u8)[own[0]:own[1]]
    finally:
        for e in engines:
            e.ctx.close()
    bad = got.view(np.uint32) != one.view(np.uint32)
    assert not bad.any(), "beta %r: %d px differ, rows %s" % (beta, int(bad.sum()), np.unique(np.nonzero(bad)[0])[:8])
    assert np.array_equal(got_u8, one_u8)


# ---- whole frames ---------------------------------------------------------------------------------------------------------------

def oracle_frames(bgr, scribble, edited, beta, n):
    """-> [(8-bit map, [fp32 depth of every level])] of n frames of one FrameState at beta's table."""
    st = ob.FrameState(bgr)
    st.lut = wt.table(beta)
    out = []
    for _ in range(n):
        u8 = st.solve(scribble, edited, MAX_ITERATIONS)
        out.append((u8, list(st.depth)))
    return out


def pinned_map(rows, cols):
    """A pinned host map with rows padded to a multiple of 4 bytes, filled with 0xA5: the last level-0 pass stores into it
    itself (a plane whose pitch is not a multiple of 4 takes the staged copy and the plan without the host map)."""
    pitch = (cols + 3) // 4 * 4
    return torch.full((rows, pitch), 0xA5, dtype=torch.uint8).pin_memory()[:, :cols]


@pytest.mark.parametrize("beta", [0.0, 1.0, 8.0], ids=wt.beta_id)
@pytest.mark.parametrize("rows,cols", [(203, 317), (541, 963)])
def test_whole_frames_into_pinned_maps(rtdd, sm_count, rows, cols, beta):
    """Frame 1 from the annotation plane, frame 2 from the two planes, both stored into a pinned host map by the last level-0
    pass (the host-map plan); every level's fp32 plane and both 8-bit maps against the oracle's frames at beta."""
    bgr, scribble, edited = synth.synth_case(rows, cols, 77 + rows)
    ann = synth.annotation_plane(scribble, edited)
    s, e = ingest(ann, bgr)
    assert np.array_equal(s, scribble) and np.array_equal(e, edited)
    want = oracle_frames(bgr, scribble, edited, beta, 2)
    ctx = rtdd.DepthDiffusion(rows, cols, beta=beta)
    try:
        ctx.frame_set_image(bgr)
        out = pinned_map(rows, cols)
        ctx.frame_solve_host_annotation(pinned_like(ann), MAX_ITERATIONS, out)
        assert_frame(ctx, want[0], [("pinned host map", out.numpy())], "beta %r frame 1 (annotation)" % beta)
        assert_plans_ran(ctx, sm_count, host_map=True)
        out.fill_(0xA5)
        ctx.frame_solve_host(pinned_like(scribble), pinned_like(edited), MAX_ITERATIONS, out)
        assert_frame(ctx, want[1], [("pinned host map", out.numpy())], "beta %r frame 2 (two planes)" % beta)
        assert_plans_ran(ctx, sm_count, host_map=True)
    finally:
        ctx.close()


def test_4k_frame_at_beta_one(rtdd, sm_count):
    """3840x2160: level 0 runs the 128x128 cluster form, here at a table with zeros from w[104]."""
    rows, cols, beta = 2160, 3840, 1.0
    bgr, scribble, edited = synth.synth_case(rows, cols, 1003)
    ann = synth.annotation_plane(scribble, edited)
    want = oracle_frames(bgr, scribble, edited, beta, 1)[0]
    ctx = rtdd.DepthDiffusion(rows, cols, beta=beta)
    try:
        ctx.frame_set_image(bgr)
        out = pinned_map(rows, cols)
        ctx.frame_solve_host_annotation(pinned_like(ann), MAX_ITERATIONS, out)
        assert_frame(ctx, want, [("pinned host map", out.numpy())], "4K at beta 1")
        assert_plans_ran(ctx, sm_count, host_map=True)
    finally:
        ctx.close()


# ---- a table reloaded inside one context ------------------------------------------------------------------------------------------

@pytest.mark.parametrize("shape,variant", [((135, 240), 0), ((301, 450), 0), ((67, 121), 1)])
def test_reloaded_table_reaches_the_cached_level_graph(rtdd, shape, variant):
    """The same call twice is one cached CUDA graph replayed; a table loaded between the two must be the one the replay reads."""
    rows, cols = shape
    gray, depth, scribble = wt.level_input("gray-steps", rows, cols, 0)
    ctx = rtdd.DepthDiffusion(rows, cols, 2, beta=0.4)
    fresh = rtdd.DepthDiffusion(rows, cols, 2, beta=1.0)
    try:
        ctx.set_sweep_variant(variant, 0)
        fresh.set_sweep_variant(variant, 0)
        s, g = to_dev(scribble), to_dev(gray)
        d = to_dev(depth)
        for beta in (0.4, 0.4, 1.0, 1e4, 0.0, 0.4):
            d.copy_(torch.from_numpy(depth))
            ctx.load_weights(beta)
            ctx.matrix_free_solver(d, s, g, ITERS, 0)
            ctx.sync()
            lut = wt.table(beta)
            want = ob.solve_level(depth, scribble, gray, ITERS, 0, 1, lut)
            assert_bits(to_host(d), want, "reloaded beta %r" % beta, gray, depth, 0, 2, lut)
            if beta == 1.0:
                d2 = to_dev(depth)
                fresh.matrix_free_solver(d2, s, g, ITERS, 0)
                fresh.sync()
                assert np.array_equal(to_host(d2).view(np.uint32), want.view(np.uint32))
    finally:
        ctx.close()
        fresh.close()


def test_reloaded_table_reaches_the_cached_frame_graphs(rtdd):
    """frame_solve and frame_solve_incremental from the coarsest level (the full frame), each replayed after a reload: every
    frame equals the oracle's replay of the same sequence of tables, state carried from frame to frame."""
    rows, cols = 541, 963
    bgr, scribble, edited = synth.synth_case(rows, cols, 606)
    st = ob.FrameState(bgr)
    ctx = rtdd.DepthDiffusion(rows, cols, beta=0.4)
    try:
        ctx.frame_set_image(bgr)
        ctx.frame_solve_host(scribble, edited, MAX_ITERATIONS, np.zeros((rows, cols), np.uint8))
        st.solve(scribble, edited, MAX_ITERATIONS)
        steps = [("solve", 0.4), ("solve", 8.0), ("incremental", 8.0), ("incremental", 0.45), ("solve", 0.45), ("incremental", 0.4)]
        for k, (call, beta) in enumerate(steps):
            ctx.load_weights(beta)
            if call == "solve":
                ctx.frame_solve(MAX_ITERATIONS)
            else:
                ctx.frame_solve_incremental(MAX_ITERATIONS, ctx.levels - 1)
            ctx.sync()
            st.lut = wt.table(beta)
            u8 = st.solve(scribble, edited, MAX_ITERATIONS)
            assert_frame(ctx, (u8, list(st.depth)), [], "step %d: %s after loading beta %r" % (k, call, beta))
    finally:
        ctx.close()


def test_reference_named_shim_loads_other_tables():
    """MainLoop over the reference-named functions: GPULoadWeights(1.0) after the loop's own 0.4, one frame equal to FrameState
    at 1.0; then GPULoadWeights(-1.0), which prints its error and keeps the table, and a second frame still at 1.0."""
    from realtimedepthdiffusion_b200 import _native
    rows, cols, iters = 203, 317, 200
    bgr, scribble, edited = synth.synth_case(rows, cols, 808)
    st = ob.FrameState(bgr)
    st.lut = wt.table(1.0)
    loop = MainLoop(_native.shims, bgr)
    try:
        assert loop.levels == st.levels
        loop.api["GPULoadWeights"](1.0)
        for frame in (1, 2):
            u8 = loop.frame(scribble, edited, iters)
            want = st.solve(scribble, edited, iters)
            assert np.array_equal(loop.depth_float.view(np.uint32), st.depth[0].view(np.uint32)), "frame %d" % frame
            assert np.array_equal(u8, want)
            loop.api["GPULoadWeights"](-1.0)
    finally:
        loop.close()


# ---- refusals ------------------------------------------------------------------------------------------------------------------------

BAD_BETAS = [-1.0, -0.4, -1e-30, -1e-45, float("-inf"), float("inf"), float("nan"), -3.4e38]


def test_refused_beta_keeps_the_previous_table(rtdd):
    rows, cols = 67, 121
    gray, depth, scribble = wt.level_input("gray-steps", rows, cols, 0)
    ctx = rtdd.DepthDiffusion(rows, cols, 1, beta=1.0)
    try:
        s, g = to_dev(scribble), to_dev(gray)
        for bad in BAD_BETAS:
            with pytest.raises(rtdd.RtddError, match="rtdd_load_weights"):
                ctx.load_weights(bad)
        for beta in (1.0, -0.0):
            if beta != 1.0:
                ctx.load_weights(beta)                  # -0.0 is accepted: the table of 0.0
                with pytest.raises(rtdd.RtddError):
                    ctx.load_weights(float("nan"))
            d = to_dev(depth)
            ctx.matrix_free_solver(d, s, g, ITERS, 0)
            ctx.sync()
            lut = wt.table(beta)
            assert_bits(to_host(d), ob.solve_level(depth, scribble, gray, ITERS, 0, 0, lut), "after refusals, beta %r" % beta,
                        gray, depth, 0, 1, lut)
    finally:
        ctx.close()


def test_refused_first_load_leaves_the_context_without_a_table(rtdd):
    rows, cols = 64, 64
    ctx = rtdd.DepthDiffusion(rows, cols, 1, beta=None)
    try:
        with pytest.raises(rtdd.RtddError):
            ctx.load_weights(-0.5)
        d, s, g = to_dev(np.zeros((rows, cols), np.float32)), to_dev(np.zeros((rows, cols), np.uint8)), to_dev(np.zeros((rows, cols), np.uint8))
        with pytest.raises(rtdd.RtddError, match="rtdd_load_weights not called"):
            ctx.matrix_free_solver(d, s, g, 3, 0)
        ctx.frame_set_image(np.zeros((rows, cols, 3), np.uint8))
        with pytest.raises(rtdd.RtddError):
            ctx.frame_solve(10)
        ctx.load_weights(0.4)
        ctx.matrix_free_solver(d, s, g, 3, 0)
        ctx.sync()
    finally:
        ctx.close()


def test_multi_gpu_create_refuses_bad_beta_and_leaves_no_handle(rtdd):
    lib = rtdd._native.lib
    devices = C.cast((C.c_int * 1)(torch.cuda.current_device()), C.c_void_p)
    for bad in (-1.0, float("nan"), float("inf")):
        h = C.c_void_p(12345)
        rc = lib.rtdd_mgpu_create(devices, 1, 64, 96, 0, bad, 0, 0, 0, C.byref(h))
        assert rc != 0 and h.value is None, (bad, rc, h.value)
    h = C.c_void_p()
    assert lib.rtdd_mgpu_create(devices, 1, 64, 96, 0, 0.4, 0, 0, 0, C.byref(h)) == 0 and h.value
    assert lib.rtdd_mgpu_destroy(h) == 0
