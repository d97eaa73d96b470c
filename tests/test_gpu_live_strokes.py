"""The live loop's re-solves after a brush stroke, rtdd_frame_solve_incremental and rtdd_frame_solve_band, bit for bit against
their CPU restatement (tests/live_reference.py).  After every call every level's fp32 depth plane and the 8-bit map must
equal the restated state's; a failure names the first differing level and its rows.

test_gpu_parity.py's two loose tests of these paths stay: they bound how far the band frame is from the parity frame, which is
another claim."""
import numpy as np
import pytest
import torch

from oracle import binding as ob
from realtimedepthdiffusion_b200 import synth
from tests import live_reference as lr
from tests.harness import to_dev, to_host

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def rtdd():
    import realtimedepthdiffusion_b200 as pkg
    return pkg


def device_planes(ctx):
    """Every level's fp32 depth plane and the 8-bit map, as device tensors."""
    return [ctx.frame_plane(ctx.PLANE_DEPTH, l) for l in range(ctx.levels)], ctx.frame_plane(ctx.PLANE_DEPTH_U8, 0)


def rows_report(got, want):
    rows = np.nonzero((got != want).reshape(got.shape[0], -1).any(axis=1))[0]
    return "%d rows differ, first %d, last %d" % (rows.size, rows[0], rows[-1])


def assert_state(ctx, st, what):
    """The context's planes equal the restated state; returns them (device tensors) for later comparisons."""
    depth, u8 = device_planes(ctx)
    for l in range(st.levels):
        got = depth[l].cpu().numpy().view(np.uint32)
        want = st.depth[l].view(np.uint32)
        assert got.shape == want.shape
        if not np.array_equal(got, want):
            g, w = got.view(np.float32), want.view(np.float32)
            pytest.fail("%s: level %d fp32 depth: %s, max |diff| %g" % (what, l, rows_report(got, want), np.nanmax(np.abs(g - w))))
    got = u8.cpu().numpy()
    want = ob.quantise_u8(st.depth[0])
    if not np.array_equal(got, want):
        pytest.fail("%s: 8-bit map: %s" % (what, rows_report(got, want)))
    return depth, u8


def assert_same_planes(ctx, planes, what):
    """The context's planes equal planes that matched the restatement earlier."""
    depth, u8 = device_planes(ctx)
    for l, (a, b) in enumerate(zip(depth, planes[0])):
        if not torch.equal(a.view(torch.int32), b.view(torch.int32)):
            pytest.fail("%s: level %d fp32 depth: %s" % (what, l, rows_report(a.cpu().numpy(), b.cpu().numpy())))
    if not torch.equal(u8, planes[1]):
        pytest.fail("%s: 8-bit map: %s" % (what, rows_report(u8.cpu().numpy(), planes[1].cpu().numpy())))


def zero_sweep_iterations(levels):
    """A frame's max_iterations for which level 0 runs 0 sweeps, level 1 one, level 2 three, ... (2^l - 1)."""
    return (1 << (levels - 1)) - 1


# ---- incremental ----------------------------------------------------------------------------------------------------


@pytest.mark.parametrize("rows,cols", [(203, 317), (540, 960), (1080, 1920), (2160, 3840), (1081, 1919)])
def test_incremental_resolves_replay_their_graphs_exactly(rtdd, rows, cols):
    """One context: a frame, then strokes painted on the device, each re-solved from a start level cycling through L-1, 0, 1,
    L-2 (one cached frame graph per start level and iteration count) with a plain frame in between, at 1000 iterations and at a
    count that gives the finest levels 0, 1, 3 ... sweeps; then from levels 0 and 1 at 1000 iterations again, replaying those
    graphs after others ran (the plain frames replay the level L-1 graph throughout).  All of it with fused_prolong 0, checked
    against the restatement; again with fused_prolong 1, against the planes of the first run."""
    bgr, scribble, edited, st = lr.first_frame(rows, cols, 700 + rows)
    L = st.levels
    small = zero_sweep_iterations(L)
    starts = [L - 1, 0, 1, L - 2]
    schedule = [(c, 1000) for c in starts] + [(c, small) for c in starts] + [(0, 1000), (1, 1000)]
    events = synth.brush_events(rows, cols, 701 + rows, len(schedule), 3)
    # (what, brush events painted first, start level, max_iterations, through rtdd_frame_solve)
    steps = [("first frame", [], L - 1, 1000, False)]
    for k, (c, iters) in enumerate(schedule):
        if k:
            steps.append(("frame of %d iterations after stroke %d" % (iters, k - 1), [], L - 1, iters, True))
        steps.append(("stroke %d, incremental from level %d, %d iterations" % (k, c, iters), events[3 * k:3 * k + 3], c, iters, False))
    want = []
    ctx = rtdd.DepthDiffusion(rows, cols)
    assert ctx.levels == L
    try:
        for fused in (0, 1):
            ctx.set_tuning("fused_prolong", fused)
            ctx.frame_set_image(bgr)
            ctx.frame_solve_host(scribble, edited, 1000)
            for i, (what, strokes, c, iters, whole_frame) in enumerate(steps):
                if i:
                    for e in strokes:
                        ctx.frame_paint(*e)
                    if whole_frame:
                        ctx.frame_solve(iters)
                    else:
                        ctx.frame_solve_incremental(iters, c)
                if fused == 0:
                    if i:
                        lr.paint(st, strokes)
                        lr.solve_incremental(st, iters, c)
                    want.append(assert_state(ctx, st, what))
                else:
                    assert_same_planes(ctx, want[i], what + ", fused_prolong 1")
    finally:
        ctx.set_tuning("fused_prolong", 0)
        ctx.close()


# ---- band -----------------------------------------------------------------------------------------------------------


@pytest.mark.parametrize("rows,cols", [(1080, 1920), (2160, 3840), (2161, 3839)])
def test_band_resolves_match_the_restatement(rtdd, rows, cols):
    """One context: a frame, then four band re-solves in a row -- a stroke in the middle (dilation 96), one touching row 0
    (dilation 24, level 0 given 6 sweeps: one partial pass), one touching the last row (dilation 96, level 0 given 0 sweeps)
    and a one-row edit with dilation 1 (a 3-row band, thinner than the 8-sweep passes) -- then the effects of the band frame's
    depth, a parity frame continuing from the band state, another band and a parity frame of a new annotation."""
    bgr, scribble, edited, st = lr.first_frame(rows, cols, 800 + rows)
    L = st.levels
    banded_levels = [l for l in (1, 0) if st.sizes[l][0] * st.sizes[l][1] >= lr.WHOLE_LEVEL_PIXELS]
    radius = int(min(rows, cols) * 0.02)
    partial, zero = 6 << (L - 1), zero_sweep_iterations(L)
    # (what, brush events, dilation, max_iterations, where every banded level's band lies: between two frozen rows, or at an edge)
    bands = [
        ("stroke in the middle, dilation 96", lr.diagonal_stroke(cols // 3, rows // 2, 128, radius), 96, 1000, "inner"),
        ("stroke touching row 0, dilation 24, %d iterations" % partial, lr.diagonal_stroke(cols // 2, 0, 64, radius), 24, partial, "top"),
        ("stroke touching the last row, dilation 96, %d iterations" % zero, lr.diagonal_stroke(cols // 4, rows - 1, 192, radius, 1), 96, zero, "bottom"),
        ("one-row edit, dilation 1", [(cols // 2, rows // 2 + 1, 0, 1)], 1, 1000, "inner"),
    ]
    ctx = rtdd.DepthDiffusion(rows, cols)
    try:
        assert ctx.levels == L
        ctx.frame_set_image(bgr)
        ctx.frame_solve_host(scribble, edited, 1000)
        assert_state(ctx, st, "first frame")

        def band(what, strokes, dilation, iters, where):
            for e in strokes:
                ctx.frame_paint(*e)
            r0, r1 = lr.paint(st, strokes)
            ctx.frame_solve_band(iters, r0, r1, dilation)
            _, banded = lr.solve_band(st, iters, r0, r1, dilation)
            assert [b[0] for b in banded] == banded_levels, (what, banded)
            for l, b0, b1 in banded:
                assert {"inner": 0 < b0 and b1 < st.sizes[l][0], "top": b0 == 0, "bottom": b1 == st.sizes[l][0]}[where], (what, banded)
            if dilation == 1:
                assert banded[-1][2] - banded[-1][1] == 3, (what, banded)
            assert_state(ctx, st, "%s: rows [%d, %d), banded (level, b0, b1) %s" % (what, r0, r1, banded))

        for b in bands:
            band(*b)
        # the effects read the band frame's depth
        desat, defocus = to_dev(np.zeros_like(bgr), 3), to_dev(np.zeros_like(bgr), 3)
        ctx.frame_effects(desat, None, defocus)
        ctx.sync()
        assert np.array_equal(to_host(desat, 3), ob.desaturate(bgr, st.gray[0], st.depth[0])), "desaturation after the band solves"
        assert np.array_equal(to_host(defocus, 3), ob.defocus(bgr, st.depth[0])), "defocus after the band solves"
        # parity frames after band solves: the strip state those leave in the levels must not reach them
        ctx.frame_solve(1000)
        lr.solve_incremental(st, 1000, L - 1)
        assert_state(ctx, st, "frame after the band solves")
        band("stroke after a frame, dilation 24", lr.diagonal_stroke(cols // 2, rows // 3, 254, radius), 24, 1000, "inner")
        scribble2, edited2 = synth.paint_events(bgr, synth.brush_events(rows, cols, 802 + rows, 2, 4), scribble.copy(), edited.copy())
        ctx.frame_solve_host(scribble2, edited2, 1000)
        st.solve(scribble2, edited2, 1000)
        assert_state(ctx, st, "host frame after a band solve")
    finally:
        ctx.close()


# ---- refused calls --------------------------------------------------------------------------------------------------


def test_refused_calls_leave_the_context_usable(rtdd):
    """Each refused call raises RtddError and changes nothing: the calls after it are still exact."""
    rows, cols = 1024, 1100          # level 0 has >= 2^20 pixels: it is banded
    bgr, scribble, edited, st = lr.first_frame(rows, cols, 900)
    L = st.levels
    ctx = rtdd.DepthDiffusion(rows, cols)
    try:
        with pytest.raises(rtdd.RtddError):
            ctx.frame_solve_band(1000, 0, 10, 8)               # no image yet
        with pytest.raises(rtdd.RtddError):
            ctx.frame_solve_incremental(1000, 0)
        ctx.frame_set_image(bgr)
        ctx.frame_solve_host(scribble, edited, 1000)
        assert_state(ctx, st, "first frame after refused calls")
        strokes = synth.brush_events(rows, cols, 901, 1, 3)
        for e in strokes:
            ctx.frame_paint(*e)
        r0, r1 = lr.paint(st, strokes)
        for args in ((1000, -1, r1, 8), (1000, r0, rows + 1, 8), (1000, r0, r0, 8), (1000, r1, r0, 8), (1000, r0, r1, 0), (-1, r0, r1, 8)):
            with pytest.raises(rtdd.RtddError):
                ctx.frame_solve_band(*args)
        for c in (-1, L):
            with pytest.raises(rtdd.RtddError):
                ctx.frame_solve_incremental(1000, c)
        ctx.frame_solve_band(1000, r0, r1, 8)
        _, banded = lr.solve_band(st, 1000, r0, r1, 8)
        assert [b[0] for b in banded] == [0]
        assert_state(ctx, st, "band solve after refused calls")
        strokes = synth.brush_events(rows, cols, 902, 1, 3)
        for e in strokes:
            ctx.frame_paint(*e)
        lr.paint(st, strokes)
        for c in (-1, L):
            with pytest.raises(rtdd.RtddError):
                ctx.frame_solve_incremental(1000, c)
        ctx.frame_solve_incremental(1000, 1)
        lr.solve_incremental(st, 1000, 1)
        assert_state(ctx, st, "incremental solve after refused calls")
    finally:
        ctx.close()
