"""GPU tests of the refocus extension (rtdd_refocus / rtdd_frame_refocus, no reference counterpart): byte-identical to the CPU
reference (tests/refocus_reference.py), identical to rtdd_defocus at the parity point f = 0, w = 0, A = K, the frame form's cached summed-area
table and its focus read on the device, and the argument errors."""
import ctypes as C

import numpy as np
import pytest
import torch

from oracle import binding as ob
from realtimedepthdiffusion_b200 import synth
from tests import refocus_reference as ref
from tests.harness import pitch, ptr, to_dev, to_host

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def rtdd():
    import realtimedepthdiffusion_b200 as pkg
    return pkg


def refocus_inputs(rows, cols, seed):
    """Image and a depth plane over [-40, 300] with NaN: the clamp is part of the definition."""
    rng = np.random.default_rng(seed)
    bgr = synth.synth_image(rows, cols, seed)
    yy, xx = np.mgrid[0:rows, 0:cols]
    depth = (130.0 + 170.0 * np.sin(xx / 41.0) * np.cos(yy / 29.0)).astype(np.float32)
    depth += rng.uniform(-0.5, 0.5, depth.shape).astype(np.float32)
    depth[rng.random((rows, cols)) < 0.01] = np.nan
    depth.flat[: min(depth.size, 5)] = np.array([np.nan, -7.0, 255.0, 262.5, 37.5], np.float32)[: min(depth.size, 5)]
    return bgr, depth


def misaligned(a, channels=1):
    """Device copy whose rows start one element past an aligned address, with an odd pitch: the scalar kernel path."""
    a = np.ascontiguousarray(a)
    flat = torch.from_numpy(a.reshape(a.shape[0], -1))
    base = torch.zeros((a.shape[0], flat.shape[1] + 3), dtype=flat.dtype, device="cuda")
    view = base[:, 1:1 + flat.shape[1]]
    view.copy_(flat)
    return view


def clamp_depth(d):
    return float(np.fmin(np.fmax(np.float32(d), np.float32(0)), np.float32(255)))


@pytest.mark.parametrize("rows,cols", [(1, 1), (5, 3), (67, 121), (203, 317), (270, 480), (1080, 1920)])
def test_refocus_equals_cpu_reference(rtdd, rows, cols):
    bgr, depth = refocus_inputs(rows, cols, rows + cols)
    K = ob.defocus_kernel_size(rows, cols)
    ctx = rtdd.DepthDiffusion(rows, cols, 1)
    planes = {"aligned": (to_dev(bgr, 3), to_dev(depth), to_dev(np.zeros_like(bgr), 3)),
              "unaligned": (misaligned(bgr, 3), misaligned(depth), misaligned(np.zeros_like(bgr), 3))}
    for f in (0.0, 37.5, 128.0, 255.0):
        for w in (0.0, 20.0):
            for a in (0, 1, 2, K, 300):
                want = ref.refocus(bgr, depth, f, w, a)
                for kind, (o, d, out) in planes.items():
                    out.fill_(0)
                    ctx.refocus(o, d, out, f, w, a)
                    ctx.sync()
                    got = to_host(out, 3)
                    assert np.array_equal(got, want), (kind, f, w, a, int((got != want).any(-1).sum()))
    ctx.close()


@pytest.mark.parametrize("aperture", [1024, 4096])
def test_refocus_4k_large_apertures_take_the_integer_mean(rtdd, aperture):
    rows, cols = 2160, 3840
    bgr, depth = refocus_inputs(rows, cols, aperture)
    ctx = rtdd.DepthDiffusion(rows, cols, 1)
    o, d, out = to_dev(bgr, 3), to_dev(depth), to_dev(np.zeros_like(bgr), 3)
    for f, w in ((0.0, 0.0), (128.0, 20.0), (255.0, 5.0)):
        dc = np.fmin(np.fmax(depth, np.float32(0)), np.float32(255))
        e = np.fmax(np.abs(dc - np.float32(f)) - np.float32(w), np.float32(0))
        h = np.trunc((np.float32(aperture) * e).astype(np.float64) / 255.0).astype(np.int64) // 2
        assert (4 * h * h > 65793).mean() > 0.01           # windows beyond the fp32-exact range
        ctx.refocus(o, d, out, f, w, aperture)
        ctx.sync()
        assert np.array_equal(to_host(out, 3), ref.refocus(bgr, depth, f, w, aperture)), (f, w)
    ctx.close()


@pytest.mark.parametrize("rows,cols", [(203, 317), (1080, 1920), (2160, 3840)])
def test_parity_point_equals_defocus_on_a_solved_depth(rtdd, rows, cols):
    bgr, scribble, edited = synth.synth_case(rows, cols, 21)
    ctx = rtdd.DepthDiffusion(rows, cols)
    ctx.frame_set_image(bgr)
    ctx.frame_solve_host(scribble, edited, 1000, None)
    d = ctx.frame_plane(ctx.PLANE_DEPTH, 0)
    o = to_dev(bgr, 3)
    want, got = to_dev(np.zeros_like(bgr), 3), to_dev(np.zeros_like(bgr), 3)
    ctx.simulate_defocus(o, d, want)
    ctx.refocus(o, d, got, 0.0, 0.0)
    ctx.sync()
    w = to_host(want, 3)
    assert np.array_equal(to_host(got, 3), w)
    assert not np.array_equal(w, bgr)
    ctx.close()


def stand_alone(rtdd, bgr, depth, f, w, a):
    rows, cols = depth.shape
    helper = rtdd.DepthDiffusion(rows, cols, 1)
    out = to_dev(np.zeros_like(bgr), 3)
    helper.refocus(to_dev(bgr, 3), to_dev(depth), out, f, w, a)
    helper.sync()
    helper.close()
    return to_host(out, 3)


@pytest.mark.parametrize("rows,cols,iters", [(203, 317, 60), (360, 641, 40)])
def test_frame_refocus_with_cached_summed_area_table(rtdd, rows, cols, iters):
    ctx = rtdd.DepthDiffusion(rows, cols)
    other_bgr, other_depth = refocus_inputs(rows, cols, 5)
    for seed in (77, 78):                                        # second round: a NEW image in the same context
        bgr, scribble, edited = synth.synth_case(rows, cols, seed)
        ctx.frame_set_image(bgr)
        ctx.frame_solve_host(scribble, edited, iters, None)
        depth = ctx.frame_plane(ctx.PLANE_DEPTH, 0).cpu().numpy()
        ys, xs = np.nonzero(scribble == 255)
        points = [(int(xs[0]), int(ys[0])), (0, 0), (cols - 1, rows - 1), (cols // 2, rows // 3)]
        out = to_dev(np.zeros_like(bgr), 3)
        for i, (x, y) in enumerate(points):
            w, a = (0.0, None) if i % 2 == 0 else (12.0, 64)
            n0 = ctx.launch_count
            ctx.frame_refocus(out, focus_point=(x, y), depth_of_field=w, aperture=a)
            ctx.sync()
            assert ctx.launch_count - n0 == (5 if i == 0 else 1)   # the table is built once per image
            assert np.array_equal(to_host(out, 3), stand_alone(rtdd, bgr, depth, clamp_depth(depth[y, x]), w, -1 if a is None else a)), (x, y)
        ctx.frame_refocus(out, focus_depth=200.0, depth_of_field=3.0, aperture=90)
        ctx.sync()
        assert np.array_equal(to_host(out, 3), stand_alone(rtdd, bgr, depth, 200.0, 3.0, 90))
        # frame_effects shares the cached table: defocus alone is one launch
        defocus = to_dev(np.zeros_like(bgr), 3)
        n0 = ctx.launch_count
        ctx.frame_effects(None, None, defocus)
        ctx.sync()
        assert ctx.launch_count - n0 == 1
        assert np.array_equal(to_host(defocus, 3), ob.defocus(bgr, depth))
        # a stand-alone refocus or defocus of ANOTHER image through the same context overwrites the scratch: rebuilt, still exact
        for borrow in ("refocus", "defocus"):
            scratch_user = to_dev(np.zeros_like(other_bgr), 3)
            if borrow == "refocus":
                ctx.refocus(to_dev(other_bgr, 3), to_dev(other_depth), scratch_user, 40.0, 5.0, 150)
                want_other = ref.refocus(other_bgr, other_depth, 40.0, 5.0, 150)
            else:
                ctx.simulate_defocus(to_dev(other_bgr, 3), to_dev(other_depth), scratch_user)
                want_other = ob.defocus(other_bgr, other_depth)
            x, y = points[0]
            n0 = ctx.launch_count
            ctx.frame_refocus(out, focus_point=(x, y), depth_of_field=0.0)
            ctx.sync()
            assert ctx.launch_count - n0 == 5, borrow
            assert np.array_equal(to_host(out, 3), stand_alone(rtdd, bgr, depth, clamp_depth(depth[y, x]), 0.0, -1)), borrow
            assert np.array_equal(to_host(scratch_user, 3), want_other), borrow
    ctx.close()


def test_captured_frame_refocus_reads_the_focus_on_the_device(rtdd):
    """A graph captured from frame_refocus(focus_point=...) on a torch stream, replayed after a new solve with other strokes,
    refocuses at the NEW depth under the point: the focus is read on the GPU and the call does no host work mid-stream."""
    rows, cols, iters = 203, 317, 120
    bgr, scribble, edited = synth.synth_case(rows, cols, 31)
    ctx = rtdd.DepthDiffusion(rows, cols)
    s = torch.cuda.Stream()
    ctx.set_stream(s)
    ctx.frame_set_image(bgr)
    ctx.frame_solve_host(scribble, edited, iters, None)
    x, y, w, a = 150, 90, 4.0, 120
    out = to_dev(np.zeros_like(bgr), 3)
    ctx.frame_refocus(out, focus_point=(x, y), depth_of_field=w, aperture=a)          # warm-up: builds the table
    ctx.sync()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=s):
        ctx.frame_refocus(out, focus_point=(x, y), depth_of_field=w, aperture=a)
    depth1 = ctx.frame_plane(ctx.PLANE_DEPTH, 0).cpu().numpy()
    colour = 17 if depth1[y, x] > 128 else 240
    ctx.frame_paint(x, y, colour, 6)                             # a stroke over the point: its depth becomes `colour`
    ctx.frame_paint(30, 40, 255 - colour, 9)
    ctx.frame_solve(iters)
    ctx.sync()
    depth2 = ctx.frame_plane(ctx.PLANE_DEPTH, 0).cpu().numpy()
    assert depth2[y, x] == colour and abs(float(depth1[y, x]) - colour) > 10.0
    out.fill_(0)
    torch.cuda.synchronize()
    with torch.cuda.stream(s):
        g.replay()
    s.synchronize()
    got = to_host(out, 3)
    assert np.array_equal(got, stand_alone(rtdd, bgr, depth2, float(colour), w, a))
    assert not np.array_equal(got, stand_alone(rtdd, bgr, depth2, clamp_depth(depth1[y, x]), w, a))
    del g
    ctx.set_stream(None)
    ctx.close()


def test_argument_errors_leave_the_context_usable(rtdd):
    from realtimedepthdiffusion_b200 import _native
    lib = _native.lib
    rows, cols = 67, 121
    bgr, depth = refocus_inputs(rows, cols, 8)
    ctx = rtdd.DepthDiffusion(rows, cols)
    h = ctx._h
    out = to_dev(np.zeros_like(bgr), 3)
    assert lib.rtdd_frame_refocus(h, ptr(out), pitch(out), -1, -1, 10.0, 0.0, -1) == -2          # before frame_set_image
    ctx.frame_set_image(bgr)
    o, d = to_dev(bgr, 3), to_dev(depth)
    po, pd, pr = pitch(o), pitch(d), pitch(out)
    nan, inf = float("nan"), float("inf")
    bad_stand_alone = [
        (None, po, d, pd, out, pr, rows, cols, 10.0, 0.0, -1),
        (o, po, None, pd, out, pr, rows, cols, 10.0, 0.0, -1),
        (o, po, d, pd, None, pr, rows, cols, 10.0, 0.0, -1),
        (o, cols * 3 - 1, d, pd, out, pr, rows, cols, 10.0, 0.0, -1),
        (o, po, d, cols * 4 - 4, out, pr, rows, cols, 10.0, 0.0, -1),
        (o, po, d, pd, out, cols * 3 - 1, rows, cols, 10.0, 0.0, -1),
        (o, po, d, pd, out, pr, -1, cols, 10.0, 0.0, -1),
        (o, po, d, pd, out, pr, rows, cols, nan, 0.0, -1),
        (o, po, d, pd, out, pr, rows, cols, -0.5, 0.0, -1),
        (o, po, d, pd, out, pr, rows, cols, 255.5, 0.0, -1),
        (o, po, d, pd, out, pr, rows, cols, 10.0, -1.0, -1),
        (o, po, d, pd, out, pr, rows, cols, 10.0, nan, -1),
        (o, po, d, pd, out, pr, rows, cols, 10.0, inf, -1),
        (o, po, d, pd, out, pr, rows, cols, 10.0, 0.0, 4097),
    ]
    bad_frame = [
        (None, pr, -1, -1, 10.0, 0.0, -1),
        (out, cols * 3 - 1, -1, -1, 10.0, 0.0, -1),
        (out, pr, -1, -1, nan, 0.0, -1),
        (out, pr, -1, -1, 256.0, 0.0, -1),
        (out, pr, cols, 0, 0.0, 0.0, -1),
        (out, pr, 0, rows, 0.0, 0.0, -1),
        (out, pr, -1, 5, 10.0, 0.0, -1),
        (out, pr, 5, -1, 10.0, 0.0, -1),
        (out, pr, -2, -2, 10.0, 0.0, -1),
        (out, pr, 5, 5, 0.0, -0.25, -1),
        (out, pr, 5, 5, 0.0, nan, -1),
        (out, pr, 5, 5, 0.0, 0.0, 4097),
    ]

    def p(t):
        return ptr(t) if t is not None else C.c_void_p(0)

    n0 = ctx.launch_count
    for args in bad_stand_alone:
        oo, opp, dd, dp, uu, up, r, c, f, w, a = args
        assert lib.rtdd_refocus(h, p(oo), opp, p(dd), dp, p(uu), up, r, c, f, w, a) == -1, args[6:]
    for args in bad_frame:
        uu, up, fx, fy, f, w, a = args
        assert lib.rtdd_frame_refocus(h, p(uu), up, fx, fy, f, w, a) == -1, args[1:]
    assert ctx.launch_count == n0
    with pytest.raises(ValueError):
        ctx.frame_refocus(out)
    with pytest.raises(rtdd.RtddError):
        ctx.frame_refocus(out, focus_point=(-1, -1))
    # still exact afterwards, both forms
    ctx.refocus(o, d, out, 37.5, 20.0, 300)
    ctx.sync()
    assert np.array_equal(to_host(out, 3), ref.refocus(bgr, depth, 37.5, 20.0, 300))
    ctx.frame_solve_host(*synth.synth_case(rows, cols, 8)[1:], 60, None)
    fd = ctx.frame_plane(ctx.PLANE_DEPTH, 0).cpu().numpy()
    ctx.frame_refocus(out, focus_point=(cols - 1, 0), depth_of_field=2.0, aperture=4096)
    ctx.sync()
    assert np.array_equal(to_host(out, 3), ref.refocus(bgr, fd, clamp_depth(fd[0, cols - 1]), 2.0, 4096))
    ctx.close()
