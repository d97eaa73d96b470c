"""GPU tests of the stereo extension (rtdd_stereo / rtdd_frame_stereo, no reference counterpart): byte-identical to the CPU
reference (tests/stereo_reference.py) from 1x1 to 4K and at the widest row, for every subset of the three outputs and side by
side in one buffer; the frame form with its convergence depth read on the device, inside a captured graph too; the cached
summed-area table of the other frame effects left valid; and the argument errors."""
import ctypes as C
import itertools

import numpy as np
import pytest
import torch

from oracle import binding as ob
from realtimedepthdiffusion_b200 import synth
from tests import stereo_reference as ref
from tests.harness import pitch, ptr, to_dev, to_host

pytestmark = pytest.mark.gpu

NAMES = ("left", "right", "anaglyph")


@pytest.fixture(scope="module")
def rtdd():
    import realtimedepthdiffusion_b200 as pkg
    return pkg


def stereo_inputs(rows, cols, seed):
    """Image and a smooth depth plane over [-40, 300] with NaN and -0: the clamp is part of the definition, and the smooth
    parts give the views real occlusions and disocclusions."""
    rng = np.random.default_rng(seed)
    bgr = synth.synth_image(rows, cols, seed)
    yy, xx = np.mgrid[0:rows, 0:cols]
    depth = (130.0 + 170.0 * np.sin(xx / 41.0) * np.cos(yy / 29.0)).astype(np.float32)
    depth += rng.uniform(-0.5, 0.5, depth.shape).astype(np.float32)
    depth[rng.random((rows, cols)) < 0.01] = np.nan
    depth[rng.random((rows, cols)) < 0.01] = np.float32(-0.0)
    depth.flat[: min(depth.size, 6)] = np.array([np.nan, -7.0, 255.0, 262.5, 37.5, -0.0], np.float32)[: min(depth.size, 6)]
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


def first_difference(got, want):
    bad = (got != want).any(-1)
    if not bad.any():
        return "equal"
    ys, xs = np.nonzero(bad)
    return "%d px differ, first (y %d, x %d): got %s want %s" % (bad.sum(), ys[0], xs[0], got[ys[0], xs[0]], want[ys[0], xs[0]])


def check_views(outs, want, what):
    for name, o, w in zip(NAMES, outs, want):
        if o is not None:
            got = to_host(o, 3)
            assert np.array_equal(got, w), (what, name, first_difference(got, w))


PARAMS_FULL = [(c, D) for D in (0, 1, 2, 57, 1024) for c in (0.0, 37.5, 128.0, 255.0)]
PARAMS_LARGE = [(0.0, 57), (37.5, 1024), (128.0, 2), (255.0, 57), (128.0, 1), (37.5, 0)]


@pytest.mark.parametrize("rows,cols", [(1, 1), (5, 3), (67, 121), (203, 317), (270, 480), (4, 16384), (1080, 1920), (2160, 3840)])
def test_stereo_equals_cpu_reference(rtdd, rows, cols):
    bgr, depth = stereo_inputs(rows, cols, rows + cols)
    ctx = rtdd.DepthDiffusion(rows, cols, 1)
    zeros = np.zeros_like(bgr)
    planes = {"aligned": (to_dev(bgr, 3), to_dev(depth), [to_dev(zeros, 3) for _ in NAMES]),
              "unaligned": (misaligned(bgr, 3), misaligned(depth), [misaligned(zeros, 3) for _ in NAMES])}
    params = PARAMS_FULL if rows * cols <= 270 * 480 or rows == 4 else PARAMS_LARGE
    for c, D in params:
        want = ref.stereo(bgr, depth, c, D)
        for kind, (o, d, outs) in planes.items():
            for out in outs:
                out.fill_(0)
            n0 = ctx.launch_count
            ctx.stereo(o, d, *outs, convergence_depth=c, max_disparity=D)
            ctx.sync()
            assert ctx.launch_count - n0 == (1 if rows * cols else 0)
            check_views(outs, want, (kind, c, D))
    ctx.close()


@pytest.mark.parametrize("rows,cols", [(67, 121), (203, 317)])
def test_every_subset_of_outputs_gives_the_same_bytes(rtdd, rows, cols):
    bgr, depth = stereo_inputs(rows, cols, 5)
    ctx = rtdd.DepthDiffusion(rows, cols, 1)
    sentinel = np.full_like(bgr, 77)
    for kind, dev in (("aligned", to_dev), ("unaligned", misaligned)):
        o, d = dev(bgr, 3), dev(depth)
        for c, D in ((37.5, 57), (255.0, 1024), (128.0, 1)):
            want = ref.stereo(bgr, depth, c, D)
            for k in (1, 2, 3):
                for subset in itertools.combinations(range(3), k):
                    outs = [dev(sentinel, 3) for _ in NAMES]
                    args = [outs[i] if i in subset else None for i in range(3)]
                    n0 = ctx.launch_count
                    ctx.stereo(o, d, *args, convergence_depth=c, max_disparity=D)
                    ctx.sync()
                    assert ctx.launch_count - n0 == 1
                    for i in range(3):
                        got = to_host(outs[i], 3)
                        if i in subset:
                            assert np.array_equal(got, want[i]), (kind, c, D, subset, NAMES[i], first_difference(got, want[i]))
                        else:
                            assert np.array_equal(got, sentinel), (kind, c, D, subset, NAMES[i], "written although not requested")
    ctx.close()


@pytest.mark.parametrize("rows,cols", [(67, 121), (31, 1001)])
def test_side_by_side_into_one_buffer(rtdd, rows, cols):
    """left = buf, right = buf + 3 cols, pitch 6 cols: at an odd cols the right half starts misaligned."""
    assert cols % 4 != 0
    bgr, depth = stereo_inputs(rows, cols, 9)
    ctx = rtdd.DepthDiffusion(rows, cols, 1)
    o, d = to_dev(bgr, 3), to_dev(depth)
    buf = torch.zeros((rows, 6 * cols), dtype=torch.uint8, device="cuda")
    ana = to_dev(np.zeros_like(bgr), 3)
    for c, D in ((0.0, 57), (200.0, 1024), (37.5, 2)):
        buf.fill_(0)
        ctx.stereo(o, d, buf[:, :3 * cols], buf[:, 3 * cols:], ana, convergence_depth=c, max_disparity=D)
        ctx.sync()
        want = ref.stereo(bgr, depth, c, D)
        got = buf.cpu().numpy().reshape(rows, 2 * cols, 3)
        assert np.array_equal(got[:, :cols], want[0]), (c, D, first_difference(got[:, :cols], want[0]))
        assert np.array_equal(got[:, cols:], want[1]), (c, D, first_difference(got[:, cols:], want[1]))
        assert np.array_equal(to_host(ana, 3), want[2]), (c, D)
    ctx.close()


@pytest.mark.parametrize("rows,cols,iters", [(203, 317, 60), (360, 641, 40)])
def test_frame_stereo_on_solved_depths(rtdd, rows, cols, iters):
    ctx = rtdd.DepthDiffusion(rows, cols)
    for seed in (77, 78):                                        # second round: a NEW image in the same context
        bgr, scribble, edited = synth.synth_case(rows, cols, seed)
        ctx.frame_set_image(bgr)
        ctx.frame_solve_host(scribble, edited, iters, None)
        depth = ctx.frame_plane(ctx.PLANE_DEPTH, 0).cpu().numpy()
        # the defocus table is built once for this image; stereo calls in between must leave it valid
        defocus = to_dev(np.zeros_like(bgr), 3)
        ctx.frame_effects(None, None, defocus)
        ctx.sync()
        defocus_bytes = to_host(defocus, 3)
        assert np.array_equal(defocus_bytes, ob.defocus(bgr, depth))
        ys, xs = np.nonzero(scribble == 255)
        points = [(int(xs[0]), int(ys[0])), (0, 0), (cols - 1, rows - 1), (cols - 1, 0), (0, rows - 1), (cols // 2, rows // 3)]
        outs = [to_dev(np.zeros_like(bgr), 3) for _ in NAMES]
        for i, (x, y) in enumerate(points):
            D = (57, 1024, 2)[i % 3]
            n0 = ctx.launch_count
            ctx.frame_stereo(*outs, convergence_point=(x, y), max_disparity=D)
            ctx.sync()
            assert ctx.launch_count - n0 == 1
            check_views(outs, ref.stereo(bgr, depth, clamp_depth(depth[y, x]), D), (seed, x, y, D))
        for c, D in ((200.0, 57), (0.0, 1), (37.5, 1024)):
            n0 = ctx.launch_count
            ctx.frame_stereo(*outs, convergence_depth=c, max_disparity=D)
            ctx.sync()
            assert ctx.launch_count - n0 == 1
            check_views(outs, ref.stereo(bgr, depth, c, D), (seed, c, D))
        ctx.frame_stereo(None, outs[1], None, convergence_depth=90.0, max_disparity=57)
        ctx.sync()
        check_views([None, outs[1], None], ref.stereo(bgr, depth, 90.0, 57), (seed, "right only"))
        defocus.fill_(0)
        n0 = ctx.launch_count
        ctx.frame_effects(None, None, defocus)
        ctx.sync()
        assert ctx.launch_count - n0 == 1                            # the table survived every stereo call
        assert np.array_equal(to_host(defocus, 3), defocus_bytes)
    ctx.close()


def test_captured_frame_stereo_reads_the_convergence_on_the_device(rtdd):
    """A graph captured from frame_stereo(convergence_point=...) on a torch stream, replayed after a new solve with other
    strokes, converges at the NEW depth under the point: it is read on the GPU and the call does no host work mid-stream."""
    rows, cols, iters, D = 203, 317, 120, 57
    bgr, scribble, edited = synth.synth_case(rows, cols, 31)
    ctx = rtdd.DepthDiffusion(rows, cols)
    s = torch.cuda.Stream()
    ctx.set_stream(s)
    ctx.frame_set_image(bgr)
    ctx.frame_solve_host(scribble, edited, iters, None)
    x, y = 150, 90
    outs = [to_dev(np.zeros_like(bgr), 3) for _ in NAMES]
    ctx.frame_stereo(*outs, convergence_point=(x, y), max_disparity=D)          # warm-up
    ctx.sync()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=s):
        ctx.frame_stereo(*outs, convergence_point=(x, y), max_disparity=D)
    depth1 = ctx.frame_plane(ctx.PLANE_DEPTH, 0).cpu().numpy()
    colour = 17 if depth1[y, x] > 128 else 240
    ctx.frame_paint(x, y, colour, 6)                             # a stroke over the point: its depth becomes `colour`
    ctx.frame_paint(30, 40, 255 - colour, 9)
    ctx.frame_solve(iters)
    ctx.sync()
    depth2 = ctx.frame_plane(ctx.PLANE_DEPTH, 0).cpu().numpy()
    assert depth2[y, x] == colour and abs(float(depth1[y, x]) - colour) > 10.0
    for o in outs:
        o.fill_(0)
    torch.cuda.synchronize()
    with torch.cuda.stream(s):
        g.replay()
    s.synchronize()
    check_views(outs, ref.stereo(bgr, depth2, float(colour), D), "replay")
    stale = ref.stereo(bgr, depth2, clamp_depth(depth1[y, x]), D)
    assert not np.array_equal(to_host(outs[0], 3), stale[0])
    del g
    ctx.set_stream(None)
    ctx.close()


def test_argument_errors_leave_the_context_usable(rtdd):
    from realtimedepthdiffusion_b200 import _native
    lib = _native.lib
    rows, cols = 67, 121
    bgr, depth = stereo_inputs(rows, cols, 8)
    ctx = rtdd.DepthDiffusion(rows, cols)
    h = ctx._h
    L, R, A = (to_dev(np.zeros_like(bgr), 3) for _ in NAMES)
    pl = pitch(L)
    assert lib.rtdd_frame_stereo(h, ptr(L), pl, ptr(R), pl, ptr(A), pl, -1, -1, 10.0, 8) == -2     # before frame_set_image
    ctx.frame_set_image(bgr)
    o, d = to_dev(bgr, 3), to_dev(depth)
    po, pd = pitch(o), pitch(d)
    nan = float("nan")
    ok = dict(o=o, po=po, d=d, pd=pd, L=L, pl=pl, R=R, pr=pl, A=A, pa=pl, rows=rows, cols=cols, c=10.0, D=8)
    bad_stand_alone = [dict(o=None), dict(d=None), dict(L=None, R=None, A=None), dict(po=cols * 3 - 1), dict(pd=cols * 4 - 4),
                       dict(pd=pd + 2), dict(pl=cols * 3 - 1), dict(pr=cols * 3 - 1), dict(pa=cols * 3 - 1), dict(rows=-1), dict(cols=-1),
                       dict(c=nan), dict(c=-0.5), dict(c=255.5), dict(D=-1), dict(D=1025)]
    bad_frame = [dict(L=None, R=None, A=None), dict(pl=cols * 3 - 1), dict(pr=cols * 3 - 1), dict(pa=cols * 3 - 1),
                 dict(c=nan), dict(c=256.0), dict(c=-1.0), dict(D=-1), dict(D=1025),
                 dict(x=cols, y=0), dict(x=0, y=rows), dict(x=-1, y=5), dict(x=5, y=-1), dict(x=-2, y=-2)]

    def p(t):
        return ptr(t) if t is not None else C.c_void_p(0)

    n0 = ctx.launch_count
    for change in bad_stand_alone:
        a = dict(ok, **change)
        assert lib.rtdd_stereo(h, p(a["o"]), a["po"], p(a["d"]), a["pd"], p(a["L"]), a["pl"], p(a["R"]), a["pr"], p(a["A"]), a["pa"],
                               a["rows"], a["cols"], a["c"], a["D"]) == -1, change
    for change in bad_frame:
        a = dict(ok, x=-1, y=-1)
        a.update(change)
        assert lib.rtdd_frame_stereo(h, p(a["L"]), a["pl"], p(a["R"]), a["pr"], p(a["A"]), a["pa"], a["x"], a["y"], a["c"], a["D"]) == -1, change
    # empty images launch nothing
    assert lib.rtdd_stereo(h, p(o), po, p(d), pd, p(L), pl, p(R), pl, p(A), pl, 0, cols, 10.0, 8) == 0
    assert lib.rtdd_stereo(h, p(o), po, p(d), pd, p(L), pl, p(R), pl, p(A), pl, rows, 0, 10.0, 8) == 0
    assert ctx.launch_count == n0
    with pytest.raises(ValueError):
        ctx.frame_stereo(L)
    with pytest.raises(ValueError):
        ctx.frame_stereo(L, convergence_point=(1, 1), convergence_depth=3.0)
    with pytest.raises(rtdd.RtddError):
        ctx.frame_stereo(L, convergence_point=(-1, -1))
    # still exact afterwards, both forms
    ctx.stereo(o, d, L, R, A, convergence_depth=37.5, max_disparity=1024)
    ctx.sync()
    check_views((L, R, A), ref.stereo(bgr, depth, 37.5, 1024), "stand-alone after errors")
    ctx.frame_solve_host(*synth.synth_case(rows, cols, 8)[1:], 60, None)
    fd = ctx.frame_plane(ctx.PLANE_DEPTH, 0).cpu().numpy()
    ctx.frame_stereo(L, R, A, convergence_point=(cols - 1, 0), max_disparity=57)
    ctx.sync()
    check_views((L, R, A), ref.stereo(bgr, fd, clamp_depth(fd[0, cols - 1]), 57), "frame after errors")
    ctx.close()


def test_rows_wider_than_the_limit_are_refused(rtdd):
    from realtimedepthdiffusion_b200 import _native
    lib = _native.lib
    rows, cols = 8, 16385
    bgr, depth = stereo_inputs(rows, cols, 3)
    ctx = rtdd.DepthDiffusion(rows, cols)
    o, d = to_dev(bgr, 3), to_dev(depth)
    outs = [to_dev(np.zeros_like(bgr), 3) for _ in NAMES]
    args = [x for t in outs for x in (ptr(t), pitch(t))]
    n0 = ctx.launch_count
    assert lib.rtdd_stereo(ctx._h, ptr(o), pitch(o), ptr(d), pitch(d), *args, rows, cols, 10.0, 8) == -1
    assert ctx.launch_count == n0
    assert lib.rtdd_stereo(ctx._h, ptr(o), pitch(o), ptr(d), pitch(d), *args, rows, cols - 1, 10.0, 8) == 0   # 16384 fits
    ctx.sync()
    assert ctx.launch_count - n0 == 1
    want = ref.stereo(bgr[:, :cols - 1], depth[:, :cols - 1], 10.0, 8)
    for name, o, w in zip(NAMES, outs, want):
        assert np.array_equal(to_host(o, 3)[:, :cols - 1], w), name
    ctx.frame_set_image(bgr)
    n0 = ctx.launch_count
    with pytest.raises(rtdd.RtddError):
        ctx.frame_stereo(*outs, convergence_depth=10.0, max_disparity=8)
    assert ctx.launch_count == n0
    ctx.close()
