"""CPU tests of the stereo extension (rtdd_stereo, no reference counterpart): the vectorised CPU reference
(tests/stereo_reference.py) against a per-pixel brute force of the definition in include/rtdd.h, the parity points, a pure
translation, holes behind a foreground square, the unique-winner claim, the integer form of the parallax rule the kernel
uses, and the C ABI's argument errors without a device."""
import math

import numpy as np
import pytest

from realtimedepthdiffusion_b200 import synth
from tests import stereo_reference as ref


def brute_stereo(bgr, depth, convergence, max_disparity):
    """The definition, one source and one target at a time.  Returns (left, right, anaglyph, collisions): collisions counts the
    targets more than one source lands on; two sources with equal d' on one target fail an assertion."""
    rows, cols = depth.shape
    D, c = np.float32(max_disparity), np.float32(convergence)
    views, collisions = [], 0
    for view in ("left", "right"):
        out = np.empty_like(bgr)
        for y in range(rows):
            landed = {}                                          # target -> [(d', x)]
            for x in range(cols):
                d = np.float32(depth[y, x])
                dc = np.float32(0) if math.isnan(d) else np.float32(min(max(float(d), 0.0), 255.0))
                dc = np.float32(0) if dc == 0 else dc            # -0 counts as +0
                s = math.trunc(float(D * np.float32(dc - c)) / 255.0)
                assert abs(s) <= max_disparity
                h_left = int(s / 2)
                t = x - h_left if view == "left" else x + (s - h_left)
                if 0 <= t < cols:
                    landed.setdefault(t, []).append((float(dc), x))
            winner = {}
            for t, srcs in landed.items():
                assert len({d for d, _ in srcs}) == len(srcs), (y, t, srcs)     # equal d' never share a target
                collisions += len(srcs) > 1
                winner[t] = min(srcs)
            for t in range(cols):
                if t in winner:
                    out[y, t] = bgr[y, winner[t][1]]
                    continue
                lt = next((u for u in range(t - 1, -1, -1) if u in winner), None)
                rt = next((u for u in range(t + 1, cols) if u in winner), None)
                if lt is None and rt is None:
                    out[y, t] = bgr[y, t]
                elif rt is None or (lt is not None and winner[lt][0] >= winner[rt][0]):
                    out[y, t] = bgr[y, winner[lt][1]]
                else:
                    out[y, t] = bgr[y, winner[rt][1]]
        views.append(out)
    left, right = views
    anaglyph = np.stack([right[..., 0], right[..., 1], left[..., 2]], axis=-1)
    return left, right, anaglyph, collisions


def odd_depth(rows, cols, rng):
    """Depths across [-40, 300] with NaN and -0: the clamp and its NaN / sign rules are part of the definition."""
    d = rng.uniform(-40.0, 300.0, (rows, cols)).astype(np.float32)
    d[rng.random((rows, cols)) < 0.05] = np.nan
    d[rng.random((rows, cols)) < 0.05] = np.float32(-0.0)
    d.flat[: min(d.size, 7)] = np.array([np.nan, -0.0, -7.0, 255.0, 262.5, 1.0, 0.0], np.float32)[: min(d.size, 7)]
    return d


def assert_views_equal(got, want, what):
    for name, g, w in zip(("left", "right", "anaglyph"), got[:3], want[:3]):
        assert np.array_equal(g, w), (what, name, int((g != w).any(-1).sum()))


SMALL = [(1, 1), (1, 9), (7, 1), (2, 3), (5, 3), (16, 16), (31, 17), (45, 47), (12, 130)]


@pytest.mark.parametrize("rows,cols", SMALL)
def test_reference_equals_brute_force(rows, cols):
    rng = np.random.default_rng(rows * 1000 + cols)
    bgr = rng.integers(0, 256, (rows, cols, 3), dtype=np.uint8)
    depth = odd_depth(rows, cols, rng)
    big = min(2 * cols + 3, 1024)                                  # large against cols: rows with no covered target
    params = [(c, D) for D in (0, 1, 2, 7, 40, big) for c in (0.0, 37.5, 255.0)]
    params += [(float(np.float32(rng.uniform(0, 255))), int(rng.integers(0, 1025))) for _ in range(4)]
    for c, D in params:
        assert_views_equal(ref.stereo(bgr, depth, c, D), brute_stereo(bgr, depth, c, D), (c, D))


def test_parity_points_are_the_identity():
    rows, cols = 37, 91
    rng = np.random.default_rng(4)
    bgr = synth.synth_image(rows, cols, 4)
    depth = odd_depth(rows, cols, rng)
    for c in (0.0, 37.5, 128.0, 255.0):
        for view in ref.stereo(bgr, depth, c, 0):                      # D = 0
            assert np.array_equal(view, bgr), c
        for view in ref.stereo(bgr, np.full((rows, cols), c, np.float32), c, 1024):   # every depth on the convergence plane
            assert np.array_equal(view, bgr), c
    for view in ref.stereo(bgr, np.full((rows, cols), -3.0, np.float32), 0.0, 1024):  # clamped onto it
        assert np.array_equal(view, bgr)


@pytest.mark.parametrize("d0,c,D", [(200.0, 128.0, 40), (20.0, 128.0, 40), (255.0, 0.0, 57), (0.0, 255.0, 1024), (0.0, 255.0, 13),
                                    (90.0, 37.5, 5)])
def test_constant_depth_is_a_translation(d0, c, D):
    rows, cols = 9, 301
    bgr = synth.synth_image(rows, cols, 6)
    _, s, h_left, h_right = ref.parallax(np.float32([[d0]]), c, D)
    s, h_left, h_right = int(s[0, 0]), int(h_left[0, 0]), int(h_right[0, 0])
    assert s != 0
    left, right, anaglyph = ref.stereo(bgr, np.full((rows, cols), d0, np.float32), c, D)
    t = np.arange(cols)
    if max(abs(h_left), abs(h_right)) < cols:
        # the uncovered edge columns repeat the nearest covered one
        assert np.array_equal(left, bgr[:, np.clip(t + h_left, 0, cols - 1)])
        assert np.array_equal(right, bgr[:, np.clip(t - h_right, 0, cols - 1)])
    want = brute_stereo(bgr, np.full((rows, cols), d0, np.float32), c, D)
    assert_views_equal((left, right, anaglyph), want, (d0, c, D))


def test_foreground_square_holes_take_the_background():
    rows, cols, y0, y1, x0, x1 = 40, 120, 10, 30, 50, 70
    rng = np.random.default_rng(12)
    bgr = rng.integers(10, 256, (rows, cols, 3), dtype=np.uint8)
    square = np.array([1, 2, 3], np.uint8)
    bgr[y0:y1, x0:x1] = square
    depth = np.full((rows, cols), 200.0, np.float32)
    depth[y0:y1, x0:x1] = 20.0
    c, D = 128.0, 40
    _, _, hl_bg, hr_bg = ref.parallax(np.float32([[200.0]]), c, D)
    _, _, hl_fg, hr_fg = ref.parallax(np.float32([[20.0]]), c, D)
    assert (int(hl_bg[0, 0]), int(hr_bg[0, 0]), int(hl_fg[0, 0]), int(hr_fg[0, 0])) == (5, 6, -8, -8)
    left, right, anaglyph = ref.stereo(bgr, depth, c, D)
    for view, shift, bg_shift in ((left, 8, -5), (right, -8, 6)):
        is_square = (view == square).all(-1)
        want = np.zeros((rows, cols), bool)
        want[y0:y1, x0 + shift:x1 + shift] = True                       # the square moves whole, the holes beside it are background
        assert np.array_equal(is_square, want)
        # disocclusion: the columns the square uncovers repeat the background column next to them
        hole = slice(x0 + bg_shift, x0 + shift) if shift > 0 else slice(x1 + shift, x1 + bg_shift)
        edge = x0 + bg_shift - 1 if shift > 0 else x1 + bg_shift
        assert (view[y0:y1, hole] == view[y0:y1, edge:edge + 1]).all()
        assert not (view[y0:y1, hole] == square).all(-1).any()
    assert_views_equal((left, right, anaglyph), brute_stereo(bgr, depth, c, D), "square")


def test_equal_depths_never_share_a_target():
    """Quantised depths make equal d' common, and the brute force asserts that two of them never land on one target;
    collisions of different depths do occur, so the nearest-wins rule is exercised."""
    rows, cols = 24, 200
    rng = np.random.default_rng(21)
    bgr = rng.integers(0, 256, (rows, cols, 3), dtype=np.uint8)
    depth = (rng.integers(0, 16, (rows, cols)) * 17.0).astype(np.float32)
    depth[:, ::7] = np.float32(-0.0)
    total = 0
    for c, D in ((0.0, 40), (128.0, 57), (37.5, 1024), (255.0, 3), (100.0, 255)):
        got = ref.stereo(bgr, depth, c, D)
        *want, collisions = brute_stereo(bgr, depth, c, D)
        assert_views_equal(got, want, (c, D))
        total += collisions
    assert total > 1000


def test_integer_parallax_equals_the_fp64_rule():
    """The kernel takes s as trunc(q) / 255 in integers (q = (float)D * (d' - c)); the definition divides in fp64.  Equal for
    every q near each multiple of 255 (a few ulps either side) and for random ones, at every D."""
    qs = []
    for D in range(0, 1025):
        n = np.arange(-D, D + 1, dtype=np.float64)
        diff = (255.0 * n / max(D, 1)).astype(np.float32)
        for k in range(-3, 4):
            di = (diff.view(np.int32) + k).view(np.float32)
            di = di[np.isfinite(di) & (np.abs(di) <= 255)]
            qs.append(np.float32(D) * di)
    rng = np.random.default_rng(5)
    dc = rng.uniform(0, 255, 200000).astype(np.float32)
    c = rng.uniform(0, 255, 200000).astype(np.float32)
    qs.append(rng.integers(0, 1025, 200000).astype(np.float32) * (dc - c))
    q = np.concatenate(qs)
    fp64 = np.trunc(q.astype(np.float64) / 255.0).astype(np.int64)
    it = np.trunc(q).astype(np.int64)
    integer = np.sign(it) * (np.abs(it) // 255)                     # C division, toward zero
    assert np.array_equal(fp64, integer)


def test_argument_errors_without_a_device():
    from realtimedepthdiffusion_b200 import _native
    lib = _native.lib
    assert lib.rtdd_stereo(None, None, 0, None, 0, None, 0, None, 0, None, 0, 1, 1, 0.0, 0) == -1
    assert lib.rtdd_stereo(None, None, 0, None, 0, None, 0, None, 0, None, 0, 1, 20000, float("nan"), 5000) == -1
    assert lib.rtdd_frame_stereo(None, None, 0, None, 0, None, 0, -1, -1, 0.0, 0) == -1
    assert lib.rtdd_frame_stereo(None, None, 0, None, 0, None, 0, 3, 4, 0.0, 2000) == -1
