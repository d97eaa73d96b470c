"""CPU tests of the live-stroke restatement (tests/live_reference.py): its incremental and band re-solves reduce to the parity
frame where they must, its frozen-row band solve agrees with an independent formulation (the band solved on its own cropped
window), and the standard stroke cases exercise what the GPU tests rely on -- banded levels, and maps the parity frame does
not reproduce."""
import numpy as np
import pytest

from oracle import binding as ob
from tests import live_reference as lr

synth = ob.pkg_file("synth")


def bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def assert_same_state(got, want, what):
    for l in range(want.levels):
        diff = np.nonzero((bits(got.depth[l]) != bits(want.depth[l])).any(axis=1))[0]
        assert diff.size == 0, "%s: level %d differs on %d rows, first %d" % (what, l, diff.size, diff[0])


def cropped_solve(depth, scribble, gray, iterations, level, max_level, lut, b0, b1):
    """solve_level_rows formulated differently: the level solved on its window [b0-1, b1+1) alone, with the window's first and
    last rows (when inside the level) made Dirichlet; rows outside [b0, b1) keep `depth`."""
    rows = depth.shape[0]
    w0, w1 = max(b0 - 1, 0), min(b1 + 1, rows)
    s = np.array(scribble[w0:w1], np.uint8, copy=True)
    if b0 > 0:
        s[0] = 255
    if b1 < rows:
        s[-1] = 255
    win = ob.solve_level(depth[w0:w1], s, gray[w0:w1], iterations, level, max_level, lut)
    out = np.array(depth, np.float32, copy=True)
    out[b0:b1] = win[b0 - w0:b1 - w0]
    return out


def test_level_iterations_match_the_frame_loop():
    # ref: src/main.cpp:263 -- the count oracle.binding.FrameState.solve uses
    assert [lr.level_iterations(1000, 5, l) for l in range(5)] == [62, 125, 250, 500, 1000]
    assert [lr.level_iterations(31, 6, l) for l in range(6)] == [0, 1, 3, 7, 15, 31]


@pytest.mark.parametrize("rows,cols", [(203, 317), (540, 960)])
def test_incremental_from_the_coarsest_level_is_the_parity_frame(rows, cols):
    bgr, scribble, edited, st = lr.first_frame(rows, cols, 31)
    parity = ob.FrameState(bgr)
    parity.solve(scribble, edited, 1000)
    lr.paint(st, synth.brush_events(rows, cols, 32, 2, 4))
    want = parity.solve(st.scribble[0], st.edited[0], 1000)
    got = lr.solve_incremental(st, 1000, st.levels - 1)
    assert np.array_equal(got, want)
    assert_same_state(st, parity, "incremental from level %d" % (st.levels - 1))


def test_incremental_from_a_finer_level_keeps_the_coarser_levels():
    rows, cols = 540, 960
    _, _, _, st = lr.first_frame(rows, cols, 41)
    coarse = [(st.depth[l].copy(), st.scribble[l].copy()) for l in range(2, st.levels)]
    lr.paint(st, synth.brush_events(rows, cols, 42, 1, 4))
    lr.solve_incremental(st, 1000, 1)
    for l, (d, s) in enumerate(coarse, start=2):
        assert np.array_equal(bits(st.depth[l]), bits(d)) and np.array_equal(st.scribble[l], s), "level %d was touched" % l
    with pytest.raises(ValueError):
        lr.solve_incremental(st, 1000, st.levels)


@pytest.mark.parametrize("rows,cols,dilation", [(1080, 1920, 1 << 20), (540, 960, 1)])
def test_band_covering_every_level_is_the_parity_frame(rows, cols, dilation):
    """A band wider than every level, and a frame whose levels are all below 2^20 pixels: every level is solved whole."""
    bgr, scribble, edited, st = lr.first_frame(rows, cols, 51)
    parity = ob.FrameState(bgr)
    parity.solve(scribble, edited, 1000)
    r0, r1 = lr.paint(st, synth.brush_events(rows, cols, 52, 1, 4))
    want = parity.solve(st.scribble[0], st.edited[0], 1000)
    got, banded = lr.solve_band(st, 1000, r0, r1, dilation)
    assert banded == []
    assert np.array_equal(got, want)
    assert_same_state(st, parity, "band solved whole")


@pytest.mark.parametrize("level", [0, 1])
@pytest.mark.parametrize("b0,b1", [(100, 103), (0, 40), (260, 300), (150, 151), (0, 1), (299, 300)])
def test_frozen_row_band_equals_the_cropped_window_solve(b0, b1, level):
    rows, cols, iters = 300, 517, 37
    gray = ob.bgr2gray(synth.synth_image(rows, cols, 9))
    rng = np.random.default_rng(b0 * 1000 + b1)
    depth = (rng.integers(0, 5, (rows, cols)) * 60 + rng.uniform(0, 14, (rows, cols))).astype(np.float32)
    scribble = np.where(rng.random((rows, cols)) < 0.1, 255, 0).astype(np.uint8)
    lut = ob.load_weights(0.4)
    masked = lr.solve_level_rows(depth, scribble, gray, iters, level, 3, lut, b0, b1)
    cropped = cropped_solve(depth, scribble, gray, iters, level, 3, lut, b0, b1)
    assert np.array_equal(bits(masked), bits(cropped))
    assert np.array_equal(bits(masked[:b0]), bits(depth[:b0])) and np.array_equal(bits(masked[b1:]), bits(depth[b1:]))
    assert not np.array_equal(bits(masked[b0:b1]), bits(depth[b0:b1]))       # the band itself was solved


# (rows, cols, stroke, dilation, max_iterations, banded levels): a stroke in the middle, touching row 0, touching the last row,
# and a one-row edit whose level-0 band (3 rows) is thinner than the 8-sweep passes of the band solve
STROKES = [
    (1080, 1920, "middle", 96, 1000, [0]),
    (1080, 1920, "top", 24, 100, [0]),
    (1080, 1920, "bottom", 24, 15, [0]),
    (1080, 1920, "row", 1, 1000, [0]),
    (2160, 3840, "middle", 96, 1000, [1, 0]),
]


def stroke(rows, cols, where):
    radius = int(min(rows, cols) * 0.02)
    if where == "middle":
        return lr.diagonal_stroke(cols // 3, rows // 2, 128, radius)
    if where == "top":
        return lr.diagonal_stroke(cols // 2, 0, 64, radius)
    if where == "bottom":
        return lr.diagonal_stroke(cols // 4, rows - 1, 192, radius, 1)
    return [(cols // 2, rows // 2 + 1, 0, 1)]          # radius 1: one pixel


@pytest.mark.parametrize("rows,cols,where,dilation,iters,levels", STROKES)
def test_band_frame_equals_its_cropped_window_formulation(rows, cols, where, dilation, iters, levels):
    """Every banded level of a real band frame -- image-edge bands and a 3-row band included -- solved both ways."""
    _, _, _, st = lr.first_frame(rows, cols, 61)
    r0, r1 = lr.paint(st, stroke(rows, cols, where))
    twin = ob.FrameState(st.bgr)
    for l in range(st.levels):
        twin.scribble[l], twin.edited[l], twin.depth[l] = st.scribble[l].copy(), st.edited[l].copy(), st.depth[l].copy()
    got, banded = lr.solve_band(st, iters, r0, r1, dilation)
    want, banded2 = lr.solve_band(twin, iters, r0, r1, dilation, level_solver=cropped_solve)
    assert [b[0] for b in banded] == levels and banded == banded2
    if where in ("middle", "row"):
        assert all(0 < b0 and b1 < st.sizes[l][0] for l, b0, b1 in banded)
    if where == "top":
        assert banded[-1][1] == 0
    if where == "bottom":
        assert banded[-1][2] == rows
    if where == "row":
        assert banded[-1][2] - banded[-1][1] == 3
    assert np.array_equal(got, want)
    assert_same_state(st, twin, "band %s" % where)


@pytest.mark.parametrize("rows,cols,levels", [(1080, 1920, [0]), (2160, 3840, [1, 0])])
def test_band_frame_differs_from_the_parity_frame(rows, cols, levels):
    """The standard one-stroke cases band the levels the GPU tests expect, and their maps are not the parity frame's: a
    comparison with the restated band frame holds the device to more than the parity frame would."""
    bgr, scribble, edited, st = lr.first_frame(rows, cols, 5)
    parity = ob.FrameState(bgr)
    parity.solve(scribble, edited, 1000)
    r0, r1 = lr.paint(st, synth.brush_events(rows, cols, 3, 1, 1))
    want = parity.solve(st.scribble[0], st.edited[0], 1000)
    got, banded = lr.solve_band(st, 1000, r0, r1, 96)
    assert [b[0] for b in banded] == levels
    assert (got != want).mean() > 0.01
    for l in range(levels[0] + 1, st.levels):          # the levels solved whole are the parity frame's
        assert np.array_equal(bits(st.depth[l]), bits(parity.depth[l]))


def test_band_arguments_are_checked():
    _, _, _, st = lr.first_frame(203, 317, 71)
    for args in ((1000, -1, 5, 8), (1000, 0, 204, 8), (1000, 5, 5, 8), (1000, 0, 5, 0), (-1, 0, 5, 8)):
        with pytest.raises(ValueError):
            lr.solve_band(st, *args)
