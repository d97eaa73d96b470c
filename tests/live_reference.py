"""CPU restatement of the two live-stroke re-solves of a frame context, rtdd_frame_solve_incremental and rtdd_frame_solve_band
(include/rtdd.h), from the oracle's primitives alone.  Neither is the reference's frame, but each is a fixed composition of
operations the oracle restates bit for bit, so each has exact expected bits.  Both functions mutate an oracle.binding.FrameState
the way the device mutates its context planes: every level's scribble, edited and depth plane ends as the context's does.

tests/test_live_reference_cpu.py checks the restatement against itself and the parity frame; tests/test_gpu_live_strokes.py
checks the device against it."""
import numpy as np

from oracle import binding as ob

synth = ob.pkg_file("synth")
# levels with fewer pixels than this are solved whole by the band re-solve (rtdd_abi.cu, rtdd_frame_solve_band)
WHOLE_LEVEL_PIXELS = 1 << 20


def level_iterations(max_iterations, levels, level):
    """Sweeps of `level` in a frame of `max_iterations` (ref: src/main.cpp:263; rtdd_level_iterations)."""
    return int(np.float32(max_iterations) / np.float32(2.0 ** ((levels - 1) - level)))


def restrict_annotations(st, coarsest):
    """pyrDown of the level-0 annotation into levels 1..coarsest; the coarser levels keep their planes."""
    for l in range(1, coarsest + 1):
        st.scribble[l], st.edited[l] = ob.pyrdown_annotation(st.scribble[l - 1], st.edited[l - 1], st.scribble[l], st.edited[l])


def solve_incremental(st, max_iterations, coarsest):
    """rtdd_frame_solve_incremental: the frame re-solved from level `coarsest` down, starting there from that level's own
    previous solution.  coarsest = levels - 1 is the parity frame.  Returns the 8-bit map."""
    L = st.levels
    if not 0 <= coarsest < L:
        raise ValueError("coarsest level %d outside [0, %d)" % (coarsest, L))
    restrict_annotations(st, coarsest)
    st.depth[coarsest] = ob.convert_to_float(st.edited[coarsest], st.depth[coarsest], st.scribble[coarsest])
    for l in range(coarsest, -1, -1):
        st.depth[l] = ob.solve_level(st.depth[l], st.scribble[l], st.gray[l], level_iterations(max_iterations, L, l), l, L - 1, st.lut)
        if l > 0:
            rows, cols = st.sizes[l - 1]
            st.depth[l - 1] = ob.convert_to_float(st.edited[l - 1], ob.pyrup_f32(st.depth[l], rows, cols), st.scribble[l - 1])
    return ob.quantise_u8(st.depth[0])


def band_rows(sizes, level, row_begin, row_end, dilation):
    """(b0, b1, whole): the rows of `level` the band re-solve solves; whole = the level is solved entirely (b0, b1 = 0, rows).
    A level is solved whole when it is the coarsest, has fewer than 2^20 pixels, or the band covers >= 60 % of its rows."""
    rows, cols = sizes[level]
    b0 = max((row_begin >> level) - dilation, 0)
    b1 = min(((row_end + (1 << level) - 1) >> level) + dilation, rows)
    whole = level == len(sizes) - 1 or rows * cols < WHOLE_LEVEL_PIXELS or (b1 - b0) * 10 >= rows * 6
    return (0, rows, True) if whole else (b0, b1, False)


def band_guess(new_coarse, old_coarse, depth, b0, b1):
    """A level's guess before its band re-solve: rows [b0, b1) take pyrUp of the coarser level's new solution; the other rows
    keep their previous solution plus the prolongated change pyrUp(new) - pyrUp(old), in fp32."""
    rows, cols = depth.shape
    up_new = ob.pyrup_f32(new_coarse, rows, cols)
    up_old = ob.pyrup_f32(old_coarse, rows, cols)
    guess = depth + (up_new - up_old)
    guess[b0:b1] = up_new[b0:b1]
    return guess


def solve_level_rows(depth, scribble, gray, iterations, level, max_level, lut, b0, b1):
    """The level solved on rows [b0, b1) only, rows b0-1 and b1 frozen (when inside the level): the whole-level solve with every
    row outside the band made Dirichlet.  Exact, since the edge weights do not read the scribble and a band row reads no row
    beyond b0-1 .. b1."""
    s = np.array(scribble, np.uint8, copy=True)
    s[:b0] = 255
    s[b1:] = 255
    return ob.solve_level(depth, s, gray, iterations, level, max_level, lut)


def solve_band(st, max_iterations, row_begin, row_end, dilation, level_solver=solve_level_rows):
    """rtdd_frame_solve_band after level-0 rows [row_begin, row_end) changed.  Returns (8-bit map, [(level, b0, b1) of every
    level solved as a band]).  level_solver: another formulation of solve_level_rows (the tests' cross-check)."""
    L = st.levels
    if dilation < 1 or row_begin < 0 or row_end > st.rows or row_end <= row_begin or max_iterations < 0:
        raise ValueError("band [%d, %d) dilation %d, %d iterations" % (row_begin, row_end, dilation, max_iterations))
    restrict_annotations(st, L - 1)
    old = [d.copy() for d in st.depth]
    banded = []
    for l in range(L - 1, -1, -1):
        b0, b1, whole = band_rows(st.sizes, l, row_begin, row_end, dilation)
        if not whole:
            banded.append((l, b0, b1))
        d = st.depth[l]
        if l < L - 1:
            d = band_guess(st.depth[l + 1], old[l + 1], d, b0, b1)
        d = ob.convert_to_float(st.edited[l], d, st.scribble[l])
        st.depth[l] = level_solver(d, st.scribble[l], st.gray[l], level_iterations(max_iterations, L, l), l, L - 1, st.lut, b0, b1)
    return ob.quantise_u8(st.depth[0]), banded


def first_frame(rows, cols, seed, max_iterations=1000):
    """(bgr, scribble, edited, state after the parity frame of a synthetic case)."""
    bgr, scribble, edited = synth.synth_case(rows, cols, seed)
    st = ob.FrameState(bgr)
    st.solve(scribble, edited, max_iterations)
    return bgr, scribble, edited, st


def diagonal_stroke(x, y, colour, radius, dabs=3):
    """Brush events of a short stroke down and to the right from (x, y)."""
    return [(x + k * radius, y + k * (radius // 2), colour, radius) for k in range(dabs)]


def paint(st, events):
    """Brush events (x, y, colour, radius) on the level-0 annotation, as rtdd_frame_paint does.  Returns the level-0 rows
    [row_begin, row_end) they touched."""
    r0, r1 = st.rows, 0
    for x, y, colour, radius in events:
        st.edited[0], st.scribble[0] = ob.paint(x, y, colour, radius, st.edited[0], st.scribble[0])
        h = radius // 2
        r0, r1 = min(r0, max(y - h, 0)), max(r1, min(y + h + 1, st.rows))
    return r0, r1
