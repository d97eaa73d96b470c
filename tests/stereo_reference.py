"""CPU reference of the stereo extension (rtdd_stereo, include/rtdd.h), written from its definition and independent of the CUDA
code.  NumPy, vectorised over the image: the z-buffer is a u64 minimum per target, key (bits(d') << 32) | x, which orders by d'
(d' >= 0, -0 made +0) and carries the winner's column; the nearest covered targets either side of a hole come from running
maximum / minimum of the covered columns.  tests/test_stereo_cpu.py checks it against a per-pixel brute force."""
import numpy as np

EMPTY = np.uint64(0xFFFFFFFFFFFFFFFF)


def clamped_depth(depth):
    """d' = fminf(fmaxf(d, 0), 255): NaN -> 0, and -0 -> +0 so that the bit patterns order like the values."""
    d = np.asarray(depth, np.float32)
    return np.fmin(np.fmax(d, np.float32(0)), np.float32(255)) + np.float32(0)


def parallax(depth, convergence, max_disparity):
    """(d', s, hL, hR): s = cvt.rzi.s32.f64((double)((float)D * (d' - c)) / 255.0), hL = s / 2 toward zero, hR = s - hL."""
    dc = clamped_depth(depth)
    q = np.float32(max_disparity) * (dc - np.float32(convergence))          # fp32, round to nearest, like the definition
    s = np.trunc(q.astype(np.float64) / 255.0).astype(np.int64)
    h_left = np.sign(s) * (np.abs(s) // 2)
    return dc, s, h_left, s - h_left


def _view(bgr, dc, targets):
    rows, cols = dc.shape
    xs = np.arange(cols)
    key = (dc.view(np.uint32).astype(np.uint64) << np.uint64(32)) | xs.astype(np.uint64)[None, :]
    ok = (targets >= 0) & (targets < cols)
    flat = (np.arange(rows)[:, None] * cols + targets)[ok]
    z = np.full(rows * cols, EMPTY, np.uint64)
    np.minimum.at(z, flat, key[ok])
    z = z.reshape(rows, cols)
    covered = z != EMPTY
    left = np.maximum.accumulate(np.where(covered, xs, -1), axis=1)                      # nearest covered at or left of t
    right = np.minimum.accumulate(np.where(covered, xs, cols)[:, ::-1], axis=1)[:, ::-1]  # ... at or right of t; cols = none
    rr = np.arange(rows)[:, None]
    zl, zr = z[rr, np.maximum(left, 0)], z[rr, np.minimum(right, cols - 1)]
    take_left = (left >= 0) & ((right == cols) | ((zl >> np.uint64(32)) >= (zr >> np.uint64(32))))   # covered t: left = right = t
    src = (np.where(take_left, zl, zr) & np.uint64(0xFFFFFFFF)).astype(np.int64)
    src = np.where((left < 0) & (right == cols), xs, src)                                 # a row with nothing covered
    return bgr[rr, src]


def stereo(bgr, depth, convergence, max_disparity):
    """bgr [rows, cols, 3] u8, depth [rows, cols] fp32 -> (left, right, anaglyph), each [rows, cols, 3] u8."""
    bgr = np.ascontiguousarray(bgr, np.uint8)
    dc, _, h_left, h_right = parallax(depth, convergence, max_disparity)
    xs = np.arange(dc.shape[1])[None, :]
    left = _view(bgr, dc, xs - h_left)
    right = _view(bgr, dc, xs + h_right)
    anaglyph = right.copy()
    anaglyph[..., 2] = left[..., 2]                                   # B, G of the right view, R of the left one
    return left, right, anaglyph
