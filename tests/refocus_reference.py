"""CPU reference of the refocus extension (rtdd_refocus, include/rtdd.h), written from its definition and independent of the
CUDA code.  NumPy, vectorised over the image: the box half-sides come from the fp32 / fp64 arithmetic the definition states, and
the window sums from an int64 summed-area table, so 4K frames with 4096-pixel apertures take well under a second per call.
tests/test_refocus_cpu.py checks it against a per-pixel brute force of the same definition."""
import numpy as np


def defocus_kernel_size(rows, cols):
    """The reference defocus's K = (int)(0.025 * (double)sqrtf((float)(rows^2 + cols^2)))."""
    return int(0.025 * float(np.sqrt(np.float32(rows * rows + cols * cols))))


def half_sides(depth, focus, depth_of_field, aperture):
    """h = a / 2 per pixel, a = cvt.rzi((double)((float)A * e) / 255), e = max(|clamp(d, 0, 255) - f| - w, 0)."""
    d = np.asarray(depth, np.float32)
    dc = np.fmin(np.fmax(d, np.float32(0)), np.float32(255))            # fmax / fmin ignore NaN: NaN -> 0
    e = np.fmax(np.abs(dc - np.float32(focus)) - np.float32(depth_of_field), np.float32(0))
    q = (np.float32(aperture) * e).astype(np.float64) / 255.0
    return np.trunc(q).astype(np.int64) // 2


def refocus(bgr, depth, focus, depth_of_field, aperture):
    """bgr [rows, cols, 3] u8, depth [rows, cols] fp32 -> refocused [rows, cols, 3] u8; aperture < 0 = the reference's K."""
    bgr = np.ascontiguousarray(bgr, np.uint8)
    rows, cols = bgr.shape[:2]
    if aperture < 0:
        aperture = defocus_kernel_size(rows, cols)
    h = half_sides(depth, focus, depth_of_field, aperture)
    out = bgr.copy()
    blur = h > 0
    if not blur.any():
        return out
    ys, xs = np.nonzero(blur)
    hb = h[blur]
    x0, x1 = np.maximum(xs - hb, 0), np.minimum(xs + hb, cols)
    y0, y1 = np.maximum(ys - hb, 0), np.minimum(ys + hb, rows)
    n = (x1 - x0) * (y1 - y0)
    for c in range(3):
        sat = np.zeros((rows + 1, cols + 1), np.int64)
        sat[1:, 1:] = bgr[..., c].astype(np.int64).cumsum(0).cumsum(1)
        s = sat[y1, x1] - sat[y0, x1] - sat[y1, x0] + sat[y0, x0]
        out[ys, xs, c] = (s // n).astype(np.uint8)
    return out
