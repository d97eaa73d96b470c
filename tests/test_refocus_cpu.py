"""CPU tests of the refocus extension (rtdd_refocus, no reference counterpart): the vectorised CPU reference
(tests/refocus_reference.py) against a per-pixel brute force of the definition in include/rtdd.h, its tie to the
reference-pinned defocus oracle at the parity point, and the C ABI's argument errors without a device."""
import glob
import os

import numpy as np
import pytest

from oracle import binding as ob
from realtimedepthdiffusion_b200 import synth
from tests import refocus_reference as ref

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def brute_refocus(bgr, depth, focus, band, aperture):
    """The definition, one window sum per pixel, fp32 where it says fp32."""
    rows, cols = depth.shape
    if aperture < 0:
        aperture = ob.defocus_kernel_size(rows, cols)
    dc = np.fmin(np.fmax(depth.astype(np.float32), np.float32(0)), np.float32(255))     # fmax / fmin: NaN -> 0
    e = np.fmax(np.abs(dc - np.float32(focus)) - np.float32(band), np.float32(0))
    q = (np.float32(aperture) * e).astype(np.float64) / 255.0
    half = np.trunc(q).astype(np.int64) // 2
    img = bgr.astype(np.int64)
    out = bgr.copy()
    for y, x in zip(*np.nonzero(half)):
        h = int(half[y, x])
        win = img[max(y - h, 0):min(y + h, rows), max(x - h, 0):min(x + h, cols)]
        out[y, x] = win.sum(axis=(0, 1)) // (win.shape[0] * win.shape[1])
    return out


def odd_depth(rows, cols, rng):
    """Depths across [-40, 300] with NaN: the clamp and its NaN rule are part of the definition."""
    d = rng.uniform(-40.0, 300.0, (rows, cols)).astype(np.float32)
    d[rng.random((rows, cols)) < 0.05] = np.nan
    d.flat[: min(d.size, 6)] = np.array([np.nan, -0.0, -7.0, 255.0, 262.5, 1.0], np.float32)[: min(d.size, 6)]
    return d


def test_parity_point_equals_reference_defocus_golden():
    """f = 0, w = 0, A = K on the depths the reference's own GPUSimulateDefocus was recorded with."""
    files = sorted(glob.glob(os.path.join(GOLD, "ref_effects_synth_*.npz")))
    assert files
    cases = {"synth_odd": (203, 317, 11)}
    for f in files:
        z = np.load(f)
        bgr, _, _ = synth.synth_case(*cases[os.path.basename(f)[len("ref_effects_"):-4]])
        depth = z["depth"]
        K = ob.defocus_kernel_size(*depth.shape)
        got = ref.refocus(bgr, depth, 0.0, 0.0, K)
        assert np.array_equal(got, z["GPUSimulateDefocus"])
        assert np.array_equal(got, ob.defocus(bgr, depth))
        assert np.array_equal(ref.refocus(bgr, depth, 0.0, 0.0, -1), got)


def test_parity_point_with_negative_and_nan_depths():
    rng = np.random.default_rng(3)
    bgr = synth.synth_image(67, 121, 3)
    depth = odd_depth(67, 121, rng)
    depth = np.where(depth > 255, np.float32(255), depth)        # the equality holds for depths <= 255 (and NaN)
    assert np.array_equal(ref.refocus(bgr, depth, 0.0, 0.0, -1), ob.defocus(bgr, depth))


SMALL = [(1, 1), (1, 9), (7, 1), (2, 3), (5, 3), (16, 16), (31, 17), (45, 47), (70, 130)]


@pytest.mark.parametrize("rows,cols", SMALL)
def test_reference_equals_brute_force(rows, cols):
    rng = np.random.default_rng(rows * 1000 + cols)
    bgr = rng.integers(0, 256, (rows, cols, 3), dtype=np.uint8)
    depth = odd_depth(rows, cols, rng)
    big = 2 * max(rows, cols) + 3                         # boxes larger than the image
    params = [(0.0, 0.0, -1), (255.0, 0.0, 1), (128.0, 20.0, 2), (37.5, 0.0, big), (255.0, 0.0, 4096)]
    for _ in range(6):
        params.append((float(np.float32(rng.uniform(0, 255))), float(np.float32(rng.uniform(0, 60))), int(rng.integers(0, big + 40))))
    for f, w, a in params:
        want = brute_refocus(bgr, depth, f, w, a)
        assert np.array_equal(ref.refocus(bgr, depth, f, w, a), want), (f, w, a)


def test_sharp_band_and_zero_aperture_are_the_identity():
    rows, cols = 60, 90
    rng = np.random.default_rng(9)
    bgr = synth.synth_image(rows, cols, 9)
    depth = odd_depth(rows, cols, rng)
    assert np.array_equal(ref.refocus(bgr, depth, 100.0, 0.0, 0), bgr)
    assert np.array_equal(ref.refocus(bgr, depth, 100.0, 300.0, 4096), bgr)     # the band covers every depth
    f, w = 100.0, 30.0
    out = ref.refocus(bgr, depth, f, w, 400)
    dc = np.fmin(np.fmax(depth, np.float32(0)), np.float32(255))
    inside = np.abs(dc - np.float32(f)) <= np.float32(w)
    assert inside.any() and (~inside).any()
    assert np.array_equal(out[inside], bgr[inside])
    assert not np.array_equal(out[~inside], bgr[~inside])


def test_reference_k_is_the_oracle_k():
    for rows, cols in ((1, 1), (203, 317), (1080, 1920), (2160, 3840), (4321, 7777)):
        assert ref.defocus_kernel_size(rows, cols) == ob.defocus_kernel_size(rows, cols)


def test_argument_errors_without_a_device():
    from realtimedepthdiffusion_b200 import _native
    lib = _native.lib
    assert lib.rtdd_refocus(None, None, 0, None, 0, None, 0, 1, 1, 0.0, 0.0, -1) == -1
    assert lib.rtdd_refocus(None, None, 0, None, 0, None, 0, 1, 1, float("nan"), -1.0, 5000) == -1
    assert lib.rtdd_frame_refocus(None, None, 0, -1, -1, 0.0, 0.0, -1) == -1
    assert lib.rtdd_frame_refocus(None, None, 0, 3, 4, 0.0, 0.0, 5000) == -1
