"""GPU tests of the depth effects and refocus at every form of the summed-area table they read (launch_sat_build in
csrc/effect_kernels.cu, chosen by image width): sat_fused_kernel<1> up to 4096 columns, <2> up to 8192, <4> up to 16384, and the
two-pass sat_rows_kernel + sat_cols_kernel beyond that.  The shapes sit on both sides of every 4096-column chunk edge and of the
16-row groups (SAT_G), and include tall narrow images whose hundreds of groups sat_aux_kernel splits unevenly across its warps.
The table is exact integers, so every output is compared byte for byte: defocus and desaturation with the CPU oracle, haze with it
within 1 grey level on < 0.1 % of values (glibc expf vs libdevice expf), refocus with tests/refocus_reference.py.  Also covered:
misaligned planes (byte loads in the table build, the effects' scalar path), row strips whose table starts below row 0 of the
image, the frame forms with their cached table, and the launch count of every call (the table costs 4 launches, 5 beyond 16384
columns).

The depth recipe makes one wrong table entry visible: most pixels get a box half-side of 0..3, so their windows are 2x2 to 6x6 and
an error in one corner changes the floor of the mean; about 1 % get a uniform depth in [0, 255], whose windows cross chunk and group
edges; row 0 holds NaN, -7, -0.0, 255 and 262.5; and on the two widest shapes of >= 33 rows a few pixels get a depth far beyond 255,
so their clipped windows exceed 65 793 pixels and defocus replays the reference's raster fp32 sums on a wide image."""
import ctypes as C
import functools

import numpy as np
import pytest
import torch

from oracle import binding as ob
from tests import refocus_reference as ref
from tests.harness import pitch, ptr, to_dev, to_host
from tests.test_gpu_refocus import clamp_depth

pytestmark = pytest.mark.gpu

SHAPES = [(17, 4095), (16, 4096),                                   # sat_fused_kernel<1>
          (1, 4097), (33, 8191), (2, 8192),                         # <2>
          (17, 8193), (5, 12289), (33, 16383), (47, 16384),         # <4>
          (1, 16385), (33, 20003), (16, 24576),                     # sat_rows_kernel + sat_cols_kernel
          (20000, 5), (4097, 9)]                                    # 1250 and 257 row groups
DEEP = {(47, 16384), (33, 20003)}           # shapes that also get depths far beyond 255 (windows above 65 793 pixels)
EXACT_SUMS = 65793                          # count * 255 < 2^24: the largest window whose fp32 sums the table reproduces
TAP_BUDGET = 3e9                            # total window area the brute-force oracle defocus may gather over the module
_taps = [0]


@pytest.fixture(scope="module")
def rtdd():
    import realtimedepthdiffusion_b200 as pkg
    return pkg


def table_launches(cols):
    return 4 if cols <= 16384 else 5


def window_areas(h, rows, cols):
    """Clipped area of the box [y-h, y+h) x [x-h, x+h) of every pixel (0 where h <= 0: the pixel is copied)."""
    yy, xx = np.indices((rows, cols), dtype=np.int64)
    h = np.maximum(h, 0)
    n = (np.minimum(xx + h, cols) - np.maximum(xx - h, 0)) * (np.minimum(yy + h, rows) - np.maximum(yy - h, 0))
    return np.where(h > 0, n, 0)


def defocus_half_sides(depth, K):
    """h = a / 2 with a = cvt.rzi((double)((float)K * d) / 255), NaN -> 0 (effect_kernels.cu)."""
    q = (np.float32(K) * depth.astype(np.float32)).astype(np.float64) / 255.0
    return np.trunc(np.nan_to_num(q, nan=0.0)).astype(np.int64) // 2


class Case:
    """Random BGR image, its gray plane and the depth recipe of the module docstring; oracle outputs computed once."""

    def __init__(self, rows, cols, seed, uniform):
        rng = np.random.default_rng(seed)
        self.rows, self.cols = rows, cols
        self.K = ob.defocus_kernel_size(rows, cols)
        self.bgr = rng.integers(0, 256, (rows, cols, 3), dtype=np.uint8)
        self.gray = ob.bgr2gray(self.bgr)
        a = rng.integers(0, 8, (rows, cols))                      # box side a = trunc(K d / 255): half-side a // 2 in 0..3
        depth = ((a + rng.uniform(0.1, 0.9, (rows, cols))) * (255.0 / self.K)).astype(np.float32)
        assert np.array_equal(defocus_half_sides(depth, self.K), a // 2)
        m = rng.random((rows, cols)) < uniform
        depth[m] = rng.uniform(0.0, 255.0, int(m.sum())).astype(np.float32)
        self.deep = None
        if (rows, cols) in DEEP:
            n = 20
            ys, xs = rng.integers(1, rows, n), rng.integers(cols // 4, 3 * cols // 4, n)
            depth[ys, xs] = rng.uniform(1200.0, 2000.0, n).astype(np.float32)
            self.deep = (ys, xs)
        special = np.array([np.nan, -7.0, -0.0, 255.0, 262.5], np.float32)
        depth[0, : min(cols, 5)] = special[: min(cols, 5)]
        self.depth = depth
        self.areas = window_areas(defocus_half_sides(depth, self.K), rows, cols)
        if self.deep is not None:
            assert (self.areas[self.deep] > EXACT_SUMS).all()      # the raster fp32 path on a wide image

    @functools.cached_property
    def defocus(self):
        _taps[0] += int(self.areas.sum())
        assert _taps[0] < TAP_BUDGET, "the oracle defocus of this module gathers %d taps" % _taps[0]
        return ob.defocus(self.bgr, self.depth)

    @functools.cached_property
    def desaturate(self):
        return ob.desaturate(self.bgr, self.gray, self.depth)

    @functools.cached_property
    def haze(self):
        return ob.haze(self.bgr, self.depth)


@functools.lru_cache(maxsize=None)
def case(rows, cols, seed=0, uniform=0.01):
    return Case(rows, cols, rows * 100003 + cols + seed, uniform)


def assert_haze(got, want):
    d = got.astype(np.int16) - want.astype(np.int16)
    assert np.abs(d).max() <= 1 and (d != 0).mean() < 1e-3


def refocus_triples(K):
    """(focus, band, aperture): the parity point with defocus, a copy everywhere, the largest aperture, a mid one."""
    return [(0.0, 0.0, K), (100.0, 5.0, 1), (255.0, 0.0, 4096), (128.0, 20.0, 300)]


def zeros_like_bgr(rows, cols):
    return to_dev(np.zeros((rows, cols, 3), np.uint8), 3)


def counted(ctx, call):
    """Kernel launches the context counts for `call`."""
    n0 = ctx.launch_count
    call()
    ctx.sync()
    return ctx.launch_count - n0


@pytest.mark.parametrize("rows,cols", SHAPES)
def test_effects_and_refocus_equal_the_references(rtdd, rows, cols):
    c = case(rows, cols)
    table = table_launches(cols)
    ctx = rtdd.DepthDiffusion(rows, cols, 1)
    o, g, d = to_dev(c.bgr, 3), to_dev(c.gray), to_dev(c.depth)
    sep = [zeros_like_bgr(rows, cols) for _ in range(3)]
    fused = [zeros_like_bgr(rows, cols) for _ in range(3)]
    assert counted(ctx, lambda: ctx.simulate_defocus(o, d, sep[2])) == table + 1
    assert counted(ctx, lambda: ctx.simulate_desaturation(o, g, d, sep[0])) == 1
    assert counted(ctx, lambda: ctx.simulate_haze(o, d, sep[1])) == 1
    assert counted(ctx, lambda: ctx.effects_fused(o, g, d, *fused)) == table + 1
    got = [to_host(t, 3) for t in sep]
    assert np.array_equal(got[2], c.defocus), int((got[2] != c.defocus).any(-1).sum())
    assert np.array_equal(got[0], c.desaturate)
    assert_haze(got[1], c.haze)
    for a, b in zip(sep, fused):
        assert torch.equal(a, b)                                   # fused == separate, bit for bit
    out = zeros_like_bgr(rows, cols)
    for f, w, a in refocus_triples(c.K):
        out.fill_(0)
        assert counted(ctx, lambda: ctx.refocus(o, d, out, f, w, a)) == table + 1
        want = ref.refocus(c.bgr, c.depth, f, w, a)
        got = to_host(out, 3)
        assert np.array_equal(got, want), (f, w, a, int((got != want).any(-1).sum()))
        if a == 4096 and rows >= 33 and cols > 8192:               # windows beyond the fp32-exact range: the u32 divide
            assert (window_areas(ref.half_sides(c.depth, f, w, a), rows, cols) > EXACT_SUMS).any()
    ctx.close()


def shifted(a, offset, row_elems):
    """Device copy of `a` whose rows start `offset` elements past an aligned address, `row_elems` elements apart."""
    a = np.ascontiguousarray(a)
    flat = torch.from_numpy(a.reshape(a.shape[0], -1))
    base = torch.zeros((a.shape[0], row_elems), dtype=flat.dtype, device="cuda")
    view = base[:, offset:offset + flat.shape[1]]
    view.copy_(flat)
    return view


def odd_bytes(a):
    """u8 plane one byte past an aligned address with an odd pitch: every row starts off a 4-byte boundary or on one by turns."""
    width = a[0].size
    return shifted(a, 1, width + 1 if (width + 1) % 2 else width + 2)


def depth_off4(depth):
    """fp32 plane 4 bytes past an aligned address, pitch = 4 mod 16 bytes: 4-byte aligned, never 16-byte aligned."""
    n = depth.shape[1] + 1
    return shifted(depth, 1, n + (1 - n) % 4)


@pytest.mark.parametrize("rows,cols", [(17, 4095), (33, 8193), (33, 20003)])
def test_misaligned_planes_equal_the_aligned_calls(rtdd, rows, cols):
    """One plane at a time off its alignment: orig (the table is built by the byte loads of sat_group_colsums, sat_fused and
    sat_rows; the effects take ALIGNED = false), depth (table vectorised, effects scalar), one output, gray (desaturation)."""
    c = case(rows, cols)
    ctx = rtdd.DepthDiffusion(rows, cols, 1)
    aligned = dict(o=to_dev(c.bgr, 3), g=to_dev(c.gray), d=to_dev(c.depth))
    f, w, a = refocus_triples(c.K)[2]

    def outputs(o, g, d, odd_out):
        new = (lambda: odd_bytes(np.zeros((rows, cols, 3), np.uint8))) if odd_out else (lambda: zeros_like_bgr(rows, cols))
        defocus, desat, refocus = new(), new(), new()
        fused = [zeros_like_bgr(rows, cols), zeros_like_bgr(rows, cols), new()]    # one misaligned output
        ctx.simulate_defocus(o, d, defocus)
        ctx.simulate_desaturation(o, g, d, desat)
        ctx.effects_fused(o, g, d, *fused)
        ctx.refocus(o, d, refocus, f, w, a)
        ctx.sync()
        return [to_host(t, 3) for t in [defocus, desat, refocus] + fused]

    base = outputs(aligned["o"], aligned["g"], aligned["d"], False)
    assert np.array_equal(base[0], c.defocus)
    assert np.array_equal(base[1], c.desaturate)
    assert np.array_equal(base[2], ref.refocus(c.bgr, c.depth, f, w, a))
    assert np.array_equal(base[3], c.desaturate) and np.array_equal(base[5], c.defocus)
    assert_haze(base[4], c.haze)
    for kind in ("orig", "depth", "out", "gray"):
        planes = dict(aligned)
        if kind == "orig":
            planes["o"] = odd_bytes(c.bgr)
        elif kind == "depth":
            planes["d"] = depth_off4(c.depth)
        elif kind == "gray":
            planes["g"] = odd_bytes(c.gray)
        got = outputs(planes["o"], planes["g"], planes["d"], kind == "out")
        for i, (x, y) in enumerate(zip(got, base)):
            assert np.array_equal(x, y), (kind, i, int((x != y).any(-1).sum()))
    ctx.close()


@pytest.mark.parametrize("rows,cols", [(1000, 8193), (1200, 16385)])
def test_row_strips_over_an_offset_table_equal_the_whole_image(rtdd, rows, cols):
    """rtdd_effects_rows in 4 strips: a middle strip's table covers its rows plus K/2 + 8 on each side, so it starts at image row
    satRow0 > 0.  Every subset of outputs; strips byte-equal to the whole-image call, which equals the oracle."""
    c = case(rows, cols, uniform=2e-4)                            # big windows sparse enough for the oracle's tap budget
    from realtimedepthdiffusion_b200._native import lib
    table = table_launches(cols)
    ctx = rtdd.DepthDiffusion(rows, cols, 1)
    o, g, d = to_dev(c.bgr, 3), to_dev(c.gray), to_dev(c.depth)
    whole = [zeros_like_bgr(rows, cols) for _ in range(3)]
    assert counted(ctx, lambda: ctx.effects_fused(o, g, d, *whole)) == table + 1
    bounds = [(k * rows) // 4 for k in range(4)] + [rows]
    for subset in ((1, 1, 1), (0, 0, 1), (1, 0, 0), (0, 1, 1)):
        strips = [zeros_like_bgr(rows, cols) for _ in range(3)]
        args = []
        for use, t in zip(subset, strips):
            args += [C.c_void_p(t.data_ptr()) if use else C.c_void_p(0), pitch(t)]
        # defocus: table + 1 (desaturation and haze ride along when all three are asked for); otherwise 1 per effect
        want_launches = (table + 1 if subset[2] else 0) + (0 if subset == (1, 1, 1) else subset[0] + subset[1])
        for k in range(4):
            n = counted(ctx, lambda: ctx._ck(lib.rtdd_effects_rows(ctx._h, ptr(o), pitch(o), ptr(g), pitch(g), ptr(d), pitch(d), *args,
                                                                   rows, cols, bounds[k], bounds[k + 1])))
            assert n == want_launches, (subset, k)
        for use, a, b in zip(subset, whole, strips):
            if use:
                assert torch.equal(a, b), subset
    got = [to_host(t, 3) for t in whole]
    assert np.array_equal(got[2], c.defocus), int((got[2] != c.defocus).any(-1).sum())
    assert np.array_equal(got[0], c.desaturate)
    assert_haze(got[1], c.haze)
    ctx.close()


def set_frame_depth(ctx, depth):
    """Copy `depth` into the frame context's level-0 depth plane (what a solve would leave there)."""
    from realtimedepthdiffusion_b200._native import lib
    p, pi, r, cc = C.c_void_p(), C.c_size_t(), C.c_int(), C.c_int()
    ctx._ck(lib.rtdd_frame_plane(ctx._h, ctx.PLANE_DEPTH, 0, C.byref(p), C.byref(pi), C.byref(r), C.byref(cc)))
    rows, cols = depth.shape
    assert (r.value, cc.value) == (rows, cols)

    class Plane:
        pass

    plane = Plane()
    plane.__cuda_array_interface__ = {"shape": (rows, cols), "typestr": "<f4", "data": (p.value, False), "strides": (pi.value, 4), "version": 2}
    ctx.sync()
    torch.as_tensor(plane, device="cuda").copy_(torch.from_numpy(depth))
    torch.cuda.synchronize()
    assert np.array_equal(ctx.frame_plane(ctx.PLANE_DEPTH, 0).cpu().numpy().view(np.uint32), depth.view(np.uint32))


@pytest.mark.parametrize("rows,cols", [(33, 8193), (47, 16384), (33, 20003)])
def test_frame_forms_with_the_cached_table(rtdd, rows, cols):
    """rtdd_frame_effects and rtdd_frame_refocus on the frame's own image and level-0 depth: the first call that needs the table
    builds it (table + 1 launches), later ones reuse it (1), and a new image makes the next call build it again."""
    table = table_launches(cols)
    ctx = rtdd.DepthDiffusion(rows, cols, 1)
    first, second = case(rows, cols), case(rows, cols, seed=1)
    x, y = cols // 3, rows // 2

    ctx.frame_set_image(first.bgr)
    set_frame_depth(ctx, first.depth)
    gray = np.ascontiguousarray(ctx.frame_plane(ctx.PLANE_GRAY, 0).cpu().numpy()[:rows, :cols])
    outs = [zeros_like_bgr(rows, cols) for _ in range(3)]
    assert counted(ctx, lambda: ctx.frame_effects(*outs)) == table + 1
    got = [to_host(t, 3) for t in outs]
    assert np.array_equal(got[0], ob.desaturate(first.bgr, gray, first.depth))
    assert_haze(got[1], first.haze)
    assert np.array_equal(got[2], first.defocus)
    only = zeros_like_bgr(rows, cols)
    assert counted(ctx, lambda: ctx.frame_effects(None, None, only)) == 1
    assert np.array_equal(to_host(only, 3), first.defocus)
    out = zeros_like_bgr(rows, cols)
    assert counted(ctx, lambda: ctx.frame_refocus(out, focus_depth=255.0, aperture=4096)) == 1
    assert np.array_equal(to_host(out, 3), ref.refocus(first.bgr, first.depth, 255.0, 0.0, 4096))
    assert counted(ctx, lambda: ctx.frame_refocus(out, focus_point=(x, y), depth_of_field=2.0, aperture=300)) == 1
    assert np.array_equal(to_host(out, 3), ref.refocus(first.bgr, first.depth, clamp_depth(first.depth[y, x]), 2.0, 300))

    ctx.frame_set_image(second.bgr)                               # a new image: the next table user rebuilds it
    set_frame_depth(ctx, second.depth)
    assert counted(ctx, lambda: ctx.frame_refocus(out, focus_point=(x, y), depth_of_field=0.0)) == table + 1
    assert np.array_equal(to_host(out, 3), ref.refocus(second.bgr, second.depth, clamp_depth(second.depth[y, x]), 0.0, second.K))
    assert counted(ctx, lambda: ctx.frame_effects(None, None, only)) == 1
    assert np.array_equal(to_host(only, 3), second.defocus)
    ctx.close()
