"""Host-side mirror of the reference's operator interface for the hot path.

`DepthDiffusion` wraps one rtdd_ctx (one per GPU).  Method names follow the
reference's free functions (ref: include/GPUSolver.h:6-10,
include/GPUImageProcessing.h:4-10, include/GPUDepthEffect.h:4-9): same argument
meaning, device planes with byte pitches; errors raise RtddError instead of the
reference's print-and-continue (the C++ shims keep that convention).
"""
import ctypes as C

import torch

from . import _native
from ._native import lib


class RtddError(RuntimeError):
    pass


def pyramid_levels(rows, cols):
    """ref: src/main.cpp:95"""
    return int(lib.rtdd_pyramid_levels(rows, cols))


def level_iterations(max_iterations, levels, level):
    """ref: src/main.cpp:263"""
    return int(lib.rtdd_level_iterations(max_iterations, levels, level))


def level_sizes(rows, cols, levels):
    """Floor sizes of the depth/scribble planes (ref: src/main.cpp:103, src/GPUSolver.cu:42-43)."""
    return [(int(rows / 2.0 ** l), int(cols / 2.0 ** l)) for l in range(levels)]


from .planes import pitched_empty, to_dev  # noqa: E402,F401


def _ptr(t):
    return C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p(0)


def _pitch(t):
    if t is None:
        return 0
    if t.dim() != 2 or (t.shape[1] > 1 and t.stride(1) != 1):
        raise ValueError("expected a 2-D plane with unit column stride")
    return t.stride(0) * t.element_size()


class DepthDiffusion:
    """One solver context on one GPU (replaces GPUAllocateDeviceMemory/GPUFreeDeviceMemory state)."""

    def __init__(self, rows, cols, levels=None, device=None, beta=0.4, strip=None):
        if not torch.cuda.is_available():
            raise RtddError("no CUDA device: this library has no CPU path")
        self.device = torch.device("cuda", torch.cuda.current_device() if device is None else device)
        self.rows, self.cols = int(rows), int(cols)
        self.levels = pyramid_levels(rows, cols) if levels is None else int(levels)
        h = C.c_void_p()
        if strip is not None:        # (nranks, halo, min_strip_pixels): window-sized planes for the levels a strip frame splits
            rc = lib.rtdd_create_strip(self.rows, self.cols, self.levels, self.device.index, int(strip[0]), int(strip[1]), int(strip[2]), C.byref(h))
        else:
            rc = lib.rtdd_create(self.rows, self.cols, self.levels, self.device.index, C.byref(h))
        if rc != 0:
            raise RtddError("rtdd_create failed with status %d" % rc)
        self._h = h
        self.sizes = level_sizes(self.rows, self.cols, self.levels)
        if beta is not None:
            self.load_weights(beta)

    # -- plumbing -------------------------------------------------------------
    def _ck(self, rc):
        if rc != 0:
            raise RtddError("%s (status %d)" % (lib.rtdd_last_error(self._h).decode(), rc))

    def close(self):
        if getattr(self, "_h", None):
            lib.rtdd_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def sync(self):
        self._ck(lib.rtdd_sync(self._h))

    def set_stream(self, stream):
        """stream: a torch.cuda.Stream, a raw cudaStream_t int, or None for the context's own stream."""
        raw = 0 if stream is None else (stream.cuda_stream if hasattr(stream, "cuda_stream") else int(stream))
        self._ck(lib.rtdd_set_stream(self._h, C.c_void_p(raw)))

    @property
    def launch_count(self):
        return int(lib.rtdd_launch_count(self._h))

    def set_sweep_variant(self, variant, sweeps_per_pass=0):
        self._ck(lib.rtdd_set_sweep_variant(self._h, variant, sweeps_per_pass))

    def set_tuning(self, key, value):
        self._ck(lib.rtdd_set_tuning(self._h, key.encode(), int(value)))

    def set_pass_plan(self, level, sweeps_of_pass):
        """The caller's own pass lengths for one level of the temporally blocked kernels ([] = back to the planner)."""
        n = len(sweeps_of_pass)
        arr = (C.c_int * max(n, 1))(*sweeps_of_pass)
        self._ck(lib.rtdd_set_pass_plan(self._h, int(level), arr, n))

    @staticmethod
    def plan_passes(rows, cols, iterations, sm_count=148, host_map=False, throughput=False):
        """(pass lengths, form) the level driver would use (host only); form: 1 = clusters of two CTAs on 128x128 regions,
        0 = single CTAs on 128x64 regions, 2 = single CTAs on 128x32 regions."""
        arr = (C.c_int * max(iterations, 1))()
        form = C.c_int()
        n = lib.rtdd_plan_passes(rows, cols, iterations, sm_count, (1 if host_map else 0) | (2 if throughput else 0), arr, max(iterations, 1), C.byref(form))
        if n < 0:
            raise ValueError("rtdd_plan_passes: %d" % n)
        return list(arr[:n]), int(form.value)

    # -- GPUSolver -------------------------------------------------------------
    def load_weights(self, beta):
        self._ck(lib.rtdd_load_weights(self._h, beta))

    def matrix_free_solver(self, depth, scribble, gray, max_iterations, level):
        """GPUMatrixFreeSolver: one level, `depth` (fp32 plane) updated in place."""
        rows, cols = depth.shape
        self._ck(lib.rtdd_solve_level(self._h, _ptr(depth), _pitch(depth), _ptr(scribble), _pitch(scribble),
                                      _ptr(gray), _pitch(gray), rows, cols, int(max_iterations), int(level)))

    def level_sweep_ms(self, level):
        """(ms, sweeps, kernel launches) of the most recent solve of `level` (device time, CUDA events)."""
        ms, it, k = C.c_float(), C.c_int(), C.c_int()
        self._ck(lib.rtdd_level_sweep_ms(self._h, int(level), C.byref(ms), C.byref(it), C.byref(k)))
        return ms.value, it.value, k.value

    def level_residual(self, level):
        r = C.c_float()
        self._ck(lib.rtdd_level_residual(self._h, int(level), C.byref(r)))
        return r.value

    def matrix_free_solver_converge(self, depth, scribble, gray, max_iterations, tolerance, level, check_every=8):
        """Extension: GPUMatrixFreeSolver honouring `tolerance`.  Returns (sweeps run, final residual)."""
        rows, cols = depth.shape
        it, res = C.c_int(), C.c_float()
        self._ck(lib.rtdd_solve_level_converge(self._h, _ptr(depth), _pitch(depth), _ptr(scribble), _pitch(scribble), _ptr(gray), _pitch(gray),
                                               rows, cols, int(max_iterations), float(tolerance), int(check_every), int(level),
                                               C.byref(it), C.byref(res)))
        return it.value, res.value

    def frame_solve_incremental(self, max_iterations, coarsest_level):
        self._ck(lib.rtdd_frame_solve_incremental(self._h, int(max_iterations), int(coarsest_level)))

    def frame_solve_band(self, max_iterations, row_begin, row_end, dilation=48):
        """Extension (not parity): re-solve only a band of rows around an edit; see rtdd_frame_solve_band."""
        self._ck(lib.rtdd_frame_solve_band(self._h, int(max_iterations), int(row_begin), int(row_end), int(dilation)))

    def selftest_division(self, n, seed=1, mode=0):
        mism = C.c_ulonglong(0)
        self._ck(lib.rtdd_selftest_division(self._h, int(n), int(seed), int(mode), C.byref(mism)))
        return mism.value

    def edge_weights_only(self, depth, gray, level):
        """The edge-weight pass without exporting the link planes (timing)."""
        rows, cols = depth.shape
        self._ck(lib.rtdd_edge_weights(self._h, _ptr(depth), _pitch(depth), _ptr(gray), _pitch(gray), rows, cols, int(level),
                                       C.c_void_p(0), C.c_void_p(0), 0))

    def edge_weights(self, depth, gray, level):
        rows, cols = depth.shape
        right = pitched_empty(rows, cols, torch.uint8, self.device)
        down = pitched_empty(rows, cols, torch.uint8, self.device)
        self._ck(lib.rtdd_edge_weights(self._h, _ptr(depth), _pitch(depth), _ptr(gray), _pitch(gray), rows, cols, int(level),
                                       _ptr(right), _ptr(down), _pitch(right)))
        return right, down

    # -- GPUImageProcessing ------------------------------------------------------
    def convert_to_float(self, src, dst, mask):
        rows, cols = dst.shape
        self._ck(lib.rtdd_convert_to_float(self._h, _ptr(src), _pitch(src), _ptr(dst), _pitch(dst), _ptr(mask), _pitch(mask), rows, cols))

    def pyrdown_annotation(self, prev_scribble, prev_edited, curr_scribble, curr_edited):
        pr, pc = prev_scribble.shape
        cr, cc = curr_scribble.shape
        self._ck(lib.rtdd_pyrdown_annotation(self._h, _ptr(prev_scribble), _pitch(prev_scribble), _ptr(prev_edited), _pitch(prev_edited), pr, pc,
                                             _ptr(curr_scribble), _pitch(curr_scribble), _ptr(curr_edited), _pitch(curr_edited), cr, cc))

    def paint_image(self, x, y, color, radius, edited, scribble):
        rows, cols = scribble.shape
        self._ck(lib.rtdd_paint(self._h, int(x), int(y), int(color), int(radius), _ptr(edited), _pitch(edited),
                                _ptr(scribble), _pitch(scribble), rows, cols))

    # -- GPUDepthEffect ----------------------------------------------------------
    def simulate_desaturation(self, orig, gray, depth, out):
        rows, cols = depth.shape
        self._ck(lib.rtdd_desaturate(self._h, _ptr(orig), _pitch(orig), _ptr(gray), _pitch(gray), _ptr(depth), _pitch(depth),
                                     _ptr(out), _pitch(out), rows, cols))

    def simulate_haze(self, orig, depth, out):
        rows, cols = depth.shape
        self._ck(lib.rtdd_haze(self._h, _ptr(orig), _pitch(orig), _ptr(depth), _pitch(depth), _ptr(out), _pitch(out), rows, cols))

    def simulate_defocus(self, orig, depth, out):
        rows, cols = depth.shape
        self._ck(lib.rtdd_defocus(self._h, _ptr(orig), _pitch(orig), _ptr(depth), _pitch(depth), _ptr(out), _pitch(out), rows, cols))

    def effects_fused(self, orig, gray, depth, desat, haze, defocus):
        rows, cols = depth.shape
        self._ck(lib.rtdd_effects_fused(self._h, _ptr(orig), _pitch(orig), _ptr(gray), _pitch(gray), _ptr(depth), _pitch(depth),
                                        _ptr(desat), _pitch(desat), _ptr(haze), _pitch(haze), _ptr(defocus), _pitch(defocus), rows, cols))

    def refocus(self, orig, depth, out, focus_depth, depth_of_field=0.0, aperture=None):
        """Extension (no reference counterpart): depth-of-field blur of `orig` by `depth` with the sharp band
        [focus_depth - depth_of_field, focus_depth + depth_of_field] and a box of at most `aperture` pixels a side
        (None = the reference defocus's K for the image size).  See rtdd_refocus in include/rtdd.h."""
        rows, cols = depth.shape
        self._ck(lib.rtdd_refocus(self._h, _ptr(orig), _pitch(orig), _ptr(depth), _pitch(depth), _ptr(out), _pitch(out), rows, cols,
                                  float(focus_depth), float(depth_of_field), -1 if aperture is None else int(aperture)))

    def stereo(self, orig, depth, left=None, right=None, anaglyph=None, convergence_depth=0.0, max_disparity=32):
        """Extension (no reference counterpart): left and right views of `orig` by `depth` (0 near, 255 far) and their red-cyan
        anaglyph, into device BGR planes, any of them None but not all.  Depth `convergence_depth` sits on the screen; depths 255
        away from it get `max_disparity` pixels of parallax.  Side by side: left = buf[:, :3*cols], right = buf[:, 3*cols:] of one
        rows x 6*cols plane.  See rtdd_stereo in include/rtdd.h."""
        rows, cols = depth.shape
        self._ck(lib.rtdd_stereo(self._h, _ptr(orig), _pitch(orig), _ptr(depth), _pitch(depth), _ptr(left), _pitch(left),
                                 _ptr(right), _pitch(right), _ptr(anaglyph), _pitch(anaglyph), rows, cols,
                                 float(convergence_depth), int(max_disparity)))

    # -- pyramid ops ---------------------------------------------------------------
    def bgr2gray(self, bgr, gray):
        rows, cols = gray.shape
        self._ck(lib.rtdd_bgr2gray(self._h, _ptr(bgr), _pitch(bgr), _ptr(gray), _pitch(gray), rows, cols))

    def pyrdown_gray(self, src, dst):
        rows, cols = src.shape
        assert dst.shape == ((rows + 1) // 2, (cols + 1) // 2)
        self._ck(lib.rtdd_pyrdown_gray(self._h, _ptr(src), _pitch(src), rows, cols, _ptr(dst), _pitch(dst)))

    def pyrup_depth(self, src, dst):
        self._ck(lib.rtdd_pyrup_depth(self._h, _ptr(src), _pitch(src), src.shape[0], src.shape[1], _ptr(dst), _pitch(dst), dst.shape[0], dst.shape[1]))

    def quantise_u8(self, src, dst):
        rows, cols = src.shape
        self._ck(lib.rtdd_quantise_u8(self._h, _ptr(src), _pitch(src), _ptr(dst), _pitch(dst), rows, cols))

    # -- whole frame (main.cpp:232-295) -----------------------------------------------
    def frame_set_image(self, bgr_host, sync=True):
        """bgr_host: uint8 numpy array or CPU tensor, rows x cols x 3, C-contiguous.  sync=False leaves the upload and the
        gray pyramid in flight on the context stream (the caller keeps bgr_host alive and unchanged until it synchronises)."""
        t = torch.as_tensor(bgr_host)
        assert t.dtype == torch.uint8 and tuple(t.shape) == (self.rows, self.cols, 3) and t.is_contiguous()
        self._keep_bgr = t
        self._ck(lib.rtdd_frame_set_image(self._h, C.c_void_p(t.data_ptr()), self.cols * 3))
        if sync:
            self.sync()

    def frame_read_depth_u8(self, depth_u8_host, sync=True):
        d = torch.as_tensor(depth_u8_host)
        assert d.dtype == torch.uint8 and tuple(d.shape) == (self.rows, self.cols) and d.is_contiguous()
        self._ck(lib.rtdd_frame_read_depth_u8(self._h, C.c_void_p(d.data_ptr()), self.cols, 1 if sync else 0))
        return d

    def _host_map(self, depth_u8_host):
        """The caller's 8-bit map: a [rows, cols] u8 host plane, rows possibly pitched.  In pinned memory with a 4-byte aligned base
        and pitch the last sweep pass stores it itself (rtdd.h, "zero_copy_out")."""
        if depth_u8_host is None:
            return None, self.cols
        d = torch.as_tensor(depth_u8_host)
        assert d.dtype == torch.uint8 and tuple(d.shape) == (self.rows, self.cols) and d.stride(1) == 1 and d.stride(0) >= self.cols
        return d, d.stride(0)

    def frame_solve_host(self, scribble_host, edited_host, max_iterations=1000, depth_u8_host=None):
        s = torch.as_tensor(scribble_host)
        e = torch.as_tensor(edited_host)
        assert s.dtype == torch.uint8 and tuple(s.shape) == (self.rows, self.cols) and s.is_contiguous()
        assert e.dtype == torch.uint8 and tuple(e.shape) == (self.rows, self.cols, 3) and e.is_contiguous()
        d, dp = self._host_map(depth_u8_host)
        self._ck(lib.rtdd_frame_solve_host(self._h, C.c_void_p(s.data_ptr()), self.cols, C.c_void_p(e.data_ptr()), self.cols * 3,
                                           int(max_iterations), C.c_void_p(d.data_ptr()) if d is not None else C.c_void_p(0), dp))
        return d

    def frame_solve_host_annotation(self, annotation_host, max_iterations=1000, depth_u8_host=None):
        """One frame from the reference's annotation format (ONE u8 plane, 32 = not annotated; ref: src/main.cpp:160-170)."""
        a = torch.as_tensor(annotation_host)
        assert a.dtype == torch.uint8 and tuple(a.shape) == (self.rows, self.cols) and a.is_contiguous()
        d, dp = self._host_map(depth_u8_host)
        self._ck(lib.rtdd_frame_solve_host_annotation(self._h, C.c_void_p(a.data_ptr()), self.cols, int(max_iterations),
                                                      C.c_void_p(d.data_ptr()) if d is not None else C.c_void_p(0), dp))
        return d

    def annotation_ingest(self, annotation, bgr, edited, scribble):
        """Device planes: annotation [rows, cols] u8, bgr / edited [rows, 3*cols] u8, scribble [rows, cols] u8."""
        rows, cols = scribble.shape
        self._ck(lib.rtdd_annotation_ingest(self._h, _ptr(annotation), _pitch(annotation), _ptr(bgr), _pitch(bgr), _ptr(edited), _pitch(edited),
                                            _ptr(scribble), _pitch(scribble), rows, cols))

    def frame_solve(self, max_iterations=1000):
        self._ck(lib.rtdd_frame_solve(self._h, int(max_iterations)))

    def frame_solve_download(self, depth_u8_host, max_iterations=1000):
        """The live loop's frame: strokes already painted on the device (frame_paint), 8-bit map into host memory."""
        d, dp = self._host_map(depth_u8_host)
        self._ck(lib.rtdd_frame_solve_download(self._h, int(max_iterations), C.c_void_p(d.data_ptr()), dp))
        return d

    def frame_paint(self, x, y, color, radius):
        self._ck(lib.rtdd_frame_paint(self._h, int(x), int(y), int(color), int(radius)))

    def frame_effects(self, desat=None, haze=None, defocus=None):
        """GPUSimulateDesaturation / Haze / Defocus on the frame's own image and solved depth (ref: src/main.cpp:190-230);
        outputs are device BGR planes, any may be None.  The defocus summed-area table is cached per image."""
        self._ck(lib.rtdd_frame_effects(self._h, _ptr(desat), _pitch(desat), _ptr(haze), _pitch(haze), _ptr(defocus), _pitch(defocus)))

    def frame_refocus(self, out, focus_point=None, focus_depth=None, depth_of_field=0.0, aperture=None):
        """refocus() of the frame's own image by its solved depth into the device BGR plane `out`, with the summed-area table
        cached per image.  Give exactly one of focus_point = (x, y), whose depth is read on the GPU (no host round trip, so a
        captured graph follows later solves), and focus_depth."""
        if (focus_point is None) == (focus_depth is None):
            raise ValueError("frame_refocus: give exactly one of focus_point and focus_depth")
        if focus_point is None:
            fx, fy, fd = -1, -1, float(focus_depth)
        else:                 # NaN: a point of (-1, -1) is refused like any other point outside the image
            fx, fy, fd = int(focus_point[0]), int(focus_point[1]), float("nan")
        self._ck(lib.rtdd_frame_refocus(self._h, _ptr(out), _pitch(out), fx, fy, fd, float(depth_of_field),
                                        -1 if aperture is None else int(aperture)))

    def frame_stereo(self, left=None, right=None, anaglyph=None, convergence_point=None, convergence_depth=None, max_disparity=32):
        """stereo() of the frame's own image by its solved depth.  Give exactly one of convergence_point = (x, y), whose depth is
        read on the GPU (no host round trip, so a captured graph follows later solves), and convergence_depth."""
        if (convergence_point is None) == (convergence_depth is None):
            raise ValueError("frame_stereo: give exactly one of convergence_point and convergence_depth")
        if convergence_point is None:
            cx, cy, cd = -1, -1, float(convergence_depth)
        else:                 # NaN: a point of (-1, -1) is refused like any other point outside the image
            cx, cy, cd = int(convergence_point[0]), int(convergence_point[1]), float("nan")
        self._ck(lib.rtdd_frame_stereo(self._h, _ptr(left), _pitch(left), _ptr(right), _pitch(right), _ptr(anaglyph), _pitch(anaglyph),
                                       cx, cy, cd, int(max_disparity)))

    PLANE_DEPTH, PLANE_GRAY, PLANE_SCRIBBLE, PLANE_EDITED, PLANE_BGR, PLANE_DEPTH_U8 = range(6)

    def frame_plane(self, which, level=0):
        """Copy of a context-owned plane as a dense torch tensor (for tests / downloads)."""
        p, pitch, r, c = C.c_void_p(), C.c_size_t(), C.c_int(), C.c_int()
        self._ck(lib.rtdd_frame_plane(self._h, which, level, C.byref(p), C.byref(pitch), C.byref(r), C.byref(c)))
        dtype = torch.float32 if which == self.PLANE_DEPTH else torch.uint8
        ch = 3 if which in (self.PLANE_EDITED, self.PLANE_BGR) else 1
        item = 4 if dtype == torch.float32 else 1
        out = torch.empty((r.value, c.value * ch), dtype=dtype, device=self.device)
        self.sync()
        _cudart_memcpy2d(out, p.value, pitch.value, c.value * ch * item, r.value)
        return out


def _cudart_memcpy2d(dst, src_ptr, src_pitch, width_bytes, rows):
    """Device-to-device copy of a pitched plane at a raw pointer into the dense tensor `dst`."""

    class _Holder:
        pass

    h = _Holder()
    h.__cuda_array_interface__ = {"shape": (src_pitch * rows,), "typestr": "|u1", "data": (src_ptr, False), "version": 2}
    flat = torch.as_tensor(h, device=dst.device)
    dst.view(torch.uint8).view(rows, -1).copy_(flat.view(rows, src_pitch)[:, :width_bytes])
    torch.cuda.synchronize(dst.device)
