"""ctypes binding of librtdd.so (the C ABI of include/rtdd.h).

There is no fallback: if the shared library has not been built, importing this
module raises.  Build it with `python -m realtimedepthdiffusion_b200.build` or
`__graft_entry__.build()`.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "librtdd.so")

if not os.path.exists(LIB_PATH):
    raise ImportError(
        "librtdd.so is missing (%s): build the CUDA extension first "
        "(python realtimedepthdiffusion_b200/build.py); there is no CPU fallback" % LIB_PATH)

lib = C.CDLL(LIB_PATH, mode=os.RTLD_LOCAL | os.RTLD_NOW)

vp, sz, i32, f32 = C.c_void_p, C.c_size_t, C.c_int, C.c_float

# name -> (restype, argtypes); every symbol include/rtdd.h declares
SIGNATURES = {
    "rtdd_create": (i32, [i32, i32, i32, i32, C.POINTER(vp)]),
    "rtdd_create_strip": (i32, [i32, i32, i32, i32, i32, i32, C.c_longlong, C.POINTER(vp)]),
    "rtdd_destroy": (i32, [vp]),
    "rtdd_load_weights": (i32, [vp, f32]),
    "rtdd_set_stream": (i32, [vp, vp]),
    "rtdd_sync": (i32, [vp]),
    "rtdd_last_error": (C.c_char_p, [vp]),
    "rtdd_launch_count": (C.c_ulonglong, [vp]),
    "rtdd_levels": (i32, [vp]),
    "rtdd_pyramid_levels": (i32, [i32, i32]),
    "rtdd_level_iterations": (i32, [i32, i32, i32]),
    "rtdd_solve_level": (i32, [vp, vp, sz, vp, sz, vp, sz, i32, i32, i32, i32]),
    "rtdd_edge_weights": (i32, [vp, vp, sz, vp, sz, i32, i32, i32, vp, vp, sz]),
    "rtdd_level_sweep_ms": (i32, [vp, i32, C.POINTER(f32), C.POINTER(i32), C.POINTER(i32)]),
    "rtdd_level_residual": (i32, [vp, i32, C.POINTER(f32)]),
    "rtdd_solve_level_converge": (i32, [vp, vp, sz, vp, sz, vp, sz, i32, i32, i32, f32, i32, i32, C.POINTER(i32), C.POINTER(f32)]),
    "rtdd_frame_solve_incremental": (i32, [vp, i32, i32]),
    "rtdd_frame_solve_download": (i32, [vp, i32, vp, sz]),
    "rtdd_frame_solve_band": (i32, [vp, i32, i32, i32, i32]),
    "rtdd_selftest_division": (i32, [vp, C.c_ulonglong, C.c_ulonglong, i32, C.POINTER(C.c_ulonglong)]),
    "rtdd_strip_init": (i32, [vp, i32, vp, sz, vp, sz, vp, sz, i32, i32, i32, i32]),
    "rtdd_strip_pass": (i32, [vp, i32, i32, i32, i32]),
    "rtdd_strip_planes": (i32, [vp, i32, C.POINTER(vp), C.POINTER(vp), C.POINTER(sz), C.POINTER(i32), C.POINTER(i32)]),
    "rtdd_strip_finish": (i32, [vp, i32, vp, sz, i32, i32]),
    "rtdd_ipc_export": (i32, [vp, vp]),
    "rtdd_ipc_import": (i32, [vp, vp, C.POINTER(vp)]),
    "rtdd_arena": (i32, [vp, C.POINTER(vp), C.POINTER(sz)]),
    "rtdd_strip_set_peers": (i32, [vp, vp, vp]),
    "rtdd_strip_neighbours": (i32, [vp, i32, i32, i32, i32, i32, i32]),
    "rtdd_strip_wait": (i32, [vp, i32]),
    "rtdd_plan_strips": (i32, [vp, vp, i32, i32, i32, C.c_longlong, vp, vp, vp]),
    "rtdd_strip_schedule": (i32, [i32, i32, i32, i32, vp, vp, i32]),
    "rtdd_plan_strip_planes": (i32, [vp, vp, i32, i32, i32, C.c_longlong, vp]),
    "rtdd_plan_blocked": (i32, [i32, i32, i32, i32, C.POINTER(i32), C.POINTER(i32)]),
    "rtdd_plan_passes": (i32, [i32, i32, i32, i32, i32, C.POINTER(i32), i32, C.POINTER(i32)]),
    "rtdd_set_pass_plan": (i32, [vp, i32, C.POINTER(i32), i32]),
    "rtdd_strip_push": (i32, [vp, i32]),
    "rtdd_strip_pull": (i32, [vp, i32]),
    "rtdd_strip_push_enable": (i32, [vp, i32, i32]),
    "rtdd_pyrup_depth_rows": (i32, [vp, vp, sz, i32, i32, vp, sz, i32, i32, i32, i32]),
    "rtdd_set_tuning": (i32, [vp, C.c_char_p, i32]),
    "rtdd_set_sweep_variant": (i32, [vp, i32, i32]),
    "rtdd_convert_to_float": (i32, [vp, vp, sz, vp, sz, vp, sz, i32, i32]),
    "rtdd_pyrdown_annotation": (i32, [vp, vp, sz, vp, sz, i32, i32, vp, sz, vp, sz, i32, i32]),
    "rtdd_paint": (i32, [vp, i32, i32, i32, i32, vp, sz, vp, sz, i32, i32]),
    "rtdd_desaturate": (i32, [vp, vp, sz, vp, sz, vp, sz, vp, sz, i32, i32]),
    "rtdd_haze": (i32, [vp, vp, sz, vp, sz, vp, sz, i32, i32]),
    "rtdd_defocus": (i32, [vp, vp, sz, vp, sz, vp, sz, i32, i32]),
    "rtdd_effects_fused": (i32, [vp, vp, sz, vp, sz, vp, sz, vp, sz, vp, sz, vp, sz, i32, i32]),
    "rtdd_refocus": (i32, [vp, vp, sz, vp, sz, vp, sz, i32, i32, f32, f32, i32]),
    "rtdd_frame_refocus": (i32, [vp, vp, sz, i32, i32, f32, f32, i32]),
    "rtdd_stereo": (i32, [vp, vp, sz, vp, sz, vp, sz, vp, sz, vp, sz, i32, i32, f32, i32]),
    "rtdd_frame_stereo": (i32, [vp, vp, sz, vp, sz, vp, sz, i32, i32, f32, i32]),
    "rtdd_bgr2gray": (i32, [vp, vp, sz, vp, sz, i32, i32]),
    "rtdd_pyrdown_gray": (i32, [vp, vp, sz, i32, i32, vp, sz]),
    "rtdd_pyrup_depth": (i32, [vp, vp, sz, i32, i32, vp, sz, i32, i32]),
    "rtdd_quantise_u8": (i32, [vp, vp, sz, vp, sz, i32, i32]),
    "rtdd_frame_set_image": (i32, [vp, vp, sz]),
    "rtdd_frame_solve_host": (i32, [vp, vp, sz, vp, sz, i32, vp, sz]),
    "rtdd_frame_solve": (i32, [vp, i32]),
    "rtdd_frame_read_depth_u8": (i32, [vp, vp, sz, i32]),
    "rtdd_frame_solve_host_annotation": (i32, [vp, vp, sz, i32, vp, sz]),
    "rtdd_annotation_ingest": (i32, [vp, vp, sz, vp, sz, vp, sz, vp, sz, i32, i32]),
    "rtdd_frame_paint": (i32, [vp, i32, i32, i32, i32]),
    "rtdd_frame_plane": (i32, [vp, i32, i32, C.POINTER(vp), C.POINTER(sz), C.POINTER(i32), C.POINTER(i32)]),
    "rtdd_frame_effects": (i32, [vp, vp, sz, vp, sz, vp, sz]),
    "rtdd_frame_set_image_device": (i32, [vp, vp, sz]),
    "rtdd_strip_pass_to": (i32, [vp, i32, i32, i32, i32, vp, sz, vp, sz]),
    "rtdd_effects_rows": (i32, [vp, vp, sz, vp, sz, vp, sz, vp, sz, vp, sz, vp, sz, i32, i32, i32, i32]),
    "rtdd_strip_frame_setup": (i32, [vp, i32, i32, i32, i32, C.c_longlong]),
    "rtdd_strip_frame_solve": (i32, [vp, i32]),
    "rtdd_strip_frame_level0": (i32, [vp, i32]),
    "rtdd_strip_frame_rows": (i32, [vp, i32, C.POINTER(i32), C.POINTER(i32), C.POINTER(i32), C.POINTER(i32), C.POINTER(i32)]),
    "rtdd_strip_frame_effects": (i32, [vp, vp, sz, vp, sz, vp, sz]),
    "rtdd_mgpu_create": (i32, [vp, i32, i32, i32, i32, f32, i32, i32, C.c_longlong, C.POINTER(vp)]),
    "rtdd_mgpu_destroy": (i32, [vp]),
    "rtdd_mgpu_devices": (i32, [vp]),
    "rtdd_mgpu_last_error": (C.c_char_p, [vp]),
    "rtdd_mgpu_context": (vp, [vp, i32]),
    "rtdd_mgpu_set_image": (i32, [vp, vp, sz]),
    "rtdd_mgpu_frame_solve_host_annotation": (i32, [vp, vp, sz, i32, vp, sz, C.POINTER(f32)]),
    "rtdd_mgpu_frame_solve": (i32, [vp, i32, C.POINTER(f32)]),
    "rtdd_mgpu_level0": (i32, [vp, i32, C.POINTER(f32)]),
    "rtdd_mgpu_batch_solve": (i32, [vp, i32, vp, sz, vp, sz, i32, vp, sz, C.POINTER(f32)]),
}

from .refnames import SHIM_SIGNATURES, SHIM_SYMBOLS, bind_reference_api  # noqa: E402,F401

for _name, (_res, _args) in SIGNATURES.items():
    _fn = getattr(lib, _name)
    _fn.restype = _res
    _fn.argtypes = _args

shims = bind_reference_api(lib)
