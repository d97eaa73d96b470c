"""The C-ABI library loads and exports every symbol include/rtdd.h declares, and the ten
reference-named C++ functions with the reference's exact (mangled) signatures.  No compute."""
import ctypes
import os
import re

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def declared_symbols():
    txt = open(os.path.join(ROOT, "include", "rtdd.h")).read()
    txt = re.sub(r"/\*.*?\*/", "", txt, flags=re.S)
    return sorted(set(re.findall(r"\b(rtdd_[a-z0-9_]+)\s*\(", txt)))


def test_every_declared_symbol_is_exported():
    from realtimedepthdiffusion_b200 import _native
    names = declared_symbols()
    assert len(names) >= 25
    for n in names:
        assert hasattr(_native.lib, n), n
        assert n in _native.SIGNATURES, "python binding lacks %s" % n
    assert sorted(_native.SIGNATURES) == names


def test_reference_named_functions_are_exported():
    from realtimedepthdiffusion_b200 import _native
    for name, sym in _native.SHIM_SYMBOLS.items():
        assert hasattr(_native.lib, sym), name


def test_reference_headers_declare_the_same_ten_functions():
    ours = set()
    for h in ("GPUSolver.h", "GPUImageProcessing.h", "GPUDepthEffect.h"):
        txt = open(os.path.join(ROOT, "include", h)).read()
        ours |= set(re.findall(r"^void\s+(GPU\w+)\s*\(", txt, flags=re.M))
    from realtimedepthdiffusion_b200 import _native
    assert ours == set(_native.SHIM_SYMBOLS)


def test_libref_exports_identical_mangled_names():
    """The mangled names the reference's own library exports (tests/golden/ref_ab.json) are the ones we bind and ship."""
    from realtimedepthdiffusion_b200 import _native
    from tests.harness import reference_golden
    ref_symbols = reference_golden("symbols")
    assert sorted(_native.SHIM_SYMBOLS.values()) == sorted(ref_symbols)
    out = os.popen("nm -D --defined-only %s" % _native.LIB_PATH).read()
    for sym in ref_symbols:
        assert re.search(r"\b%s\b" % sym, out), sym


def test_host_helpers_without_a_gpu():
    from realtimedepthdiffusion_b200 import _native
    lib = _native.lib
    # SURVEY.md section 6 table (src/main.cpp:95,263)
    assert lib.rtdd_pyramid_levels(1080, 1920) == 5
    assert lib.rtdd_pyramid_levels(2160, 3840) == 6
    assert lib.rtdd_pyramid_levels(16384, 16384) == 9
    assert lib.rtdd_pyramid_levels(624, 672) == 4
    assert lib.rtdd_pyramid_levels(10, 10) == 1
    assert [lib.rtdd_level_iterations(1000, 6, l) for l in range(6)] == [31, 62, 125, 250, 500, 1000]
    assert [lib.rtdd_level_iterations(1000, 9, l) for l in range(9)] == [3, 7, 15, 31, 62, 125, 250, 500, 1000]
    # argument errors are reported without touching a device
    assert lib.rtdd_create(0, 10, 1, -1, ctypes.byref(ctypes.c_void_p())) == -1
    assert lib.rtdd_destroy(None) == -1
    assert lib.rtdd_solve_level(None, None, 0, None, 0, None, 0, 1, 1, 1, 0) == -1
