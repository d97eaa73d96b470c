"""The drop-in claim from the reference's own language: tests/cpp/main_like.cpp is written only against the three
reference-named headers (like main.cpp).  It must compile and link against librtdd.so without source changes (CPU test)
and, on a GPU, produce the output it produced when linked against the reference's own kernels (tests/golden/ref_ab.json)."""
import os
import re
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SRC = os.path.join(ROOT, "tests", "cpp", "main_like.cpp")
BUILD = os.path.join(ROOT, "tests", "cpp", "_build")
CUDA = os.environ.get("CUDA_HOME", "/usr/local/cuda")


def build(tag, libdir, lib):
    os.makedirs(BUILD, exist_ok=True)
    out = os.path.join(BUILD, "main_like_" + tag)
    cmd = ["g++", "-std=c++17", "-O1", SRC, "-I", os.path.join(ROOT, "include"), "-I", os.path.join(CUDA, "include"),
           "-L", libdir, "-l" + lib, "-L", os.path.join(CUDA, "lib64"), "-lcudart", "-Wl,-rpath," + libdir, "-o", out]
    r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    assert r.returncode == 0, r.stdout
    return out


def test_main_like_links_against_librtdd_unchanged():
    exe = build("rtdd", os.path.join(ROOT, "realtimedepthdiffusion_b200", "lib"), "rtdd")
    undefined = subprocess.run(["nm", "-u", "-C", exe], stdout=subprocess.PIPE, text=True).stdout
    for fn in ("GPUAllocateDeviceMemory", "GPUFreeDeviceMemory", "GPULoadWeights", "GPUMatrixFreeSolver", "GPUConvertToFloat",
               "GPUPyrDownAnnotation", "GPUPaintImage", "GPUSimulateDefocus", "GPUSimulateDesaturation", "GPUSimulateHaze"):
        assert re.search(r"\b%s\(" % fn, undefined), fn        # resolved at load time from librtdd.so


def main_like_line(tag, libdir, lib, rows, cols, iters):
    """The checksum line main_like prints when linked against lib<lib>.so in `libdir`."""
    exe = build(tag, libdir, lib)
    r = subprocess.run([exe, str(rows), str(cols), str(iters)], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=280)
    assert r.returncode == 0, r.stdout
    return [ln for ln in r.stdout.splitlines() if ln.startswith("levels")][-1]


@pytest.mark.gpu
@pytest.mark.parametrize("rows,cols,iters", [(203, 317, 100), (624, 672, 1000)])
def test_main_like_same_output_with_reference_kernels_and_with_librtdd(rows, cols, iters):
    """Linked against librtdd.so, main_like prints the line it printed when linked against the reference's own kernels
    (tests/golden/ref_ab.json)."""
    from tests.harness import reference_golden
    want = reference_golden("main_like")["%dx%dx%d" % (rows, cols, iters)]
    assert main_like_line("rtdd", os.path.join(ROOT, "realtimedepthdiffusion_b200", "lib"), "rtdd", rows, cols, iters) == want


# ---- the multi-GPU entry points from a C++ host ------------------------------------------------------------------------------

def build_mgpu_host():
    os.makedirs(BUILD, exist_ok=True)
    out = os.path.join(BUILD, "mgpu_host")
    libdir = os.path.join(ROOT, "realtimedepthdiffusion_b200", "lib")
    cmd = ["g++", "-std=c++17", "-O1", os.path.join(ROOT, "tests", "cpp", "mgpu_host.cpp"), "-I", os.path.join(ROOT, "include"),
           "-I", os.path.join(CUDA, "include"), "-L", libdir, "-lrtdd", "-L", os.path.join(CUDA, "lib64"), "-lcudart", "-Wl,-rpath," + libdir, "-o", out]
    r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    assert r.returncode == 0, r.stdout
    return out


def test_mgpu_host_links_against_the_c_abi():
    """tests/cpp/mgpu_host.cpp uses only include/rtdd.h + the CUDA runtime: rtdd_mgpu_* and rtdd_strip_frame_* resolve from librtdd.so."""
    exe = build_mgpu_host()
    undefined = subprocess.run(["nm", "-u", exe], stdout=subprocess.PIPE, text=True).stdout
    for fn in ("rtdd_mgpu_create", "rtdd_mgpu_set_image", "rtdd_mgpu_frame_solve_host_annotation", "rtdd_mgpu_batch_solve", "rtdd_mgpu_destroy",
               "rtdd_strip_frame_effects", "rtdd_strip_frame_rows"):
        assert re.search(r"\b%s\b" % fn, undefined), fn


@pytest.mark.gpu
@pytest.mark.parametrize("ngpus,rows,cols,iters", [(2, 1536, 2048, 1000), (2, 1081, 1923, 300)])
def test_mgpu_host_strips_effects_and_batch_identical_to_one_gpu(ngpus, rows, cols, iters):
    """One process, one host thread per GPU inside librtdd.so, peer access instead of IPC: strips, effects on strips and the batch
    must reproduce the single-GPU bytes.  Needs >= 2 GPUs (gpurun --gpus 2); the program itself reports 'skipped' otherwise."""
    exe = build_mgpu_host()
    r = subprocess.run([exe, str(ngpus), str(rows), str(cols), str(iters)], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=280)
    assert r.returncode == 0, r.stdout
    if "skipped" in r.stdout:
        pytest.skip(r.stdout.strip())
    assert "all identical" in r.stdout, r.stdout


# ---- the per-frame download from a C++ host: pageable, cudaHostRegister'ed and cudaHostAlloc'ed planes -------------------------------

def build_pinned_map():
    os.makedirs(BUILD, exist_ok=True)
    out = os.path.join(BUILD, "pinned_map")
    libdir = os.path.join(ROOT, "realtimedepthdiffusion_b200", "lib")
    cmd = ["g++", "-std=c++17", "-O1", os.path.join(ROOT, "tests", "cpp", "pinned_map.cpp"), "-I", os.path.join(ROOT, "include"),
           "-I", os.path.join(CUDA, "include"), "-L", libdir, "-lrtdd", "-L", os.path.join(CUDA, "lib64"), "-lcudart", "-Wl,-rpath," + libdir, "-o", out]
    r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    assert r.returncode == 0, r.stdout
    return out


def test_pinned_map_links_against_the_c_abi():
    exe = build_pinned_map()
    undefined = subprocess.run(["nm", "-u", exe], stdout=subprocess.PIPE, text=True).stdout
    for fn in ("rtdd_frame_solve_host_annotation", "rtdd_frame_solve_download", "rtdd_frame_paint"):
        assert re.search(r"\b%s\b" % fn, undefined), fn


@pytest.mark.gpu
@pytest.mark.parametrize("rows,cols,iters", [(540, 960, 1000), (271, 483, 300)])
def test_pinned_map_same_bytes_whatever_the_host_plane(rows, cols, iters):
    """rtdd_frame_solve_host_annotation / rtdd_frame_solve_download from C++: the map stored by the last pass into page-locked planes
    (cudaHostRegister on an ordinary allocation, cudaHostAlloc) equals the staged copy into a pageable one."""
    exe = build_pinned_map()
    r = subprocess.run([exe, str(rows), str(cols), str(iters)], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=280)
    assert r.returncode == 0, r.stdout
    assert "identical" in r.stdout and "MISMATCH" not in r.stdout, r.stdout
