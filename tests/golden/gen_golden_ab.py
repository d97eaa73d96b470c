"""Records tests/golden/ref_ab.json: what the reference's own kernels compute in the A/B tests (test_gpu_parity.py,
test_gpu_scale_parity.py, test_cpp_dropin.py, test_abi_symbols.py), as sha256 hashes and checksum lines.  Needs a GPU.

  python tests/golden/gen_golden_ab.py [--api ref|rtdd] [out.json]      (default out: tests/golden/ref_ab.json)

--api ref (default) drives oracle/_ref/libref.so, the reference's src/*.cu compiled unmodified by
realtimedepthdiffusion_b200/build.py when the reference's sources are at hand.  --api rtdd drives librtdd.so's
reference-named functions instead; that records the reference's results only for a build of librtdd.so that the A/B tests
had found bit-identical to libref.so in the same process.  The committed file was recorded that way: the reference's sources
are not part of this repository, and the kernels of the commit that added the file are the ones those same-process A/B
tests had passed with on a B200.  Every test case calls the same functions as the tests themselves.
"""
import argparse
import json
import os
import re
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

from oracle import binding as ob                       # noqa: E402
from realtimedepthdiffusion_b200 import _native, synth  # noqa: E402
from tests import test_cpp_dropin, test_gpu_parity, test_gpu_scale_parity as scale  # noqa: E402


def exported_reference_names(path):
    """The mangled names of the ten reference-named functions among the library's defined dynamic symbols."""
    out = subprocess.run(["nm", "-D", "--defined-only", path], stdout=subprocess.PIPE, text=True, check=True).stdout
    names = []
    for m in re.finditer(r"\b_Z(\d+)(GPU\w+)", out):
        if m.group(2)[: int(m.group(1))] in _native.SHIM_SYMBOLS:
            names.append(m.group(0))
    return sorted(set(names))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--api", choices=["ref", "rtdd"], default="ref")
    ap.add_argument("out", nargs="?", default=os.path.join(ROOT, "tests", "golden", "ref_ab.json"))
    args = ap.parse_args()
    if args.api == "ref":
        api, libpath, libdir, libname = ob.ref_api(), ob.LIBREF, os.path.dirname(ob.LIBREF), "ref"
    else:
        api, libpath, libdir, libname = _native.shims, _native.LIB_PATH, os.path.dirname(_native.LIB_PATH), "rtdd"
    rec = {"recorded_with": os.path.relpath(libpath, ROOT)}

    rec["symbols"] = exported_reference_names(libpath)
    assert len(rec["symbols"]) == 10, rec["symbols"]

    rec["effects_and_paint_203x317"] = test_gpu_parity.effects_and_paint(api)
    print("effects_and_paint", flush=True)

    bgr, events, frames = scale.stroke_replay_1080p()
    rec["stroke_replay_1080p"] = scale.main_loop_hashes(api, bgr, frames)
    print("stroke_replay_1080p", len(frames), "frames", flush=True)

    bgr, scribble, edited = synth.synth_case(2160, 3840, 1003)
    rec["frame_4k"] = scale.main_loop_hashes(api, bgr, [(scribble, edited)], effects=True)
    print("frame_4k", flush=True)

    size, sweeps = 16384, 64
    gray, depth, scribble, d = scale.finest_level(api, size, sweeps)
    rec["level0_%d_x%d" % (size, sweeps)] = {"inputs": [scale.dev_sha(gray), scale.dev_sha(depth), scale.dev_sha(scribble)],
                                             "depth": scale.dev_sha(d)}
    del gray, depth, scribble, d
    print("level0_16384", flush=True)

    bgr, depth, out = scale.defocus_7400(api)
    rec["defocus_7400"] = {"inputs": [scale.dev_sha(bgr), scale.dev_sha(depth)], "out": scale.dev_sha(out)}
    del bgr, depth, out
    print("defocus_7400", flush=True)

    rec["main_like"] = {"%dx%dx%d" % c: test_cpp_dropin.main_like_line(libname, libdir, libname, *c) for c in ((203, 317, 100), (624, 672, 1000))}
    print("main_like", rec["main_like"], flush=True)

    with open(args.out, "w") as f:
        json.dump(rec, f, indent=1, sort_keys=True)
        f.write("\n")
    print("written", args.out, os.path.getsize(args.out), "bytes")


if __name__ == "__main__":
    main()
