"""Refocus against defocus on the GPU: device time per call (CUDA events), 1080p and 4K.

  stand-alone   rtdd_defocus  vs  rtdd_refocus at aperture K        (both build the summed-area table every call)
  cached        rtdd_frame_effects(defocus only)  vs  rtdd_frame_refocus at apertures K, 4K and 1024 (table cached per image)

Inputs are a solved depth of a synthetic scribbled image (the solver's range, [0, 255]).  The refocus cases use focus 0 and no
sharp band, so at aperture K every pixel asks for the same box as defocus; `click` focuses on the depth under the image centre
with a band of 10.  Each case is warmed up, then timed in `--rounds` rounds of `--reps` back-to-back calls, the cases of one
size interleaved round by round; the median round is reported, with the spread.  No cache flush between calls: at 1080p the
working set (image, depth, table, output: about 60 MB) fits in the 126 MB L2, at 4K (about 215 MB) it does not.

python tools/bench_refocus.py [--sizes 1080x1920,2160x3840] [--reps 50] [--rounds 6] [--out FILE.json]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import realtimedepthdiffusion_b200 as rtdd                  # noqa: E402
from realtimedepthdiffusion_b200 import synth               # noqa: E402
from realtimedepthdiffusion_b200.api import to_dev          # noqa: E402


def card():
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader,nounits"],
                           stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True, timeout=30).stdout.strip().split(",")
        info["power_limit_w"] = float(q[0])
        info["sm_max_mhz"] = float(q[1])
    except Exception as e:                      # the numbers are still device times; say why the card line is short
        info["power_limit_w"] = None
        info["nvidia_smi_error"] = str(e)
    return info


def bench_size(rows, cols, reps, rounds):
    s = torch.cuda.Stream()
    bgr, scribble, edited = synth.synth_case(rows, cols, 1003)
    ctx = rtdd.DepthDiffusion(rows, cols)
    ctx.set_stream(s)
    ctx.frame_set_image(bgr)
    ctx.frame_solve_host(scribble, edited, 1000, None)
    ctx.sync()
    depth = ctx.frame_plane(ctx.PLANE_DEPTH, 0)
    K = int(0.025 * float(np.sqrt(np.float32(rows * rows + cols * cols))))      # the reference defocus's box side (rtdd.h)
    o, d = to_dev(bgr, 3), to_dev(depth.cpu().numpy())
    out = [to_dev(np.zeros_like(bgr), 3) for _ in range(2)]
    cases = {
        "standalone_defocus": lambda: ctx.simulate_defocus(o, d, out[0]),
        "standalone_refocus_K": lambda: ctx.refocus(o, d, out[1], 0.0, 0.0, K),
        "cached_defocus": lambda: ctx.frame_effects(None, None, out[0]),
        "cached_refocus_K": lambda: ctx.frame_refocus(out[1], focus_depth=0.0, aperture=K),
        "cached_refocus_4K": lambda: ctx.frame_refocus(out[1], focus_depth=0.0, aperture=4 * K),
        "cached_refocus_1024": lambda: ctx.frame_refocus(out[1], focus_depth=0.0, aperture=1024),
        "cached_refocus_click_K": lambda: ctx.frame_refocus(out[1], focus_point=(cols // 2, rows // 2), depth_of_field=10.0, aperture=K),
    }
    # the parity point really is the same computation (cheap check, not a test)
    ctx.simulate_defocus(o, d, out[0])
    ctx.refocus(o, d, out[1], 0.0, 0.0, K)
    ctx.sync()
    assert torch.equal(out[0], out[1]), "refocus at the parity point differs from defocus"
    times = {k: [] for k in cases}
    with torch.cuda.stream(s):
        for fn in cases.values():                       # warm-up; the cached cases after a stand-alone call rebuild once here
            for _ in range(10):
                fn()
        s.synchronize()
        for _ in range(rounds):
            for name, fn in cases.items():
                if name.startswith("cached"):
                    fn()                                # the table is the frame's again after a stand-alone call
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(s)
                for _ in range(reps):
                    fn()
                e1.record(s)
                e1.synchronize()
                times[name].append(e0.elapsed_time(e1) / reps)
    ctx.set_stream(None)
    ctx.close()
    res = {}
    for name, t in times.items():
        res[name] = {"ms_median": statistics.median(t), "ms_min": min(t), "ms_max": max(t), "calls": reps * rounds}
    res["K"] = K
    res["cached_refocus_K_over_cached_defocus"] = res["cached_refocus_K"]["ms_median"] / res["cached_defocus"]["ms_median"]
    res["standalone_refocus_K_over_standalone_defocus"] = res["standalone_refocus_K"]["ms_median"] / res["standalone_defocus"]["ms_median"]
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", default="1080x1920,2160x3840", help="rows x cols, comma separated")
    ap.add_argument("--reps", type=int, default=50)
    ap.add_argument("--rounds", type=int, default=6)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_refocus: needs a CUDA device")
    if a.reps * a.rounds < 200:
        sys.exit("bench_refocus: at least 200 timed calls per case (--reps x --rounds)")
    result = {"card": card(), "reps": a.reps, "rounds": a.rounds, "sizes": {}}
    print("card: %s, power limit %s W" % (result["card"]["name"], result["card"].get("power_limit_w")), flush=True)
    for sz in a.sizes.split(","):
        rows, cols = (int(v) for v in sz.lower().split("x"))
        r = bench_size(rows, cols, a.reps, a.rounds)
        result["sizes"]["%dx%d" % (cols, rows)] = r
        print("%dx%d (K = %d)" % (cols, rows, r["K"]))
        for name, v in r.items():
            if isinstance(v, dict):
                print("  %-26s %8.4f ms  (min %.4f, max %.4f)" % (name, v["ms_median"], v["ms_min"], v["ms_max"]))
        print("  cached refocus at K / cached defocus: %.3f;  stand-alone: %.3f" %
              (r["cached_refocus_K_over_cached_defocus"], r["standalone_refocus_K_over_standalone_defocus"]), flush=True)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(result, f, indent=1)
            f.write("\n")


if __name__ == "__main__":
    main()
