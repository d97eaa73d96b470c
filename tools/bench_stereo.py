"""Stereo views on the GPU: device time per call (CUDA events) at 1080p, 4K and 8K, with the cached refocus pass as a point of
comparison.

  stereo_all          rtdd_frame_stereo, left + right + anaglyph
  stereo_left_right   rtdd_frame_stereo, left + right (side by side into one buffer)
  stereo_anaglyph     rtdd_frame_stereo, anaglyph only
  stereo_all_D0       stereo_all at maximum disparity 0: every column covered by its own source, no hole to resolve
  refocus_cached_K    rtdd_frame_refocus at aperture K, focus 0 (summed-area table cached per image)

Inputs are a solved depth of a synthetic scribbled image (the solver's range, [0, 255]); the stereo cases converge at depth 128
with a maximum disparity of cols / 32 pixels (60 at 1080p, 120 at 4K, 240 at 8K).  Each case is warmed up and captured as a
CUDA graph of `--reps` back-to-back calls, so host launch overhead stays out of the device time; the graphs are replayed in
`--rounds` rounds, the cases of one size interleaved round by round, and the median round is reported with the spread.  No
cache flush between calls: the 1080p working set fits in the 126 MB L2, 4K (133 MB for all three outputs) just does not, 8K
does not.  Bytes: 7 B/px read (BGR + fp32 depth) + 3 B/px written per output; the effective
bandwidth is those bytes over the median time.

python tools/bench_stereo.py [--sizes 1080x1920,2160x3840,4320x7680] [--reps 50] [--rounds 6] [--out FILE.json]
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

COPY_RATE_GBS = 6535.4          # BASELINE.md: torch copy, read + write bytes, B200


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
    K = int(0.025 * float(np.sqrt(np.float32(rows * rows + cols * cols))))      # the reference defocus's box side (rtdd.h)
    D = cols // 32
    zeros = np.zeros_like(bgr)
    left, right, ana, out = (to_dev(zeros, 3) for _ in range(4))
    sbs = torch.zeros((rows, 6 * cols), dtype=torch.uint8, device="cuda")
    cases = {
        "stereo_all": (lambda: ctx.frame_stereo(left, right, ana, convergence_depth=128.0, max_disparity=D), 3),
        "stereo_left_right": (lambda: ctx.frame_stereo(sbs[:, :3 * cols], sbs[:, 3 * cols:], None, convergence_depth=128.0,
                                                       max_disparity=D), 2),
        "stereo_anaglyph": (lambda: ctx.frame_stereo(None, None, ana, convergence_depth=128.0, max_disparity=D), 1),
        "stereo_all_D0": (lambda: ctx.frame_stereo(left, right, ana, convergence_depth=128.0, max_disparity=0), 3),
        "refocus_cached_K": (lambda: ctx.frame_refocus(out, focus_depth=0.0, aperture=K), 1),
    }
    times = {k: [] for k in cases}
    graphs = {}
    with torch.cuda.stream(s):
        for fn, _ in cases.values():                    # warm-up; builds the refocus table once
            for _ in range(10):
                fn()
        s.synchronize()
        for name, (fn, _) in cases.items():             # `reps` calls per graph: a 1080p pass is shorter than a host launch
            graphs[name] = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graphs[name], stream=s):
                for _ in range(reps):
                    fn()
            graphs[name].replay()
        s.synchronize()
        for _ in range(rounds):
            for name, g in graphs.items():
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(s)
                g.replay()
                e1.record(s)
                e1.synchronize()
                times[name].append(e0.elapsed_time(e1) / reps)
    del graphs
    ctx.set_stream(None)
    ctx.close()
    res = {"K": K, "max_disparity": D}
    for name, t in times.items():
        med = statistics.median(t)
        r = {"ms_median": med, "ms_min": min(t), "ms_max": max(t), "calls": reps * rounds}
        if name.startswith("stereo"):
            nbytes = rows * cols * (7 + 3 * cases[name][1])
            r["bytes"] = nbytes
            r["gb_per_s"] = nbytes / (med * 1e-3) / 1e9
            r["of_copy_rate"] = r["gb_per_s"] / COPY_RATE_GBS
        res[name] = r
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", default="1080x1920,2160x3840,4320x7680", help="rows x cols, comma separated")
    ap.add_argument("--reps", type=int, default=50)
    ap.add_argument("--rounds", type=int, default=6)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_stereo: needs a CUDA device")
    if a.reps * a.rounds < 200:
        sys.exit("bench_stereo: at least 200 timed calls per case (--reps x --rounds)")
    result = {"card": card(), "reps": a.reps, "rounds": a.rounds, "copy_rate_gb_per_s": COPY_RATE_GBS, "sizes": {}}
    print("card: %s, power limit %s W" % (result["card"]["name"], result["card"].get("power_limit_w")), flush=True)
    for sz in a.sizes.split(","):
        rows, cols = (int(v) for v in sz.lower().split("x"))
        r = bench_size(rows, cols, a.reps, a.rounds)
        result["sizes"]["%dx%d" % (cols, rows)] = r
        print("%dx%d (D = %d, K = %d)" % (cols, rows, r["max_disparity"], r["K"]))
        for name, v in r.items():
            if isinstance(v, dict):
                bw = "  %7.0f GB/s = %.2f of copy" % (v["gb_per_s"], v["of_copy_rate"]) if "gb_per_s" in v else ""
                print("  %-18s %8.4f ms  (min %.4f, max %.4f)%s" % (name, v["ms_median"], v["ms_min"], v["ms_max"], bw), flush=True)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(result, f, indent=1)
            f.write("\n")


if __name__ == "__main__":
    main()
