"""Run ON THE GPU BOX (gpurun): drives the reference's own kernels (oracle/_ref/libref.so,
compiled unmodified from /root/reference/src) and records golden outputs under
gpurun_out/golden/ (copied afterwards into tests/golden/ and committed).

For every case the reference's per-level fp32 solver outputs are recorded as sha256 of the raw
bytes (bit-exactness pin), the coarse levels and a strided sample in full, plus the u8 results.
"""
import ctypes as C
import hashlib
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

from oracle import binding as ob                       # noqa: E402
from realtimedepthdiffusion_b200 import synth          # noqa: E402
from tests.harness import MainLoop, pitch, ptr, to_dev, to_host  # noqa: E402
from realtimedepthdiffusion_b200.api import pitched_empty        # noqa: E402

OUT = os.path.join(ROOT, "gpurun_out", "golden")


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def load_case(name):
    if name in ("dog", "womanparasol"):
        z = np.load(os.path.join(ROOT, "tests", "golden", "inputs_%s.npz" % name))
        bgr, ann = z["bgr"], z["annotation"]
        scribble = np.where(ann != 32, 255, 0).astype(np.uint8)           # main.cpp:163-168
        edited = bgr.copy()
        edited[ann != 32] = ann[ann != 32][:, None]
        return bgr, scribble, edited
    rows, cols, seed = CASES[name]
    return synth.synth_case(rows, cols, seed)


CASES = {"synth_odd": (203, 317, 11), "synth_small": (96, 130, 12), "synth_tiny": (45, 47, 13)}


def solver_case(api, name, max_iterations):
    bgr, scribble, edited = load_case(name)
    loop = MainLoop(api, bgr)
    u8 = loop.frame(scribble, edited, max_iterations, keep_levels=True)
    rec = {"levels": np.int32(loop.levels), "max_iterations": np.int32(max_iterations), "depth_u8": u8}
    for l, d in loop.per_level.items():
        rec["in_sha_%d" % l] = sha(d["in"])
        rec["out_sha_%d" % l] = sha(d["out"])
        if d["out"].size <= 160 * 170:
            rec["in_%d" % l] = d["in"]
            rec["out_%d" % l] = d["out"]
        else:
            rec["out_sample_%d" % l] = d["out"][::7, ::5].copy()
    # second frame: state carried over (coarsest depth persists), one more stroke
    ev = synth.brush_events(loop.rows, loop.cols, 99, 1, 6)
    scribble2, edited2 = synth.paint_events(bgr, ev, scribble.copy(), edited.copy())
    u8b = loop.frame(scribble2, edited2, max_iterations, keep_levels=True)
    rec["frame2_depth_u8"] = u8b
    rec["frame2_out_sha_0"] = sha(loop.per_level[0]["out"])
    depth0 = loop.depth_float.copy()
    # the reference's weight plane of level 0 (global deviceIndexToWeight, src/GPUSolver.cu:17)
    loop.close()
    return rec, bgr, loop.gray_host[0], depth0


def effects_case(api, bgr, gray, depth):
    rows, cols = depth.shape
    o = to_dev(bgr, 3)
    g = to_dev(gray[:rows, :cols].copy())
    d = to_dev(depth)
    rec = {}
    for name in ("GPUSimulateDesaturation", "GPUSimulateHaze", "GPUSimulateDefocus"):
        out = pitched_empty(rows, cols, torch.uint8, "cuda", channels=3, fill=0)
        torch.cuda.synchronize()
        if name == "GPUSimulateDesaturation":
            api[name](ptr(o), pitch(o), ptr(g), pitch(g), ptr(d), pitch(d), ptr(out), pitch(out), rows, cols)
        else:
            api[name](ptr(o), pitch(o), ptr(d), pitch(d), ptr(out), pitch(out), rows, cols)
        torch.cuda.synchronize()
        rec[name] = to_host(out, 3)
    return rec


def compact_effects(depth_sha, eff):
    """Dog is 672x624: keep hashes of the exact effects and a strided sample of haze (whose CPU oracle is +-1)."""
    return {"depth_sha": depth_sha,
            "desaturation_sha": sha(eff["GPUSimulateDesaturation"]), "defocus_sha": sha(eff["GPUSimulateDefocus"]),
            "haze_sha": sha(eff["GPUSimulateHaze"]), "haze_sample": eff["GPUSimulateHaze"][::4, ::4].copy(),
            "desaturation_sample": eff["GPUSimulateDesaturation"][::8, ::8].copy(),
            "defocus_sample": eff["GPUSimulateDefocus"][::8, ::8].copy()}


def weights_case(api, libref, rows, cols, seed, levels, level):
    """loadIndexToWeight through a 0-iteration GPUMatrixFreeSolver call; reads deviceIndexToWeight[level]."""
    rng = np.random.default_rng(seed)
    gray = synth.synth_image(rows, cols, seed)[..., 0].copy()
    depth = (rng.integers(0, 5, (rows, cols)) * 64 + rng.uniform(-6, 6, (rows, cols))).astype(np.float32)
    depth[rng.random((rows, cols)) < 0.01] = 300.7          # >= 256 wraps through the byte store
    depth[rng.random((rows, cols)) < 0.01] = -3.5           # negatives -> 0
    scribble = np.zeros((rows, cols), np.uint8)
    api["GPUAllocateDeviceMemory"](rows << level, cols << level, levels)
    api["GPULoadWeights"](0.4)
    dd, gg, ss = to_dev(depth), to_dev(gray), to_dev(scribble)
    torch.cuda.synchronize()
    api["GPUMatrixFreeSolver"](ptr(dd), pitch(dd), ptr(ss), pitch(ss), ptr(gg), pitch(gg), rows, cols, 0.4, 0, 1e-5, level)
    torch.cuda.synchronize()
    table = C.POINTER(C.c_void_p).in_dll(libref, "deviceIndexToWeight")
    dev_ptr = table[level]
    idx = torch.empty((rows, cols, 2), dtype=torch.int32, device="cuda")
    # device -> device copy through torch: wrap the raw pointer
    class H:  # noqa: E742
        pass
    h = H()
    h.__cuda_array_interface__ = {"shape": (rows, cols, 2), "typestr": "<i4", "data": (dev_ptr, False), "version": 2}
    idx.copy_(torch.as_tensor(h, device="cuda"))
    torch.cuda.synchronize()
    api["GPUFreeDeviceMemory"](levels)
    return {"gray": gray, "depth": depth, "int2": idx.cpu().numpy(), "level": np.int32(level), "levels": np.int32(levels)}


def dataset_goldens(api):
    """All 12 dataset pairs (BASELINE configs[0]) through the reference's own kernels, native resolution, 1000 sweeps at the
    coarsest level: per-level sha256 of the fp32 outputs, sha of the u8 map, and the same for a second frame with one more
    stroke (state carried over).  Hashes only -- the inputs are in tests/golden/dataset/."""
    import json
    from tests import dataset
    out = {}
    for name in dataset.NAMES:
        bgr, scribble, edited, _ = dataset.load_pair(name)
        loop = MainLoop(api, bgr)
        u8 = loop.frame(scribble, edited, 1000, keep_levels=True)
        rec = {"rows": loop.rows, "cols": loop.cols, "levels": loop.levels, "sizes": [list(x) for x in loop.sizes],
               "out_sha": {str(l): sha(d["out"]) for l, d in loop.per_level.items()},
               "in_sha": {str(l): sha(d["in"]) for l, d in loop.per_level.items()},
               "depth_u8_sha": sha(u8), "depth_u8_sample": u8[::64, ::64].tolist()}
        ev = synth.brush_events(loop.rows, loop.cols, 99, 1, 6)
        s2, e2 = synth.paint_events(bgr, ev, scribble.copy(), edited.copy())
        u8b = loop.frame(s2, e2, 1000, keep_levels=True)
        rec["frame2_out_sha_0"] = sha(loop.per_level[0]["out"])
        rec["frame2_depth_u8_sha"] = sha(u8b)
        loop.close()
        out[name] = rec
        print("dataset", name, loop.cols, "x", loop.rows, "levels", loop.levels, flush=True)
    with open(os.path.join(OUT, "ref_dataset.json"), "w") as f:
        json.dump(out, f, indent=1, sort_keys=True)


def main():
    os.makedirs(OUT, exist_ok=True)
    api = ob.ref_api()
    if "--dataset" in sys.argv:
        dataset_goldens(api)
        print("golden written to", OUT)
        return
    libref = C.CDLL(ob.LIBREF)    # same handle dlopen returns again (already loaded)
    dog = None
    only = sys.argv[1:]
    for name, iters in (("dog", 1000), ("womanparasol", 1000), ("synth_odd", 200), ("synth_small", 120), ("synth_tiny", 60)):
        if only and name not in only:
            continue
        rec, bgr, gray, depth0 = solver_case(api, name, iters)
        np.savez_compressed(os.path.join(OUT, "ref_solver_%s.npz" % name), **rec)
        print("solver", name, "levels", int(rec["levels"]), flush=True)
        if name in ("synth_odd",):
            eff = effects_case(api, bgr, gray, depth0)
            np.savez_compressed(os.path.join(OUT, "ref_effects_%s.npz" % name), depth=depth0, **eff)
            print("effects", name, flush=True)
        if name == "dog":
            dog = (bgr, gray, depth0)
    if only:
        print("golden written to", OUT)
        return
    # effects on Dog: u8 outputs only (depth is reproducible from the solver golden via sha)
    eff = effects_case(api, *dog)
    np.savez_compressed(os.path.join(OUT, "ref_effects_dog.npz"), **compact_effects(sha(dog[2]), eff))
    for i, (rows, cols, levels, level) in enumerate(((67, 120, 3, 2), (135, 240, 3, 1), (97, 131, 2, 0))):
        rec = weights_case(api, libref, rows, cols, 50 + i, levels, level)
        np.savez_compressed(os.path.join(OUT, "ref_weights_%d.npz" % i), **rec)
        print("weights", i, flush=True)
    print("golden written to", OUT)


if __name__ == "__main__":
    main()
