"""A progressive preview loop (vrj_render_progressive, max_passes = 1 per call) against one max_passes = 0 call and against
vrj_render_adaptive with the same parameters, on C3 (scene_main, recursion limit 8) and C5 (scene_main "mixed", limit 128)
at 1920x1080, every array in device memory.

Per config and repeat: the device time (VrjStats.device_ms summed over the calls) and the host wall time of each of the
three ways to the same frame; the per-call overhead of the loop, (loop - one call) / (calls - 1), in device and wall time;
one denoised preview per iteration (vrj_denoise into device memory plus the 6 MB srgb8 copy back; the first-hit features
come from one vrj_render_aux per frame, timed apart); and whether the three final states are bit-identical.  Writes JSON to
the path given and prints the card name and power limit with the numbers.

    python tools/progressive_loop.py out.json [--repeats 3] [--min 4] [--pass-samples 4] [--max 64] [--rel-error 0.05]"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np

import vanrijn_b200 as V
from vanrijn_b200 import capi, scenes

ap = argparse.ArgumentParser()
ap.add_argument("out")
ap.add_argument("--repeats", type=int, default=3)
ap.add_argument("--width", type=int, default=1920)
ap.add_argument("--height", type=int, default=1080)
ap.add_argument("--min", type=int, default=4)
ap.add_argument("--pass-samples", type=int, default=4)
ap.add_argument("--max", type=int, default=64)
ap.add_argument("--rel-error", type=float, default=0.05)
ap.add_argument("--aux-spp", type=int, default=4)
args = ap.parse_args()

W, H = args.width, args.height
NPIX = W * H
FULL = capi.Tile(0, W, 0, H)
L = capi.cuda()
if L.vrj_device_count() < 1:
    sys.exit("progressive_loop.py needs a CUDA device")
smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
card = smi.stdout.strip().splitlines()[0] if smi.returncode == 0 and smi.stdout.strip() else "unknown (nvidia-smi failed)"
STATE = (("colour_sum", 24), ("colour_bias", 24), ("weight", 8), ("weight_bias", 8), ("y_sq_sum", 8))


class Frame:
    def __init__(self):
        self.ptr = {name: L.vrj_alloc_device(0, NPIX * b) for name, b in STATE + (("colour", 24),)}
        assert all(self.ptr.values()), "vrj_alloc_device failed"

    def out(self, accumulate, st):
        ao = capi.AccumOut(memory=capi.MEM_DEVICE, accumulate=accumulate, stats=C.pointer(st))
        for name in ("colour", "colour_sum", "colour_bias", "weight", "weight_bias"):
            setattr(ao, name, self.ptr[name])
        return ao

    def fetch(self):
        res = {}
        for name, b in STATE:
            res[name] = np.zeros(NPIX * b // 8)
            capi.check(L.vrj_copy_to_host(0, res[name].ctypes.data, self.ptr[name], NPIX * b))
        return res

    def free(self):
        for p in self.ptr.values():
            L.vrj_free_device(p)


def progressive(hs, f, p, max_passes, accumulate):
    pp = capi.ProgressiveParams(min_samples=args.min, max_samples=args.max, pass_samples=args.pass_samples, max_passes=max_passes,
                                rel_error=args.rel_error)
    st, pst = capi.Stats(), capi.ProgressiveStats()
    capi.check(L.vrj_render_progressive(hs.device_scene(0), C.byref(FULL), H, W, C.byref(p), C.byref(pp), C.byref(f.out(accumulate, st)),
                                        f.ptr["y_sq_sum"], C.byref(pst)))
    return st, pst


def run(hs, kw):
    p, keep = hs.make_params(spp=0, **kw)
    fa, fo, fl = Frame(), Frame(), Frame()
    try:
        # vrj_render_adaptive
        st, ast = capi.Stats(), capi.AdaptiveStats()
        ap_ = capi.AdaptiveParams(min_samples=args.min, max_samples=args.max, pass_samples=args.pass_samples, rel_error=args.rel_error)
        t0 = time.perf_counter()
        capi.check(L.vrj_render_adaptive(hs.device_scene(0), C.byref(FULL), H, W, C.byref(p), C.byref(ap_), C.byref(fa.out(0, st)),
                                         fa.ptr["y_sq_sum"], C.byref(ast)))
        adaptive = {"device_ms": st.device_ms, "wall_ms": (time.perf_counter() - t0) * 1e3, "passes": ast.passes, "samples": ast.samples}
        # one max_passes = 0 call
        t0 = time.perf_counter()
        st, pst = progressive(hs, fo, p, 0, 0)
        one = {"device_ms": st.device_ms, "wall_ms": (time.perf_counter() - t0) * 1e3, "passes": pst.passes, "samples": pst.samples}
        # the loop: max_passes = 1 per call, a denoised preview after each pass
        aux_ptr = {"normal": L.vrj_alloc_device(0, NPIX * 24), "depth": L.vrj_alloc_device(0, NPIX * 8),
                   "material": L.vrj_alloc_device(0, NPIX * 4), "colour": L.vrj_alloc_device(0, NPIX * 24), "srgb8": L.vrj_alloc_device(0, NPIX * 3)}
        pa, keep_a = hs.make_params(spp=args.aux_spp, **kw)
        ao = capi.AuxOut(memory=capi.MEM_DEVICE, normal=aux_ptr["normal"], depth=aux_ptr["depth"], material=aux_ptr["material"],
                         stats=C.pointer(capi.Stats()))
        t0 = time.perf_counter()
        capi.check(L.vrj_render_aux(hs.device_scene(0), C.byref(FULL), H, W, C.byref(pa), C.byref(ao)))
        aux_ms = (time.perf_counter() - t0) * 1e3
        dp = capi.DenoiseParams(iterations=4, sigma_luminance=32.0, sigma_normal=128.0, sigma_depth=0.5)
        rgb = np.zeros(NPIX * 3, np.uint8)
        loop_dev = loop_wall = 0.0
        calls, preview_wall, preview_dev = 0, [], []
        while True:
            t0 = time.perf_counter()
            st, pst = progressive(hs, fl, p, 1, 1 if calls else 0)
            loop_wall += (time.perf_counter() - t0) * 1e3
            loop_dev += st.device_ms
            calls += 1
            if pst.passes == 0:
                break
            ms = C.c_double(0.0)
            t0 = time.perf_counter()
            capi.check(L.vrj_denoise(0, capi.MEM_DEVICE, W, H, fl.ptr["colour_sum"], fl.ptr["weight"], fl.ptr["y_sq_sum"], aux_ptr["normal"],
                                     aux_ptr["depth"], aux_ptr["material"], C.byref(dp), aux_ptr["colour"], aux_ptr["srgb8"], C.byref(ms)))
            capi.check(L.vrj_copy_to_host(0, rgb.ctypes.data, aux_ptr["srgb8"], NPIX * 3))
            preview_wall.append((time.perf_counter() - t0) * 1e3)
            preview_dev.append(ms.value)
        for q in aux_ptr.values():
            L.vrj_free_device(q)
        loop = {"device_ms": loop_dev, "wall_ms": loop_wall, "calls": calls, "passes": calls - 1,
                "overhead_device_ms_per_call": (loop_dev - one["device_ms"]) / max(1, calls - 1),
                "overhead_wall_ms_per_call": (loop_wall - one["wall_ms"]) / max(1, calls - 1)}
        preview = {"aux_wall_ms": aux_ms, "denoise_device_ms_median": float(np.median(preview_dev)) if preview_dev else None,
                   "denoise_plus_copy_wall_ms_median": float(np.median(preview_wall)) if preview_wall else None}
        sa, so, sl = fa.fetch(), fo.fetch(), fl.fetch()
        identical = all(np.array_equal(sa[n].view(np.uint64), so[n].view(np.uint64)) and np.array_equal(so[n].view(np.uint64), sl[n].view(np.uint64))
                        for n, _ in STATE)
        return {"adaptive": adaptive, "one_call": one, "loop": loop, "preview": preview, "states_bit_identical": bool(identical)}
    finally:
        for f in (fa, fo, fl):
            f.free()


results = {"card": card, "width": W, "height": H, "min": args.min, "pass_samples": args.pass_samples, "max": args.max,
           "rel_error": args.rel_error, "configs": {}}
print("card, power limit: %s" % card)
for name, spec, depth in (("C3", scenes.scene_main(), 8), ("C5", scenes.scene_main(variant="mixed"), 128)):
    hs = V.build_scene(spec)
    kw = dict(max_depth=depth, seed=1)
    run(hs, kw)  # warm-up: modules, scratch blocks, pooled device memory
    reps = [run(hs, kw) for _ in range(args.repeats)]
    results["configs"][name] = reps
    for i, r in enumerate(reps):
        a, o, lp, pv = r["adaptive"], r["one_call"], r["loop"], r["preview"]
        print("%s rep %d: adaptive %.2f ms dev / %.2f ms wall; one call %.2f / %.2f; loop of %d calls %.2f / %.2f "
              "(overhead %.3f ms dev, %.3f ms wall per call); passes %d, samples/pixel %.2f; denoised preview %.2f ms dev, "
              "%.2f ms wall with copy (aux once %.2f ms wall); bit-identical %s"
              % (name, i, a["device_ms"], a["wall_ms"], o["device_ms"], o["wall_ms"], lp["calls"], lp["device_ms"], lp["wall_ms"],
                 lp["overhead_device_ms_per_call"], lp["overhead_wall_ms_per_call"], o["passes"], o["samples"] / NPIX,
                 pv["denoise_device_ms_median"] or 0.0, pv["denoise_plus_copy_wall_ms_median"] or 0.0, pv["aux_wall_ms"],
                 r["states_bit_identical"]))
with open(args.out, "w") as fh:
    json.dump(results, fh, indent=1)
