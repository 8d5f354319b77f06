"""The planned loop (vrj_plan_counts -> vrj_render_counts) against vrj_render_adaptive and uniform sampling, on C3
(scene_main, recursion limit 8) and C5 (scene_main "mixed", limit 128) at 1920x1080.

For each config: a reference image by uniform sampling at --ref-spp (other sample indices than the runs compared); then the
planned loop with a pilot of 4 and of 16 samples (min_samples; the loop runs until a plan asks for no sample), the adaptive
render with the same rule (pilot 4), the uniform render at the planned loop's (pilot 4) total samples and the uniform render
at its device time.  Each reports device ms (the sum of the render calls' CUDA-event times; the plans run on a stream of
their own and are reported apart, as plan_ms, host clock), rounds or passes, wavefront batches and the relative RMSE of Y
against the reference, sqrt(mean((Y - Y_ref)^2) / mean(Y_ref^2)).  Finally the overhead of the count path: a uniform map
c = --overhead-spp through vrj_render_counts against vrj_render_tile at that spp (the same image, bit for bit).  The state
stays in device memory, as a progressive renderer keeps it.  Every timed run is repeated --repeats times.  Writes JSON to
the path given and prints the card name and power limit with the numbers.

    python tools/planned_quality.py out.json [--repeats 3] [--ref-spp 1024]"""
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
ap.add_argument("--ref-spp", type=int, default=1024)
ap.add_argument("--width", type=int, default=1920)
ap.add_argument("--height", type=int, default=1080)
ap.add_argument("--pass-samples", type=int, default=4)
ap.add_argument("--max", type=int, default=256)
ap.add_argument("--rel-error", type=float, default=0.02)
ap.add_argument("--overhead-spp", type=int, default=16)
ap.add_argument("--configs", default="C3,C5")
args = ap.parse_args()

W, H = args.width, args.height
NPIX = W * H
FULL = (0, W, 0, H)
REF_OFFSET = 1 << 40  # the reference's samples are not the compared runs' samples
L = capi.cuda()

if L.vrj_device_count() < 1:
    sys.exit("planned_quality.py needs a CUDA device")
smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
card = smi.stdout.strip().splitlines()[0] if smi.returncode == 0 and smi.stdout.strip() else "unknown (nvidia-smi failed)"


def rel_rmse(y, ref):
    return float(np.sqrt(np.mean((y - ref) ** 2) / np.mean(ref ** 2)))


def summary(vals):
    return {"runs": vals, "median": float(np.median(vals)), "min": float(np.min(vals)), "max": float(np.max(vals))}


class DeviceFrame:
    """colour, the state and a count map in device memory (vrj_alloc_device zero-fills)"""
    SIZES = {"colour": 24, "colour_sum": 24, "colour_bias": 24, "weight": 8, "weight_bias": 8, "y_sq_sum": 8, "counts": 4}

    def __init__(self):
        self.ptr = {k: L.vrj_alloc_device(0, NPIX * b) for k, b in self.SIZES.items()}
        assert all(self.ptr.values())

    def free(self):
        for p in self.ptr.values():
            L.vrj_free_device(p)

    def y(self):
        c = np.zeros(NPIX * 3)
        capi.check(L.vrj_copy_to_host(0, c.ctypes.data, self.ptr["colour"], c.nbytes))
        return c.reshape(-1, 3)[:, 1]

    def accum_out(self, st, accumulate):
        ao = capi.AccumOut(memory=capi.MEM_DEVICE, accumulate=1 if accumulate else 0)
        for k in ("colour", "colour_sum", "colour_bias", "weight", "weight_bias"):
            setattr(ao, k, self.ptr[k])
        ao.stats = C.pointer(st)
        return ao


def planned(hs, kw, pilot):
    """the planned loop from a zero state; returns (render device ms, plan ms, rounds, batches, samples, Y)"""
    f = DeviceFrame()
    p, keep = hs.make_params(spp=0, **kw)
    rule = capi.AdaptiveParams(min_samples=pilot, max_samples=args.max, pass_samples=args.pass_samples, rel_error=args.rel_error)
    t = capi.Tile(*FULL)
    ms = plan_ms = 0.0
    rounds = batches = samples = 0
    started = False
    while True:
        ps = capi.PlanStats()
        t0 = time.perf_counter()
        capi.check(L.vrj_plan_counts(0, capi.MEM_DEVICE, NPIX, f.ptr["weight"], f.ptr["colour_sum"], f.ptr["y_sq_sum"], C.byref(rule),
                                     f.ptr["counts"], C.byref(ps)))
        plan_ms += (time.perf_counter() - t0) * 1e3
        if ps.samples == 0:
            break
        st, cs = capi.Stats(), capi.CountsStats()
        capi.check(L.vrj_render_counts(hs.device_scene(0), C.byref(t), H, W, C.byref(p), f.ptr["counts"], C.byref(f.accum_out(st, started)),
                                       f.ptr["y_sq_sum"], C.byref(cs)))
        started = True
        ms += st.device_ms
        rounds, batches, samples = rounds + 1, batches + cs.batches, samples + cs.samples
    y = f.y()
    f.free()
    return ms, plan_ms, rounds, batches, samples, y


def uniform(hs, spp, kw, ref):
    ms, err = [], None
    for r in range(args.repeats):
        u = hs.render(FULL, H, W, spp=spp, want=("colour",), **kw)
        ms.append(u["stats"].device_ms)
        err = rel_rmse(u["colour"].reshape(-1, 3)[:, 1], ref)
    return {"spp": spp, "samples": spp * NPIX, "device_ms": summary(ms), "rel_rmse_y": err}


results = {"card": card, "width": W, "height": H, "ref_spp": args.ref_spp, "repeats": args.repeats,
           "rule": {"pass_samples": args.pass_samples, "max_samples": args.max, "rel_error": args.rel_error, "abs_floor": 0.0},
           "configs": {}}
print("card: %s" % card, flush=True)
CONFIGS = {"C3": (lambda: scenes.scene_main(), 8), "C5": (lambda: scenes.scene_main(variant="mixed"), 128)}
for name in args.configs.split(","):
    make, depth = CONFIGS[name]
    hs = V.build_scene(make())
    kw = dict(max_depth=depth, seed=1)
    hs.render((0, 64, 0, 64), H, W, spp=2, **kw)  # warm-up: module load, scratch blocks
    hs.render_adaptive((0, 64, 0, 64), H, W, 2, 4, 2, 0.1, **kw)
    hs.render_counts((0, 64, 0, 64), H, W, np.full(64 * 64, 2, np.uint32), **kw)
    ref_out = hs.render(FULL, H, W, spp=args.ref_spp, want=("colour",), **dict(kw, sample_offset=REF_OFFSET))
    ref = ref_out["colour"].reshape(-1, 3)[:, 1]
    res = {"max_depth": depth, "reference_device_ms": ref_out["stats"].device_ms}
    for pilot in (4, 16):
        ms, pms = [], []
        for r in range(args.repeats):
            m, pm, rounds, batches, samples, y = planned(hs, kw, pilot)
            ms.append(m), pms.append(pm)
        res["planned_pilot%d" % pilot] = {"device_ms": summary(ms), "plan_ms": summary(pms), "rounds": rounds, "batches": batches,
                                          "samples": samples, "mean_spp": samples / NPIX, "rel_rmse_y": rel_rmse(y, ref)}
    ms = []
    for r in range(args.repeats):
        a = hs.render_adaptive(FULL, H, W, 4, args.max, args.pass_samples, args.rel_error, want=("colour",), **kw)
        ms.append(a["stats"].device_ms)
    res["adaptive"] = {"device_ms": summary(ms), "passes": int(a["adaptive"].passes), "samples": int(a["adaptive"].samples),
                       "mean_spp": a["adaptive"].samples / NPIX, "batches": int(a["stats"].resolve_launches),
                       "rel_rmse_y": rel_rmse(a["colour"].reshape(-1, 3)[:, 1], ref)}
    P = res["planned_pilot4"]
    eq_samples = max(1, int(round(P["samples"] / NPIX)))
    res["uniform_equal_samples"] = uniform(hs, eq_samples, kw, ref)
    ms_per_spp = res["uniform_equal_samples"]["device_ms"]["median"] / eq_samples
    eq_time = max(1, int(round(P["device_ms"]["median"] / ms_per_spp)))
    res["uniform_equal_time"] = uniform(hs, eq_time, kw, ref)
    S = args.overhead_spp
    t_c, t_u = [], []
    for r in range(args.repeats):
        c = hs.render_counts(FULL, H, W, np.full(NPIX, S, np.uint32), want=("colour",), **kw)
        u = hs.render(FULL, H, W, spp=S, want=("colour",), **kw)
        t_c.append(c["stats"].device_ms), t_u.append(u["stats"].device_ms)
    same = bool(np.array_equal(c["colour"].view(np.uint64), u["colour"].view(np.uint64)))
    res["overhead_uniform_map"] = {"spp": S, "counts_device_ms": summary(t_c), "tile_device_ms": summary(t_u),
                                   "ratio_of_medians": float(np.median(t_c) / np.median(t_u)), "bit_equal": same}
    results["configs"][name] = res
    A, U, T, O = res["adaptive"], res["uniform_equal_samples"], res["uniform_equal_time"], res["overhead_uniform_map"]
    for pilot in (4, 16):
        P = res["planned_pilot%d" % pilot]
        print("%s planned (pilot %d): %.1f ms [%.1f-%.1f] + plans %.1f ms host, %d rounds, %d batches, %.2f spp/px, relRMSE %.4f" %
              (name, pilot, P["device_ms"]["median"], P["device_ms"]["min"], P["device_ms"]["max"], P["plan_ms"]["median"],
               P["rounds"], P["batches"], P["mean_spp"], P["rel_rmse_y"]), flush=True)
    print("%s adaptive: %.1f ms, %d passes, %d batches, %.2f spp/px, relRMSE %.4f | uniform %d spp %.1f ms relRMSE %.4f | "
          "uniform equal time %d spp %.1f ms relRMSE %.4f | uniform map %d: counts %.2f ms vs tile %.2f ms (bit equal: %s)" %
          (name, A["device_ms"]["median"], A["passes"], A["batches"], A["mean_spp"], A["rel_rmse_y"], U["spp"], U["device_ms"]["median"],
           U["rel_rmse_y"], T["spp"], T["device_ms"]["median"], T["rel_rmse_y"], S, O["counts_device_ms"]["median"],
           O["tile_device_ms"]["median"], same), flush=True)
    del hs
with open(args.out, "w") as f:
    json.dump(results, f, indent=1)
print("wrote %s" % args.out)
