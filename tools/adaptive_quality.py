"""Adaptive against uniform sampling on C3 (scene_main, recursion limit 8) and C5 (scene_main "mixed", limit 128) at 1920x1080.

For each config: a reference image by uniform sampling at --ref-spp (other sample indices than the runs compared); then the
adaptive render, the uniform render at equal total samples (spp = adaptive samples / pixels, rounded) and the uniform render
at equal device time (spp from the uniform run's time per spp), each with device ms, total samples and the relative RMSE
of Y against the reference, sqrt(mean((Y - Y_ref)^2) / mean(Y_ref^2)).  Finally the machinery's overhead: an adaptive call
with min_samples == max_samples against vrj_render_tile at that spp (same image, bit for bit).  Every timed run is repeated
--repeats times.  Writes JSON to the path given and prints the card name and power limit with the numbers.

    python tools/adaptive_quality.py out.json [--repeats 3] [--ref-spp 1024]"""
import argparse
import json
import os
import subprocess
import sys

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
ap.add_argument("--min", type=int, default=4)
ap.add_argument("--pass-samples", type=int, default=4)
ap.add_argument("--max", type=int, default=256)
ap.add_argument("--rel-error", type=float, default=0.02)
ap.add_argument("--overhead-spp", type=int, default=16)
args = ap.parse_args()

W, H = args.width, args.height
NPIX = W * H
FULL = (0, W, 0, H)
REF_OFFSET = 1 << 40  # the reference's samples are not the compared runs' samples

if capi.cuda().vrj_device_count() < 1:
    sys.exit("adaptive_quality.py needs a CUDA device")
smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
card = smi.stdout.strip().splitlines()[0] if smi.returncode == 0 and smi.stdout.strip() else "unknown (nvidia-smi failed)"


def y_of(out):
    return out["colour"].reshape(-1, 3)[:, 1]


def rel_rmse(y, ref):
    return float(np.sqrt(np.mean((y - ref) ** 2) / np.mean(ref ** 2)))


def summary(vals):
    return {"runs": vals, "median": float(np.median(vals)), "min": float(np.min(vals)), "max": float(np.max(vals))}


def uniform(hs, spp, kw, ref):
    ms, err = [], None
    for r in range(args.repeats):
        u = hs.render(FULL, H, W, spp=spp, want=("colour",), **kw)
        ms.append(u["stats"].device_ms)
        err = rel_rmse(y_of(u), ref)  # the same image every repeat
    return {"spp": spp, "samples": spp * NPIX, "device_ms": summary(ms), "rel_rmse_y": err}


results = {"card": card, "width": W, "height": H, "ref_spp": args.ref_spp, "repeats": args.repeats,
           "adaptive_params": {"min_samples": args.min, "pass_samples": args.pass_samples, "max_samples": args.max,
                               "rel_error": args.rel_error, "abs_floor": 0.0}, "configs": {}}
print("card: %s" % card, flush=True)
for name, spec, depth in (("C3", scenes.scene_main(), 8), ("C5", scenes.scene_main(variant="mixed"), 128)):
    hs = V.build_scene(spec)
    kw = dict(max_depth=depth, seed=1)
    hs.render((0, 64, 0, 64), H, W, spp=2, **kw)  # warm-up: module load, scratch blocks
    hs.render_adaptive((0, 64, 0, 64), H, W, 2, 4, 2, 0.1, **kw)
    ref_out = hs.render(FULL, H, W, spp=args.ref_spp, want=("colour",), **dict(kw, sample_offset=REF_OFFSET))
    ref = y_of(ref_out)
    res = {"max_depth": depth, "reference_device_ms": ref_out["stats"].device_ms}
    ms, samples = [], None
    for r in range(args.repeats):
        a = hs.render_adaptive(FULL, H, W, args.min, args.max, args.pass_samples, args.rel_error, want=("colour", "weight"), **kw)
        ms.append(a["stats"].device_ms)
        samples = int(a["adaptive"].samples)
        ad = a["adaptive"].as_dict()
        err = rel_rmse(y_of(a), ref)
        counts = np.bincount(a["weight"].astype(np.int64))
    res["adaptive"] = {"samples": samples, "mean_spp": samples / NPIX, "device_ms": summary(ms), "rel_rmse_y": err, "stats": ad,
                       "pixels_per_count": {str(c): int(n) for c, n in enumerate(counts) if n}}
    eq_samples = max(1, int(round(samples / NPIX)))
    res["uniform_equal_samples"] = uniform(hs, eq_samples, kw, ref)
    ms_per_spp = res["uniform_equal_samples"]["device_ms"]["median"] / eq_samples
    eq_time = max(1, int(round(res["adaptive"]["device_ms"]["median"] / ms_per_spp)))
    res["uniform_equal_time"] = uniform(hs, eq_time, kw, ref)
    # overhead: min == max renders exactly what vrj_render_tile renders
    S = args.overhead_spp
    t_ad, t_un = [], []
    for r in range(args.repeats):
        t_ad.append(hs.render_adaptive(FULL, H, W, S, S, 1, 0.01, want=("colour",), **kw)["stats"].device_ms)
        t_un.append(hs.render(FULL, H, W, spp=S, want=("colour",), **kw)["stats"].device_ms)
    res["overhead_min_eq_max"] = {"spp": S, "adaptive_device_ms": summary(t_ad), "uniform_device_ms": summary(t_un),
                                  "ratio_of_medians": float(np.median(t_ad) / np.median(t_un))}
    results["configs"][name] = res
    A, U, T = res["adaptive"], res["uniform_equal_samples"], res["uniform_equal_time"]
    print("%s (depth %d, reference %d spp): adaptive %.2f spp/px %.1f ms [%.1f-%.1f] relRMSE %.4f | uniform %d spp %.1f ms relRMSE %.4f"
          " | uniform equal time %d spp %.1f ms relRMSE %.4f | overhead at %d spp: %.1f vs %.1f ms" %
          (name, depth, args.ref_spp, A["mean_spp"], A["device_ms"]["median"], A["device_ms"]["min"], A["device_ms"]["max"],
           A["rel_rmse_y"], U["spp"], U["device_ms"]["median"], U["rel_rmse_y"], T["spp"], T["device_ms"]["median"],
           T["rel_rmse_y"], S, res["overhead_min_eq_max"]["adaptive_device_ms"]["median"],
           res["overhead_min_eq_max"]["uniform_device_ms"]["median"]), flush=True)
    del hs
with open(args.out, "w") as f:
    json.dump(results, f, indent=1)
print("wrote %s" % args.out)
