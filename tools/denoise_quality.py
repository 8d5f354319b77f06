"""Denoised against noisy and against uniform sampling at equal device time, on C3 (scene_main, recursion limit 8) and C5
(scene_main "mixed", limit 128) at 1920x1080.

For each config: a reference image by uniform sampling at --ref-spp (sample_offset 1 << 40, other samples than the runs
compared).  For each spp of --spps: the frame from vrj_render_adaptive with min_samples == max_samples == spp (the uniform
frame plus y_sq_sum), the first-hit features from vrj_render_aux at 1 spp, and vrj_denoise over a grid of parameters.  The
relative RMSE of Y against the reference, sqrt(mean((Y - Y_ref)^2) / mean(Y_ref^2)), is taken before and after.

The proposed default is the parameter set with the lowest mean, over every config and spp, of the WORST log(denoised /
noisy error) among the frame's parts: the whole frame on C3; on C5 the pixels whose first hit (sample 0) is specular
(reflective or dielectric: the mirror and glass spheres and the reflective mesh) and the other pixels, taken apart.  Scored
on the whole frame alone, C5's specular pixels dominate and the search picks a blur that smears the caustics on the
diffuse ground.  With it, the render, the aux pass and the denoise are timed separately (device_ms, --repeats runs after a
warm-up) and the denoised frame is compared with a uniform render at EQUAL TOTAL DEVICE TIME: spp = (render + aux +
denoise) / (the uniform render's time per spp), rounded.  Writes JSON to the path given and prints the card name and
power limit with the numbers, and the errors of the two parts of C5 separately.

    python tools/denoise_quality.py out.json [--repeats 3] [--ref-spp 1024] [--spps 4,16,64]"""
import argparse
import itertools
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np

import vanrijn_b200 as V
from vanrijn_b200 import capi, host, scenes

ap = argparse.ArgumentParser()
ap.add_argument("out")
ap.add_argument("--repeats", type=int, default=3)
ap.add_argument("--ref-spp", type=int, default=1024)
ap.add_argument("--width", type=int, default=1920)
ap.add_argument("--height", type=int, default=1080)
ap.add_argument("--spps", default="4,16,64")
ap.add_argument("--iterations", default="3,4,5,6")
ap.add_argument("--sigma-luminance", default="1,2,4,8,16,32")
ap.add_argument("--sigma-normal", default="32,128")
ap.add_argument("--sigma-depth", default="0.1,0.5,2")
args = ap.parse_args()

W, H = args.width, args.height
NPIX = W * H
FULL = (0, W, 0, H)
REF_OFFSET = 1 << 40
SPPS = [int(x) for x in args.spps.split(",")]
GRID = list(itertools.product([int(x) for x in args.iterations.split(",")], [float(x) for x in args.sigma_luminance.split(",")],
                              [float(x) for x in args.sigma_normal.split(",")], [float(x) for x in args.sigma_depth.split(",")]))
CONFIGS = (("C3", lambda: scenes.scene_main(), 8), ("C5", lambda: scenes.scene_main(variant="mixed"), 128))

if capi.cuda().vrj_device_count() < 1:
    sys.exit("denoise_quality.py needs a CUDA device")
smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
card = smi.stdout.strip().splitlines()[0] if smi.returncode == 0 and smi.stdout.strip() else "unknown (nvidia-smi failed)"
print("card: %s" % card, flush=True)


def y_of(colour):
    return colour.reshape(-1, 3)[:, 1]


def rel_rmse(y, ref, sel=None):
    if sel is not None:
        y, ref = y[sel], ref[sel]
    return float(np.sqrt(np.mean((y - ref) ** 2) / np.mean(ref ** 2)))


def summary(vals):
    return {"runs": vals, "median": float(np.median(vals)), "min": float(np.min(vals)), "max": float(np.max(vals))}


def frame(hs, spp, kw):
    return hs.render_adaptive(FULL, H, W, spp, spp, 1, 0.01, want=("colour", "colour_sum", "weight", "y_sq_sum"), **kw)


def params_dict(p):
    return dict(iterations=p[0], sigma_luminance=p[1], sigma_normal=p[2], sigma_depth=p[3])


# ---- phase 1: the parameter grid on every config and spp ----
state, sweep = {}, {}
for name, make_spec, depth in CONFIGS:
    hs = V.build_scene(make_spec())
    kw = dict(max_depth=depth, seed=1)
    hs.render((0, 64, 0, 64), H, W, spp=2, **kw)  # warm-up: module load, scratch blocks
    ref = y_of(hs.render(FULL, H, W, spp=args.ref_spp, want=("colour",), **dict(kw, sample_offset=REF_OFFSET))["colour"])
    aux = hs.render_aux(FULL, H, W, spp=1, want=("normal", "depth", "material"), **kw)
    specular_ids = [i for i, m in enumerate(hs.spec.materials) if m.kind in (scenes.MAT_REFLECTIVE, scenes.MAT_DIELECTRIC)]
    specular = np.isin(aux["material"], specular_ids)
    state[name] = (hs, kw, ref, aux, specular)
    for spp in SPPS:
        f = frame(hs, spp, kw)
        noisy = rel_rmse(y_of(f["colour"]), ref)
        parts = [specular, ~specular] if specular.any() else [None]
        part_noisy = [rel_rmse(y_of(f["colour"]), ref, sel) for sel in parts]
        errs, worst = [], []
        for p in GRID:
            g = host.denoise(f["colour_sum"], f["weight"], f["y_sq_sum"], aux, W, H, **params_dict(p))
            errs.append(rel_rmse(y_of(g["colour"]), ref))
            worst.append(max(np.log(rel_rmse(y_of(g["colour"]), ref, sel) / e0) for sel, e0 in zip(parts, part_noisy)))
        sweep[(name, spp)] = (noisy, errs, worst)
        best = int(np.argmin(errs))
        print("%s %3d spp: noisy %.4f, best denoised %.4f at %s" % (name, spp, noisy, errs[best], params_dict(GRID[best])), flush=True)

score = [float(np.mean([worst[i] for _, _, worst in sweep.values()])) for i in range(len(GRID))]
chosen = GRID[int(np.argmin(score))]
print("chosen: %s (geometric mean of the worst part's denoised / noisy error %.3f)" % (params_dict(chosen), float(np.exp(min(score)))),
      flush=True)

# ---- phase 2: timings and the equal-time comparison with the chosen parameters ----
results = {"card": card, "width": W, "height": H, "ref_spp": args.ref_spp, "repeats": args.repeats, "chosen": params_dict(chosen),
           "grid": [params_dict(p) for p in GRID], "configs": {}}
for name, _, depth in CONFIGS:
    hs, kw, ref, aux, specular = state[name]
    res = {"max_depth": depth, "specular_first_hit_pixels": int(specular.sum()), "spp": {}}
    aux_ms = []
    for r in range(args.repeats + 1):
        aux_ms.append(hs.render_aux(FULL, H, W, spp=1, want=("normal", "depth", "material"), **kw)["stats"].device_ms)
    res["aux_device_ms"] = summary(aux_ms[1:])
    for spp in SPPS:
        noisy, errs, _ = sweep[(name, spp)]
        render_ms, den_ms = [], []
        for r in range(args.repeats + 1):
            f = frame(hs, spp, kw)
            render_ms.append(f["stats"].device_ms)
            g = host.denoise(f["colour_sum"], f["weight"], f["y_sq_sum"], aux, W, H, **params_dict(chosen))
            den_ms.append(g["device_ms"])
        clean = rel_rmse(y_of(g["colour"]), ref)
        spec_err = {}
        if specular.any():
            for part, sel in (("specular", specular), ("other", ~specular)):
                spec_err[part] = {"noisy": rel_rmse(y_of(f["colour"]), ref, sel), "denoised": rel_rmse(y_of(g["colour"]), ref, sel)}
        total = float(np.median(render_ms[1:]) + np.median(aux_ms[1:]) + np.median(den_ms[1:]))
        u_ms = [hs.render(FULL, H, W, spp=spp, want=("colour",), **kw)["stats"].device_ms for r in range(args.repeats)]
        eq_spp = max(1, int(round(total / (float(np.median(u_ms)) / spp))))
        eq_ms = []
        for r in range(args.repeats):
            u = hs.render(FULL, H, W, spp=eq_spp, want=("colour",), **kw)
            eq_ms.append(u["stats"].device_ms)
        eq_err = rel_rmse(y_of(u["colour"]), ref)
        row = {"render_device_ms": summary(render_ms[1:]), "denoise_device_ms": summary(den_ms[1:]), "uniform_device_ms": summary(u_ms),
               "total_device_ms": total, "rel_rmse_y_noisy": noisy, "rel_rmse_y_denoised": clean,
               "rel_rmse_y_best_in_grid": float(min(errs)), "best_in_grid": params_dict(GRID[int(np.argmin(errs))]),
               "uniform_equal_time": {"spp": eq_spp, "device_ms": summary(eq_ms), "rel_rmse_y": eq_err},
               "denoised_beats_equal_time_uniform": bool(clean < eq_err), "by_first_hit": spec_err}
        res["spp"][str(spp)] = row
        print("%s %3d spp: render %.2f ms + aux %.2f ms + denoise %.2f ms = %.2f ms | relRMSE Y noisy %.4f -> denoised %.4f | "
              "uniform at equal time: %d spp %.2f ms relRMSE %.4f -> %s" %
              (name, spp, row["render_device_ms"]["median"], res["aux_device_ms"]["median"], row["denoise_device_ms"]["median"], total,
               noisy, clean, eq_spp, row["uniform_equal_time"]["device_ms"]["median"], eq_err,
               "denoised wins" if clean < eq_err else "uniform wins"), flush=True)
        for part, e in spec_err.items():
            print("    %s first hits: noisy %.4f -> denoised %.4f" % (part, e["noisy"], e["denoised"]), flush=True)
    results["configs"][name] = res
with open(args.out, "w") as f:
    json.dump(results, f, indent=1)
print("wrote %s" % args.out)
