#!/usr/bin/env python
"""bench.py -- Mrays/s and spp/s of the path-traced "bunny" frame (BASELINE.json metric).

Workload (config C3 of SURVEY.md 8d): src/main.rs scene (plane + 3 spheres + bunny BVH, all
Lambertian), 1920x1080, SimpleRandomIntegrator, recursion limit 8, seed 1.  One "step" = one pass of
the hot path over one batch: --spp samples per pixel of the whole frame on EACH GPU (weak scaling:
GPU g of G renders samples g, g+G, g+2G, ...) into one [npix x 4] (sum X, sum Y, sum Z, sum w) device
buffer, followed, for G > 1, by ONE NCCL reduce of that buffer into rank 0 (issued asynchronously: the
reduce of step k overlaps the rendering of step k+1) and the addition into rank 0's frame.

    python bench.py --gpus 1 --steps K --warmup W                     (one JSON line)
    python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...
    python bench.py --impl reference ...     the reference's algorithm on the host cores (CPU oracle)
    python bench.py ... --dump-outputs DIR   also writes the frame of the timed steps as DIR/*.npy (same arguments, same inputs)

Besides the contract's keys the line carries: `reduce_check` (the reduced frame's weights and an oracle crop),
`strong` (one fixed-size frame, --total-spp samples split over the ranks), `e2e_ref_signature` (the reference's own
calling pattern: worker threads issuing 1-spp, limit-128 partial_render_scene calls + host merge_tile),
`sharded_check` (vrj_render_sharded, the C-ABI multi-GPU path, against one GPU) and `extra_configs` (C2, C4, C5).

The Stanford bunny OBJ is a Git-LFS pointer in the reference snapshot; unless $VANRIJN_BUNNY_OBJ points at
the real file the mesh is the deterministic 81 920-triangle proxy (vanrijn_b200/scenes.py), and
`config.mesh` says so.
"""
import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))  # oraclelib: used ONLY by the checks, the cpu_baseline and the reference leg

WIDTH, HEIGHT, MAX_DEPTH, SEED = 1920, 1080, 8, 1


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--spp", type=int, default=64, help="samples per pixel per step per GPU (one wavefront batch up to 64 at 1080p)")
    ap.add_argument("--total-spp", type=int, default=1024, help="samples per pixel of the strong-scaling frame (config C3: 1024), split over the GPUs")
    ap.add_argument("--width", type=int, default=WIDTH)
    ap.add_argument("--height", type=int, default=HEIGHT)
    ap.add_argument("--filter", default="f32", choices=["f32", "f64", "f32x4", "q16"],
                    help="conservative BVH box filter: 2-wide f32, 2-wide f64, 4-wide f32 or 16-bit nodes (results identical)")
    ap.add_argument("--precision", default="f64", choices=["f64", "f32"],
                    help="f64 = the reference's type (parity path, the headline); f32 = VRJ_PRECISION_F32_FAST, reported separately")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip strong / e2e_ref_signature / sharded_check / extra_configs")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the frame they left (colour_sum, weight) to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


DUMP_BYTES = 64 * 10 ** 6  # at most this much .npy data from --dump-outputs


def dump_outputs(out_dir, frame, H, W):
    """The timed path's result as its caller holds it after the last step: the frame's per-pixel XYZ sums (float64) and
    sample weights (float32: whole sample counts, exact).  A frame too large for DUMP_BYTES is reduced to a fixed, seeded
    sample of pixels, whose row-major indices go to pixel_index.npy."""
    import numpy as np
    npix = H * W
    f = frame.cpu().numpy()
    colour_sum, weight = f[:npix * 3].reshape(npix, 3), f[npix * 3:].astype(np.float32)
    per_pixel = colour_sum.itemsize * 3 + weight.itemsize
    if npix * per_pixel <= DUMP_BYTES:
        arrays = {"colour_sum": colour_sum.reshape(H, W, 3), "weight": weight.reshape(H, W)}
    else:
        n = (DUMP_BYTES - 4096) // (per_pixel + 8)  # 4 KB left for the .npy headers
        idx = np.sort(np.random.default_rng(0).choice(npix, n, replace=False))
        arrays = {"colour_sum": colour_sum[idx], "weight": weight[idx], "pixel_index": idx.astype(np.float64)}
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.ascontiguousarray(a))


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        try:
            return float(json.load(open(path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, device):
        self.device = device
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.device), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[1]))
                mx.append(float(r[2]))
                for n, v in zip(names, r[4:8]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            except Exception:
                continue
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def oracle_scene(spec):
    import oraclelib as O
    return O, O.OracleScene(spec)


def cpu_sample(orc_mod, orc, width, height, spp, traverse, threads=0, depth=MAX_DEPTH):
    """One bounded sample of the workload on the host cores: the full frame at reduced resolution."""
    t0 = time.perf_counter()
    r = orc.render((0, width, 0, height), height, width, spp=spp, max_depth=depth, seed=SEED, traverse=traverse,
                   threads=threads)
    dt = time.perf_counter() - t0
    return r["stats"], dt


def run_reference(args, spec, mesh_name):
    """--impl reference: the reference's own algorithm for the path (reference-order BVH traversal, f64) on
    the host cores.  The Rust crate cannot be built in this image (no cargo/rustc), so this is the C++
    oracle port; it omits the Rust version's per-call heap allocations, i.e. it is a favourable stand-in."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    O, orc = oracle_scene(spec)
    cores = os.cpu_count() or 1
    sw, sh, sspp = args.width, args.height, 4  # one step = 4 spp of the full frame (~15 M ray queries, ~1.3 s on 16 cores)
    for _ in range(max(1, args.warmup)):
        cpu_sample(O, orc, sw, sh, sspp, O.TRAVERSE_REFERENCE)
    rays, secs = 0, 0.0
    for _ in range(args.steps):
        st, dt = cpu_sample(O, orc, sw, sh, sspp, O.TRAVERSE_REFERENCE)
        rays += st.rays
        secs += dt
    value = rays / secs / 1e6
    sample = "%dx%d full frame, %d spp per step, depth %d, reference-order traversal" % (sw, sh, sspp, MAX_DEPTH)
    line = {"impl": "reference", "metric": "Mrays/s", "value": value, "unit": "Mrays/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * secs / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "spp_per_s": (args.steps * sspp * sw * sh / (args.width * args.height)) / secs,
            "config": {"workload": "C3 main.rs scene path trace %dx%d depth %d" % (args.width, args.height, MAX_DEPTH),
                       "mesh": mesh_name, "integrator": "SimpleRandom", "sample": sample},
            "cpu_baseline": {"value": value, "unit": "Mrays/s", "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": value, "unit": "Mrays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def pinned_array(capi, np, count):
    ptr = capi.cuda().vrj_alloc_host(count * 8)
    if not ptr:
        raise SystemExit("vrj_alloc_host failed")
    return np.ctypeslib.as_array(C.cast(ptr, C.POINTER(C.c_double)), (count,))


def extra_config(name, V, capi, scenes, np, device):
    """One of BASELINE.json's other configurations at full size: a few device-timed calls, the same call end to end
    (host output arrays), and the traversal counters of the device's own ordered walk.  Outside the headline timing."""
    kw = dict(seed=SEED)
    t0 = time.perf_counter()
    if name == "C2":
        spec, lights, amb = scenes.scene_direct(subdivisions=6, obj=True)
        W, H, spp = 1920, 1080, 1
        kw.update(integrator=capi.INTEGRATOR_WHITTED, lights=lights, ambient=amb, max_depth=0)
        what = "bunny BVH, Whitted, max_depth 0, one directional light + ambient, 1 spp"
    elif name == "C4":
        spec = scenes.scene_grid(copies=11)
        W, H, spp = 3840, 2160, 15  # 15 spp at 4K = the 128 Mi-path budget of one wavefront batch
        kw.update(max_depth=8)
        what = "11 x 11 bunny copies (9 912 320 triangles) + plane, SimpleRandom, depth 8, 15 spp per call (one wavefront batch)"
    else:
        spec = scenes.scene_main(subdivisions=6, obj=True, variant="mixed")
        W, H, spp = 1920, 1080, 64  # one wavefront batch, like the bench step: the latency-bound tail (the few paths that run to
        kw.update(max_depth=128)    # the limit: ~5 ms whatever the batch size) is paid once per batch
        what = "main.rs scene with mirror sphere, diamond sphere, reflective bunny; SimpleRandom, recursion limit 128, 64 spp per call (one wavefront batch)"
    hs = V.build_scene(spec, device_builder="upload")
    t1 = time.perf_counter()
    hs.device_scene(device)
    t2 = time.perf_counter()
    npix = W * H
    pinned = {"colour": pinned_array(capi, np, npix * 3), "weight": pinned_array(capi, np, npix)}
    tile = (0, W, 0, H)
    best, e2e_best, st = None, None, None
    for i in range(10 if name == "C2" else 4):  # C2 is one 1-spp frame per call (2.4 ms): more calls for a stable best-of
        t = time.perf_counter()
        r = hs.render(tile, H, W, spp=spp, sample_offset=i * spp, want=("colour", "weight"), buffers=pinned, device=device, **kw)
        dt = time.perf_counter() - t
        st = r["stats"]
        if i == 0:
            continue  # warm-up: scratch allocation
        m = st.rays / st.device_ms / 1e3
        best = m if best is None else max(best, m)
        e = st.rays / dt / 1e6
        e2e_best = e if e2e_best is None else max(e2e_best, e)
    ok = bool(np.all(pinned["weight"] == spp) and np.all(np.isfinite(pinned["colour"])))
    rc = hs.render(tile, H, W, spp=1, want=("weight",), device=device, count_traversal=True, **kw)["stats"]
    V_, T_ = rc.node_visits / max(1, rc.rays), rc.triangle_tests / max(1, rc.rays)
    out = {"what": what, "width": W, "height": H, "spp_per_call": spp, "Mrays_per_s_device": best, "e2e_Mrays_per_s": e2e_best,
           "spp_per_s_device": spp / (st.device_ms / 1e3), "rays_per_call": st.rays, "device_ms_per_call": st.device_ms,
           "kernel_ms": {"k_trace": st.primary_ms + st.bounce_ms, "k_raygen+k_shade": st.shade_ms, "k_resolve": st.resolve_ms,
                         "k_tail": st.tail_ms},
           "launches_per_call": int(st.kernel_launches), "d2h_bytes_per_call": npix * 32,
           "V_nodes_per_ray": V_, "T_tris_per_ray": T_, "bytes_per_ray": 32.0 * V_ + 48.0 * T_ + 144.0,
           "scene_bytes": hs.device_bytes(device), "host_scene_s": t1 - t0, "upload_and_device_build_s": t2 - t1,
           "weights_ok_finite": ok}
    for a in pinned.values():
        capi.cuda().vrj_free_host(a.ctypes.data)
    del hs
    capi.cuda().vrj_release_scratch()
    return out


def main():
    args = parse()
    from vanrijn_b200 import scenes
    spec = scenes.scene_main(subdivisions=6, obj=True)
    mesh_name = scenes.bunny_obj_path()[1]
    if args.impl == "reference":
        return run_reference(args, spec, mesh_name)

    import numpy as np
    import torch
    import torch.distributed as dist
    import vanrijn_b200 as V
    from vanrijn_b200 import capi, host, sharding

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available() or capi.cuda().vrj_device_count() < 1:
        raise SystemExit("bench.py needs a CUDA device: the render loop has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    host_group = None
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
        host_group = dist.new_group(backend="gloo")  # host-side barriers that keep no kernel spinning on the GPUs

    W, H, spp = args.width, args.height, args.spp
    npix = W * H
    bvh_filter = {"f64": capi.FILTER_F64, "f32x4": capi.FILTER_F32X4, "q16": capi.FILTER_Q16}.get(args.filter, capi.FILTER_F32)
    precision = capi.PRECISION_F32_FAST if args.precision == "f32" else capi.PRECISION_F64
    hs = V.build_scene(spec)
    hs.device_scene(local)
    scene_bytes = hs.device_bytes(local)
    tile = (0, W, 0, H)
    render_kw = dict(max_depth=MAX_DEPTH, seed=SEED, bvh_filter=bvh_filter, precision=precision)
    # One [npix x 4] buffer per step in flight: (sum X, sum Y, sum Z) for every pixel, then (sum w) -- what ONE NCCL reduce
    # moves (SURVEY 8e).  k_resolve writes straight into it; there is no staging copy.  `frame` is the image so far.
    frame = torch.zeros(npix * 4, dtype=torch.float64, device=dev)
    bufs = [torch.zeros(npix * 4, dtype=torch.float64, device=dev) for _ in range(2)]
    pending = [None, None]
    samples_in_frame = 0

    def retire(i):
        """Step buffer i is about to be reused (or read): its reduce must have landed, and rank 0 adds it to the frame."""
        if pending[i] is not None:
            pending[i].wait()
            if rank == 0:
                frame.add_(bufs[i])
            pending[i] = None
            torch.cuda.current_stream().synchronize()  # the library renders on its own stream

    def step(k):
        nonlocal samples_in_frame
        # sharded by sample index: this rank renders samples offset, offset+world, ... (vanrijn_b200/sharding.py)
        offset, stride = sharding.shard_samples(rank, world, k, spp)
        if world == 1:
            # one GPU: the frame's Kahan accumulators continue in place (DeviceAccumulationBuffer semantics)
            st = hs.render_device(tile, H, W, frame.data_ptr(), frame.data_ptr() + npix * 24, device=local, accumulate=(k > 0),
                                  spp=spp, sample_offset=offset, sample_stride=stride, **render_kw)
        else:
            i = k & 1
            retire(i)
            b = bufs[i]
            st = hs.render_device(tile, H, W, b.data_ptr(), b.data_ptr() + npix * 24, device=local, accumulate=False,
                                  spp=spp, sample_offset=offset, sample_stride=stride, **render_kw)
            # the one exchange step: (sum XYZ, sum w) of all ranks into rank 0, asynchronously (NCCL over NVLink)
            pending[i] = dist.reduce(b, dst=0, op=dist.ReduceOp.SUM, async_op=True)
        samples_in_frame += spp * world
        return st

    def fence():
        if world > 1:
            retire(0), retire(1)
            dist.barrier()
        torch.cuda.synchronize()

    for k in range(args.warmup):
        step(k)
    fence()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    agg = {"rays": 0, "launches": 0, "device_ms": 0.0, "trace_ms": 0.0, "trace_launches": 0, "staged": 0,
           "shade_ms": 0.0, "resolve_ms": 0.0, "tail_ms": 0.0, "primary": 0, "bounce": 0, "shade_launches": 0}
    fence()
    t0 = time.perf_counter()
    for k in range(args.steps):
        st = step(args.warmup + k)
        agg["rays"] += st.rays
        agg["launches"] += int(st.kernel_launches) + (1 if world > 1 else 0)
        agg["device_ms"] += st.device_ms
        agg["trace_ms"] += st.primary_ms + st.bounce_ms
        agg["trace_launches"] += int(st.primary_launches + st.bounce_launches)
        agg["staged"] += int(st.staged_rays)
        agg["shade_ms"] += st.shade_ms
        agg["resolve_ms"] += st.resolve_ms
        agg["tail_ms"] += st.tail_ms
        agg["primary"] += int(st.primary_rays)
        agg["bounce"] += int(st.bounce_rays)
        agg["shade_launches"] += int(st.shade_launches)
    fence()
    wall = time.perf_counter() - t0
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, frame, H, W)

    # ---- reduce_check (outside the timed region): the frame on rank 0 holds every sample of every rank exactly once
    reduce_check = None
    if rank == 0:
        try:
            total_spp = samples_in_frame
            wts = frame[npix * 3:]
            if not bool(torch.all(wts == float(total_spp))):
                raise AssertionError("weights differ from %d" % total_spp)
            O, orc = oracle_scene(spec)
            c0, r0, cw, ch = (W * 5) // 8, (H * 5) // 8, 12, 8   # a crop on the bunny and the floor under it
            if c0 + cw > W or r0 + ch > H:
                c0, r0, cw, ch = 0, 0, min(W, 12), min(H, 8)
            ref = orc.render((c0, c0 + cw, r0, r0 + ch), H, W, spp=total_spp, max_depth=MAX_DEPTH, seed=SEED,
                             traverse=O.TRAVERSE_ORDERED)
            got = frame[:npix * 3].view(H, W, 3)[r0:r0 + ch, c0:c0 + cw].cpu().numpy().reshape(-1)
            want = ref["colour_sum"]
            err = float(np.max(np.abs(got - want) / np.maximum(np.abs(want), 1e-30)))
            if precision == capi.PRECISION_F64 and not err < 1e-9:
                raise AssertionError("crop differs from the oracle: %.3e" % err)
            reduce_check = {"status": "ok", "weight_all_pixels": total_spp, "ranks": world,
                            "oracle_crop": "%dx%d at (%d,%d), %d spp" % (cw, ch, c0, r0, total_spp), "max_rel_err": err}
        except Exception as e:  # reported, never hidden
            reduce_check = {"status": "FAILED: %s" % e}

    # ---- strong scaling: ONE frame of --total-spp samples per pixel split over the ranks, one reduce at the end
    strong = None
    if not args.no_extra:
        per_rank = [args.total_spp // world + (1 if g < args.total_spp % world else 0) for g in range(world)]
        mine = per_rank[rank]
        b = bufs[0]
        fence()
        ts = time.perf_counter()
        st = None
        if mine:
            st = hs.render_device(tile, H, W, b.data_ptr(), b.data_ptr() + npix * 24, device=local, accumulate=False, spp=mine,
                                  sample_offset=rank, sample_stride=world, **render_kw)
        else:
            b.zero_()
        if world > 1:
            dist.reduce(b, dst=0, op=dist.ReduceOp.SUM)
        fence()
        t_strong = time.perf_counter() - ts
        tt = torch.tensor([t_strong, float(st.rays if st else 0), float(st.device_ms if st else 0.0)], dtype=torch.float64, device=dev)
        if world > 1:
            tmax = tt.clone()
            dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
            dist.all_reduce(tt, op=dist.ReduceOp.SUM)
            t_strong, dev_ms_max = float(tmax[0]), float(tmax[2])
        else:
            dev_ms_max = float(tt[2])
        if rank == 0:
            okw = bool(torch.all(b[npix * 3:] == float(args.total_spp)))
            strong = {"scaling": "strong", "total_spp": args.total_spp, "n_gpus": world, "frame_ms": 1e3 * t_strong,
                      "device_ms_max_over_ranks": dev_ms_max, "value": float(tt[1]) / t_strong / 1e6, "unit": "Mrays/s",
                      "spp_per_s": args.total_spp / t_strong, "weights_ok": okw,
                      "what": "one %dx%d frame of %d spp sharded by sample index over %d GPU(s) + one NCCL reduce; wall clock "
                              "between fences, max over ranks" % (W, H, args.total_spp, world)}

    # ---- end-to-end: the public call with HOST buffers, every step.  Per step every rank uploads the scene as the host
    # holds it before any device work (primitives + the mesh's triangles in file order; the BVH is built on the device
    # inside vrj_scene_create), renders its sample shard, the shards are reduced to rank 0, and rank 0 alone copies the
    # frame's (colour, weight) -- what AccumulationBuffer::merge_tile and to_image_rgb_u8 read -- to page-locked host memory.
    hs_e2e = V.build_scene(spec, device_builder="upload")
    desc = hs_e2e.desc()
    e2e_rays, e2e_secs, e2e_create, upload_bytes, e2e_steps = 0, 0.0, 0.0, 0, 0
    out_bytes = npix * 4 * 8
    pinned = {"colour": pinned_array(capi, np, npix * 3), "weight": pinned_array(capi, np, npix)}
    host_frame = torch.empty(npix * 4, dtype=torch.float64).pin_memory() if (world > 1 and rank == 0) else None
    fence()
    for k in range(args.steps + 1):
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()
        t1 = time.perf_counter()
        h = C.c_void_p()
        capi.check(capi.cuda().vrj_scene_create(C.byref(desc), local, C.byref(h)))   # H2D: the flattened scene
        t2 = time.perf_counter()
        upload_bytes = int(capi.cuda().vrj_scene_upload_bytes(h))
        hs._dev["e2e"] = h
        off, stride = sharding.shard_samples(rank, world, k, spp)
        if world == 1:
            r = hs.render(tile, H, W, device="e2e", buffers=pinned, want=("colour", "weight"), spp=spp, sample_offset=off,
                          sample_stride=stride, **render_kw)                                                # D2H: colour + weight
            rays_k = r["stats"].rays
        else:
            b = bufs[0]
            st = hs.render_device(tile, H, W, b.data_ptr(), b.data_ptr() + npix * 24, device="e2e", accumulate=False, spp=spp,
                                  sample_offset=off, sample_stride=stride, **render_kw)
            dist.reduce(b, dst=0, op=dist.ReduceOp.SUM)
            if rank == 0:
                host_frame.copy_(b, non_blocking=True)                                                        # D2H: rank 0 only
            torch.cuda.synchronize()
            rays_k = st.rays
        capi.cuda().vrj_scene_destroy(h)
        del hs._dev["e2e"]
        dt = time.perf_counter() - t1
        if k > 0:  # the first iteration warms allocator and staging paths
            e2e_rays += rays_k
            e2e_secs += dt
            e2e_create += t2 - t1
            e2e_steps += 1
    fence()

    # ---- max over ranks / totals over ranks
    t = torch.tensor([wall, e2e_secs, agg["device_ms"]], dtype=torch.float64, device=dev)
    c = torch.tensor([agg["rays"], e2e_rays, agg["launches"]], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(c, op=dist.ReduceOp.SUM)
    wall_max, e2e_max, devms_max = [float(x) for x in t.tolist()]
    rays_all, e2e_rays_all, launches_all = [float(x) for x in c.tolist()]

    # ---- the C-ABI multi-GPU path (vrj_comm_* / vrj_render_sharded) against one GPU: rank 0, when its process sees two GPUs.
    # The other ranks wait in a HOST barrier (gloo), so nothing of theirs runs on the devices meanwhile.
    sharded_check = None
    if rank == 0 and not args.no_extra:
        try:
            ndev = capi.cuda().vrj_device_count()
            if ndev < 2:
                sharded_check = {"status": "skipped: this process sees %d GPU" % ndev}
            else:
                small = scenes.scene_main(subdivisions=4, obj=False)
                hs2 = V.build_scene(small)
                w2, h2, spp2 = 320, 180, 6
                devs = list(range(min(ndev, 4)))
                one = hs2.render((0, w2, 0, h2), h2, w2, spp=spp2, max_depth=MAX_DEPTH, seed=3, device=0, want=("colour_sum", "weight"))
                many = hs2.render_sharded(devs, (0, w2, 0, h2), h2, w2, spp=spp2, max_depth=MAX_DEPTH, seed=3)
                if not np.array_equal(many["weight"], one["weight"]):
                    raise AssertionError("weights differ")
                err = float(np.max(np.abs(many["colour_sum"] - one["colour_sum"]) / np.maximum(np.abs(one["colour_sum"]), 1e-30)))
                if not err < 1e-12:
                    raise AssertionError("colour sums differ: %.3e" % err)
                if many["stats"].rays != one["stats"].rays:
                    raise AssertionError("ray counts differ")
                sharded_check = {"status": "ok", "devices": devs, "max_rel_err_vs_one_gpu": err, "rays": int(one["stats"].rays),
                                 "what": "vrj_comm_create + vrj_comm_scene_create + vrj_render_sharded (ncclReduce inside the library)"}
                del hs2
        except Exception as e:
            sharded_check = {"status": "FAILED: %s" % e}
    if world > 1:
        dist.barrier(group=host_group)
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- the reference's own calling pattern (main.rs:192-217): worker threads issue partial_render_scene calls with the
    # reference's hard-coded parameters (1 spp, recursion limit 128, whole-frame tile), each returning a host
    # AccumulationBuffer; the calling thread merge_tile()s.  Two forms: the buffer as the reference type has it (five
    # arrays, 182 MB per call) and carrying colour + weight only (all merge_tile reads; 66 MB per call).
    ref_sig = None
    if world == 1 and not args.no_extra:
        try:
            ref_sig = {"what": "N worker threads x partial_render_scene(scene, tile, h, w) [1 spp, RECURSION_LIMIT 128, whole-frame tile] + "
                               "merge_tile on the calling thread, as src/main.rs:192-217; wall clock of the whole loop.  colour_only: the "
                               "tile buffer carries what merge_tile reads (colours + one weight); five_arrays: the reference type's five arrays",
                       "bounds_per_call": {"d2h_colour_only_bytes": npix * 24, "d2h_five_arrays_bytes": npix * 88,
                                           "merge_tile_bytes_read_written": npix * (32 + 24 + 32)}}
            best = None
            for key, kahan, calls in (("colour_only", False, 192), ("five_arrays", True, 48)):
                for workers in (4, 8):
                    host.render_like_main(hs, W, H, 6 * workers, workers, kahan_state=kahan, device=local)   # warm-up: scratch blocks, pinned pool
                    colour, weight, st = host.render_like_main(hs, W, H, calls, workers, kahan_state=kahan, device=local)
                    if not np.all(weight == calls):
                        raise AssertionError("merged weights differ from %d" % calls)
                    r = {"value": st["rays"] / st["wall_s"] / 1e6, "unit": "Mrays/s", "threads": workers, "calls": calls,
                         "ms_per_call": 1e3 * st["wall_s"] / calls, "d2h_bytes_per_call": st["bytes_to_host"] / calls,
                         "merge_tile_ms_per_call": 1e3 * st["merge_s"] / calls, "device_ms_per_call": st["device_ms"] / calls,
                         "worker_ms_per_call": 1e3 * st["call_s"] / calls, "spp_per_s": calls / st["wall_s"],
                         "merge_passes": int(st["merge_passes"]), "calls_per_wavefront": st["wavefront_calls"] / calls}
                    ref_sig["%s_%d_threads" % (key, workers)] = r
                    if key == "colour_only" and (best is None or r["value"] > best["value"]):
                        best = r
            ref_sig["value"], ref_sig["unit"], ref_sig["threads"] = best["value"], "Mrays/s", best["threads"]
        except Exception as e:
            ref_sig = {"status": "FAILED: %s" % e}

    extra = None
    if world == 1 and not args.no_extra:
        extra = {}
        for name in ("C2", "C5", "C4"):
            try:
                extra[name] = extra_config(name, V, capi, scenes, np, local)
            except Exception as e:
                extra[name] = {"status": "FAILED: %s" % e}

    # ---- rank 0: rooflines and the CPU baseline
    peak, peak_src = peaks()
    O, orc = oracle_scene(spec)
    sw, sh = W // 8, H // 8
    st_ord, _ = cpu_sample(O, orc, sw, sh, 1, O.TRAVERSE_ORDERED)   # V, T of the ordered + pruned walk (SURVEY 8d)
    V_ = st_ord.node_visits / st_ord.rays
    T_ = st_ord.tri_tests / st_ord.rays
    bytes_per_ray = 32.0 * V_ + 48.0 * T_ + 144.0
    kernel_ms = {"k_trace": agg["trace_ms"], "k_raygen+k_shade": agg["shade_ms"], "k_resolve": agg["resolve_ms"]}
    dominant = max(kernel_ms, key=kernel_ms.get)
    traffic = {}
    tpath = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tpath):
        try:
            traffic = json.load(open(tpath))
        except Exception:
            traffic = {}
    # k_raygen + k_shade stream the path queues through HBM.  Algorithmic bytes: a primary path reads its 16-byte hit record
    # and writes a 16-byte result; every bounce ray is written once (96 B state + 16 B stage-1 hit + 4 B list entry) and read
    # once (96 B + 16 B) by the next level: 32 B per primary path + 228 B per bounce ray.
    shade_bytes = 32.0 * agg["primary"] + 228.0 * agg["bounce"]
    shade_s = agg["shade_ms"] / 1e3
    shade_ach = shade_bytes / shade_s / 1e9 if shade_s > 0 else 0.0
    # k_trace fetches 64-byte node records (one per two box tests) and triangle records at data-dependent addresses from a
    # scene that is L2-resident by design: its yard-stick is the measured rate of dependent 64-byte gathers from L2
    # (tools/l2_gather_peak.cu -> profiles/r02_l2_gather_peak.json), not HBM.
    trace_s = agg["trace_ms"] / 1e3
    trace_bytes = (32.0 * V_ + 48.0 * T_) * agg["rays"] + 64.0 * agg["staged"]
    trace_ach = trace_bytes / trace_s / 1e9 if trace_s > 0 else 0.0
    l2_peak, l2_src = None, "profiles/r02_l2_gather_peak.json missing"
    gpath = os.path.join(ROOT, "profiles", "r02_l2_gather_peak.json")
    if os.path.exists(gpath):
        try:
            g = json.load(open(gpath))
            # the traversal's own access pattern without its arithmetic: root-to-leaf walks of a median-split tree of the bench
            # mesh's size (top levels from L1, the rest from L2), every lane on a path of its own
            walk = [r for r in g["tree_walk"]["results"] if r["leaves"] == 81920 and r["ctas_per_sm"] == 6]
            l2_peak = walk[0]["GBps"]
            l2_src = ("measured: root-to-leaf walks of a 5 MB median-split tree, one 64-byte record per step, one walk per lane, 6 CTAs/SM "
                      "(tools/l2_gather_peak.cu -> profiles/r02_l2_gather_peak.json tree_walk); uniform dependent gathers from L2 reach "
                      "%.0f GB/s.  Lanes of a warp that fetch the same record share one access, which the walk on incoherent paths "
                      "does not model: camera rays can exceed it" % [r for r in g["results"] if r.get("record_bytes", 64) == 64 and r["table_mb"] == 5 and r["ctas_per_sm"] == 6][0]["GBps_1chain"])
        except Exception:
            pass
    step_achieved = bytes_per_ray * agg["rays"] / (agg["device_ms"] / 1e3) / 1e9
    per_kernel = {
        "k_raygen+k_shade": {"bound": "hbm", "achieved": shade_ach, "peak": peak, "unit": "GB/s", "frac": shade_ach / peak,
                             "algorithmic_bytes_per_launch": shade_bytes / max(1, agg["shade_launches"]),
                             "avg_launch_ms": agg["shade_ms"] / max(1, agg["shade_launches"]),
                             "share_of_step": agg["shade_ms"] / max(1e-9, agg["device_ms"]),
                             "traffic": traffic.get("k_shade_dram_bytes_per_launch"),
                             "what": "32 B per primary path + 228 B per bounce ray / CUDA-event time of the k_raygen and k_shade launches; "
                                     "the kernels are bound by binary64 issue and latency, not by this stream (DESIGN 3.2)"},
        "k_trace": {"bound": "l2-gather", "achieved": trace_ach, "peak": l2_peak, "unit": "GB/s",
                    "frac": (trace_ach / l2_peak) if l2_peak else None, "peak_source": l2_src,
                    "frac_of_hbm": trace_ach / peak,
                    "algorithmic_bytes_per_launch": trace_bytes / max(1, agg["trace_launches"]),
                    "avg_launch_ms": agg["trace_ms"] / max(1, agg["trace_launches"]),
                    "share_of_step": agg["trace_ms"] / max(1e-9, agg["device_ms"]),
                    "traffic": traffic.get("k_trace_dram_bytes_per_launch"),
                    "what": "(32 V + 48 T) B x all ray queries + 64 B per staged ray / CUDA-event time of the k_trace launches; V, T = the "
                            "oracle's ordered + pruned per-query means (SURVEY 8d)"},
    }
    dom = per_kernel.get(dominant, per_kernel["k_raygen+k_shade"])
    roofline = {"bound": "hbm", "kernel": dominant, "achieved": dom["achieved"], "peak": peak, "unit": "GB/s",
                "frac": dom["achieved"] / peak, "traffic": dom.get("traffic"), "peak_source": peak_src,
                "algorithmic_bytes_per_launch": dom["algorithmic_bytes_per_launch"], "avg_launch_ms": dom["avg_launch_ms"],
                "kernel_share_of_step": dom["share_of_step"],
                "bytes_per_ray": bytes_per_ray, "V_nodes_per_ray": V_, "T_tris_per_ray": T_,
                "whole_step": {"achieved": step_achieved, "frac": step_achieved / peak,
                               "what": "SURVEY 8d: bytes_per_ray (32 V + 48 T + 144) x all ray queries / CUDA-event time of all kernels of the step"},
                "kernels": per_kernel,
                "note": "`kernel` is the kernel class with the largest share of the step's CUDA-event time; both classes are listed "
                        "under `kernels`.  The scene (BVH + triangles) is L2-resident by design, so k_trace is measured against an "
                        "L2 gather peak, with its fraction of the HBM figure given for reference only."}
    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        cores = os.cpu_count() or 1
        cw, ch, cspp = W, H, min(spp, 32)  # the full frame at half the step's spp: ~10 s of CPU
        cpu_sample(O, orc, W // 8, H // 8, 1, O.TRAVERSE_REFERENCE)  # warm-up
        st_ref, dt = cpu_sample(O, orc, cw, ch, cspp, O.TRAVERSE_REFERENCE)
        cpu = {"value": st_ref.rays / dt / 1e6, "unit": "Mrays/s", "cores": cores, "kind": "port",
               "sample": "%dx%d full frame x %d spp, depth %d, reference-order traversal, %.1f s" % (cw, ch, cspp, MAX_DEPTH, dt)}

    value = rays_all / wall_max / 1e6
    line = {"metric": "Mrays/s", "value": value, "unit": "Mrays/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * wall_max / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32" if args.precision == "f32" else "f64", "data": "synthetic",
            "spp_per_s": args.steps * spp * world / wall_max,
            "device_ms_per_step": devms_max / args.steps,
            "config": {"workload": "C3 main.rs scene path trace %dx%d depth %d" % (W, H, MAX_DEPTH), "mesh": mesh_name,
                       "integrator": "SimpleRandom", "spp_per_step_per_gpu": spp, "bvh_filter": args.filter,
                       "precision": "f32-fast (no parity claim)" if args.precision == "f32" else "f64 (the reference's type)",
                       "sharding": "sample index mod n_gpus; one NCCL reduce of the [npix x 4] (sumXYZ, weight) buffer to rank 0 per step, "
                                   "overlapped with the next step's rendering",
                       "l2": "inputs larger than L2: %.1f GB of path state per step; the %.0f MB scene is L2-resident by design"
                             % (min(spp, (1 << 27) // npix) * npix * 336 / 1e9, scene_bytes / 1e6)},
            "e2e": {"value": e2e_rays_all / e2e_max / 1e6, "unit": "Mrays/s", "h2d_bytes_per_step": int(upload_bytes) * world,
                    "d2h_bytes_per_step": int(out_bytes), "steps": e2e_steps,
                    "ms_per_step": 1e3 * e2e_max / e2e_steps, "scene_upload_ms_per_step": 1e3 * e2e_create / e2e_steps,
                    "what": "per step: vrj_scene_create from the host's triangles on every rank (BVH built on the device) + vrj_render_tile of "
                            "the rank's sample shard" + (" into page-locked host (colour, weight) arrays" if world == 1 else
                                                         " + one NCCL reduce to rank 0 + rank 0 copies the frame's (sumXYZ, weight) to page-locked host memory") +
                            " + vrj_scene_destroy"},
            "gpu_launches": int(launches_all), "clocks": clocks, "roofline": roofline, "cpu_baseline": cpu,
            "kernel_ms": dict(kernel_ms, k_tail=agg["tail_ms"]),
            "reduce_check": reduce_check, "strong": strong, "sharded_check": sharded_check,
            "e2e_ref_signature": ref_sig, "extra_configs": extra}
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
