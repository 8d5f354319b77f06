"""Adaptive sampling (vrj_render_adaptive) on the GPU.  Run on the B200 box with `-m gpu`.

The bar is bit equality throughout: a pixel that ends with n samples must hold exactly what vrj_render_tile with spp = n
gives it, and the stopping rule and pass schedule, replayed in numpy from the per-sample Y values, must predict every
pixel's count and its y_sq_sum."""
import ctypes as C
import threading

import numpy as np
import pytest

import vanrijn_b200 as V
from vanrijn_b200 import capi, scenes
from vanrijn_b200.capi import dp

pytestmark = pytest.mark.gpu

ARRAYS = (("colour", 3), ("colour_sum", 3), ("colour_bias", 3), ("weight", 1), ("weight_bias", 1))
W, H = 37, 23                 # odd image
TILE = (5, 30, 3, 20)         # odd tile: 25 x 17 pixels
NPIX = (TILE[1] - TILE[0]) * (TILE[3] - TILE[2])
MIN, PASS, MAX = 4, 4, 32


def bits(a):
    return np.ascontiguousarray(a).view(np.uint64)


def small_scene(whitted):
    spec = scenes.scene_main(subdivisions=2, obj=False)
    kw = dict(max_depth=6, seed=3)
    if whitted:
        light = spec.spectrum("grey", 1.0)
        kw.update(integrator=capi.INTEGRATOR_WHITTED, lights=[((1.0, 1.0, -1.0), light)])
    return V.build_scene(spec), kw


def adaptive_device(hs, tile, height, width, min_samples, max_samples, pass_samples, rel_error, abs_floor=0.0, **kw):
    """vrj_render_adaptive with every output (y_sq_sum included) in device memory, copied back afterwards."""
    L = capi.cuda()
    sc, ec, sr, er = tile
    npix = (ec - sc) * (er - sr)
    p, keep = hs.make_params(spp=0, **kw)
    ap = capi.AdaptiveParams(min_samples=min_samples, max_samples=max_samples, pass_samples=pass_samples,
                             rel_error=rel_error, abs_floor=abs_floor)
    ao = capi.AccumOut(memory=capi.MEM_DEVICE, accumulate=0)
    dev = {}
    for name, per in ARRAYS + (("y_sq_sum", 1),):
        dev[name] = (L.vrj_alloc_device(0, npix * per * 8), per)
        assert dev[name][0]
        if name != "y_sq_sum":
            setattr(ao, name, dev[name][0])
    st, ast = capi.Stats(), capi.AdaptiveStats()
    ao.stats = C.pointer(st)
    t = capi.Tile(*tile)
    try:
        capi.check(L.vrj_render_adaptive(hs.device_scene(0), C.byref(t), height, width, C.byref(p), C.byref(ap), C.byref(ao),
                                         dev["y_sq_sum"][0], C.byref(ast)))
        out = {}
        for name, (ptr, per) in dev.items():
            out[name] = np.zeros(npix * per)
            capi.check(L.vrj_copy_to_host(0, out[name].ctypes.data, ptr, npix * per * 8))
    finally:
        for ptr, _ in dev.values():
            L.vrj_free_device(ptr)
    out["stats"], out["adaptive"] = st, ast
    return out


def render_adaptive(hs, memory, *args, **kw):
    if memory == capi.MEM_DEVICE:
        return adaptive_device(hs, *args, **kw)
    return hs.render_adaptive(*args, **kw)


def allowed_counts(lo, step, hi):
    return sorted(set(min(lo + j * step, hi) for j in range((hi - lo + step - 1) // step + 1)))


def spread_run(hs, memory, kw):
    """An adaptive render of the small tile whose counts take at least three values, some below and some at MAX."""
    for rel in (0.5, 0.3, 0.2, 0.1, 0.05, 0.02):
        a = render_adaptive(hs, memory, TILE, H, W, MIN, MAX, PASS, rel, **kw)
        counts = np.unique(a["weight"])
        if len(counts) >= 3 and counts.min() < MAX and counts.max() == MAX:
            return a, rel
    pytest.fail("no rel_error gave a spread of sample counts")


@pytest.mark.parametrize("memory", [capi.MEM_HOST, capi.MEM_DEVICE], ids=["host", "device"])
@pytest.mark.parametrize("stride,offset", [(1, 5), (2, 7)])
@pytest.mark.parametrize("precision", [capi.PRECISION_F64, capi.PRECISION_F32_FAST], ids=["f64", "f32fast"])
@pytest.mark.parametrize("whitted", [False, True], ids=["simple_random", "whitted_light"])
def test_each_pixel_equals_the_uniform_render_of_its_count(whitted, precision, stride, offset, memory):
    hs, kw = small_scene(whitted)
    kw.update(precision=precision, sample_stride=stride, sample_offset=offset)
    a, rel = spread_run(hs, memory, kw)
    assert set(np.unique(a["weight"])) <= set(allowed_counts(MIN, PASS, MAX))
    for n in np.unique(a["weight"]):
        u = hs.render(TILE, H, W, spp=int(n), **kw)
        sel = a["weight"] == n
        for name, per in ARRAYS:
            g, r = a[name].reshape(-1, per)[sel], u[name].reshape(-1, per)[sel]
            assert np.array_equal(bits(g), bits(r)), (name, int(n), rel)


def replay(Y, rel_error, abs_floor, lo, step, hi):
    """The header's pass schedule and stopping rule in numpy on the per-sample Y values Y[k, pixel] (binary64, the same
    operations in the same order: numpy never fuses a multiply-add).  Returns (count, colour_sum.y, y_sq_sum, passes,
    converged)."""
    npix = Y.shape[1]
    w, wb, s, b, q = (np.zeros(npix) for _ in range(5))
    held = np.zeros(npix, np.int64)
    active = np.ones(npix, bool)
    converged = np.zeros(npix, bool)
    count, done, passes = lo, 0, 0
    while True:
        for k in range(done, done + count):
            c = Y[k, active]
            wy = 1.0 - wb[active]
            wt = w[active] + wy
            wb[active] = (wt - w[active]) - wy
            w[active] = wt
            yy = c * 1.0 - b[active]
            ty = s[active] + yy
            b[active] = (ty - s[active]) - yy
            s[active] = ty
            q[active] = q[active] + c * c
        held[active] += count
        done += count
        passes += 1
        n, sy, qq = w[active], s[active], q[active]
        with np.errstate(all="ignore"):
            m = sy * (1.0 / n)
            v = (qq - sy * m) / (n - 1.0)
            v = np.where(v < 0.0, 0.0, v)
            t = rel_error * np.where(m > abs_floor, m, abs_floor)
            conv = v <= t * t * n
        idx = np.flatnonzero(active)
        converged[idx[conv]] = True
        if done >= hi:
            break
        active[idx[conv]] = False
        if not active.any():
            break
        count = min(step, hi - done)
    return held, s, q, passes, converged


@pytest.mark.parametrize("abs_floor", [0.0, 0.05])
def test_stopping_rule_replayed_exactly(abs_floor):
    hs, kw = small_scene(False)
    kw.update(sample_offset=11, sample_stride=1)
    a, rel = spread_run(hs, capi.MEM_HOST, dict(kw, abs_floor=abs_floor))
    # a 1-spp render's colour_sum.y is that sample's Y exactly (0 + y)
    Y = np.stack([hs.render(TILE, H, W, spp=1, **dict(kw, sample_offset=11 + k))["colour_sum"].reshape(-1, 3)[:, 1] for k in range(MAX)])
    held, s, q, passes, converged = replay(Y, rel, abs_floor, MIN, PASS, MAX)
    assert np.array_equal(held.astype(np.float64), a["weight"])
    assert np.array_equal(bits(s), bits(a["colour_sum"].reshape(-1, 3)[:, 1]))
    assert np.array_equal(bits(q), bits(a["y_sq_sum"]))
    ast, st = a["adaptive"], a["stats"]
    assert ast.passes == passes
    assert ast.pixels_converged == int(converged.sum()) and ast.pixels_unconverged == NPIX - int(converged.sum())
    assert ast.samples == st.primary_rays == int(a["weight"].sum()) == int(held.sum())


@pytest.mark.parametrize("whitted", [False, True], ids=["simple_random", "whitted_light"])
def test_min_equal_max_is_the_uniform_call(whitted):
    hs, kw = small_scene(whitted)
    want = ("colour", "colour_sum", "colour_bias", "weight", "weight_bias", "srgb8")
    full = (0, W, 0, H)
    a = hs.render_adaptive(full, H, W, 8, 8, 3, 0.01, want=want + ("y_sq_sum",), **kw)
    u = hs.render(full, H, W, spp=8, want=want, **kw)
    for name, _ in ARRAYS:
        assert np.array_equal(bits(a[name]), bits(u[name])), name
    assert np.array_equal(a["srgb8"], u["srgb8"])
    ast = a["adaptive"]
    assert ast.passes == 1 and ast.samples == 8 * W * H == a["stats"].primary_rays == u["stats"].primary_rays
    assert ast.pixels_converged + ast.pixels_unconverged == W * H
    for name in ("bounce_rays", "shadow_rays", "paths_missed", "paths_escaped", "paths_depth_limited"):
        assert getattr(a["stats"], name) == getattr(u["stats"], name), name


def test_argument_errors_and_empty_tile():
    hs, kw = small_scene(False)
    L = capi.cuda()
    scene = hs.device_scene(0)
    t = capi.Tile(*TILE)

    def call(ap_kw, spp=0, **ao_kw):
        p, keep = hs.make_params(spp=spp, **kw)
        ap = capi.AdaptiveParams(**dict(dict(min_samples=4, max_samples=8, pass_samples=2, rel_error=0.1), **ap_kw))
        buf = np.zeros(NPIX * 32)
        ao = capi.AccumOut(memory=capi.MEM_HOST, colour=buf.ctypes.data, **ao_kw)
        return L.vrj_render_adaptive(scene, C.byref(t), H, W, C.byref(p), C.byref(ap), C.byref(ao), None, None)

    assert call({}) == capi.OK
    for ap_kw, spp in [(dict(min_samples=1), 0), (dict(min_samples=8, max_samples=4), 0), (dict(pass_samples=0), 0),
                       (dict(rel_error=0.0), 0), (dict(rel_error=-1.0), 0), (dict(rel_error=float("nan")), 0),
                       (dict(rel_error=float("inf")), 0), (dict(abs_floor=-1.0), 0), ({}, 4)]:
        assert call(ap_kw, spp) == 1, (ap_kw, spp)  # VRJ_ERR_INVALID_ARGUMENT
        assert L.vrj_last_error().decode(), (ap_kw, spp)
    photons = np.zeros(NPIX * 16)
    assert call({}, accumulate=1) == 3  # VRJ_ERR_UNSUPPORTED
    assert b"accumulate" in L.vrj_last_error()
    assert call({}, photons=photons.ctypes.data) == 3
    assert b"photons" in L.vrj_last_error()
    e = hs.render_adaptive((4, 4, 0, H), H, W, 4, 8, 2, 0.1, **kw)
    assert e["adaptive"].passes == 0 and e["adaptive"].samples == 0 and e["stats"].primary_rays == 0


def test_c5_full_size_and_concurrent_with_a_uniform_call():
    """C5 (mixed materials, recursion limit 128) at 1920x1080: counts in the allowed set, converged pixels finite, fewer
    samples than the uniform max; then the same call concurrently with a vrj_render_tile on the same scene from another thread,
    each result equal to its single-call result."""
    hs = V.build_scene(scenes.scene_main(variant="mixed"))
    W5, H5 = 1920, 1080
    full = (0, W5, 0, H5)
    npix = W5 * H5
    kw = dict(max_depth=128, seed=5)
    a = hs.render_adaptive(full, H5, W5, 4, 64, 4, 0.25, want=("colour", "colour_sum", "weight", "y_sq_sum"), **kw)
    w = a["weight"]
    assert set(np.unique(w)) <= set(allowed_counts(4, 4, 64))
    stopped = w < 64
    assert stopped.any()
    assert np.all(np.isfinite(a["colour"].reshape(-1, 3)[stopped]))
    ast = a["adaptive"]
    assert ast.samples == int(w.sum()) == a["stats"].primary_rays and ast.samples < npix * 64
    assert ast.pixels_converged + ast.pixels_unconverged == npix
    u = hs.render(full, H5, W5, spp=8, want=("colour", "weight"), **dict(kw, sample_offset=1000))
    res = {}

    def run_uniform():
        res["u"] = hs.render(full, H5, W5, spp=8, want=("colour", "weight"), **dict(kw, sample_offset=1000))

    th = threading.Thread(target=run_uniform)
    th.start()
    a2 = hs.render_adaptive(full, H5, W5, 4, 64, 4, 0.25, want=("colour", "colour_sum", "weight", "y_sq_sum"), **kw)
    th.join()
    for name in ("colour", "colour_sum", "weight", "y_sq_sum"):
        assert np.array_equal(bits(a2[name]), bits(a[name])), name
    for name in ("colour", "weight"):
        assert np.array_equal(bits(res["u"][name]), bits(u[name])), name
    assert a2["adaptive"].as_dict() == ast.as_dict()
