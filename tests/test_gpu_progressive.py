"""Progressive rendering (vrj_render_progressive) on the GPU.  Run on the B200 box with `-m gpu`.

The bar is the one of test_gpu_adaptive.py: bit equality.  A fresh call equals vrj_render_adaptive, any split of the
passes into calls ends in the same state, an adaptive state can be continued, and after the rule changes between calls
every pixel still holds exactly what vrj_render_tile gives it at its own count, with the counts a numpy replay of the
header's schedule predicts."""
import ctypes as C
import os
import subprocess
import threading

import numpy as np
import pytest

import vanrijn_b200 as V
from vanrijn_b200 import capi, host, scenes

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
KAHAN = (("colour_sum", 3), ("colour_bias", 3), ("weight", 1), ("weight_bias", 1))
STATE = KAHAN + (("y_sq_sum", 1),)
W, H = 37, 23                 # odd image
TILE = (5, 30, 3, 20)         # odd tile: 25 x 17 pixels
NPIX = (TILE[1] - TILE[0]) * (TILE[3] - TILE[2])
MIN, PASS, MAX = 4, 4, 32


def bits(a):
    """Float arrays as their bit patterns (so -0.0 != 0.0 and NaNs compare); other arrays as they are."""
    a = np.ascontiguousarray(a)
    return a.view(np.uint64) if a.dtype == np.float64 else a


def small_scene(whitted):
    spec = scenes.scene_main(subdivisions=2, obj=False)
    kw = dict(max_depth=6, seed=3)
    if whitted:
        light = spec.spectrum("grey", 1.0)
        kw.update(integrator=capi.INTEGRATOR_WHITTED, lights=[((1.0, 1.0, -1.0), light)])
    return V.build_scene(spec), kw


class Frame:
    """A frame's state (the five arrays) plus colour and srgb8, in host or device memory, continued call after call."""

    def __init__(self, memory, tile, height, width):
        self.memory, self.tile, self.height, self.width = memory, tile, height, width
        self.npix = (tile[1] - tile[0]) * (tile[3] - tile[2])
        self.L = capi.cuda()
        self.started = False
        self.arr, self.ptr = {}, {}
        for name, per, dtype in [(n, p, np.float64) for n, p in STATE] + [("colour", 3, np.float64), ("srgb8", 3, np.uint8)]:
            self.arr[name] = np.zeros(self.npix * per, dtype)
            if memory == capi.MEM_DEVICE:
                self.ptr[name] = self.L.vrj_alloc_device(0, max(8, self.arr[name].nbytes))
                assert self.ptr[name]
            else:
                self.ptr[name] = self.arr[name].ctypes.data

    def close(self):
        if self.memory == capi.MEM_DEVICE:
            for p in self.ptr.values():
                self.L.vrj_free_device(p)
        self.ptr = {}

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def accum_out(self, st):
        ao = capi.AccumOut(memory=self.memory, accumulate=1 if self.started else 0)
        for name in ("colour", "colour_sum", "colour_bias", "weight", "weight_bias", "srgb8"):
            setattr(ao, name, self.ptr[name])
        ao.stats = C.pointer(st)
        return ao

    def progressive(self, hs, mn, mx, ps, rel, abs_floor=0.0, max_passes=0, **kw):
        p, keep = hs.make_params(spp=0, **kw)
        pp = capi.ProgressiveParams(min_samples=mn, max_samples=mx, pass_samples=ps, max_passes=max_passes,
                                    rel_error=rel, abs_floor=abs_floor)
        st, pst = capi.Stats(), capi.ProgressiveStats()
        t = capi.Tile(*self.tile)
        capi.check(self.L.vrj_render_progressive(hs.device_scene(0), C.byref(t), self.height, self.width, C.byref(p), C.byref(pp),
                                                 C.byref(self.accum_out(st)), self.ptr["y_sq_sum"], C.byref(pst)))
        self.started = True
        return st, pst

    def adaptive(self, hs, mn, mx, ps, rel, abs_floor=0.0, **kw):
        """vrj_render_adaptive into this frame's arrays (the state a progressive call then continues)."""
        p, keep = hs.make_params(spp=0, **kw)
        ap = capi.AdaptiveParams(min_samples=mn, max_samples=mx, pass_samples=ps, rel_error=rel, abs_floor=abs_floor)
        st, ast = capi.Stats(), capi.AdaptiveStats()
        t = capi.Tile(*self.tile)
        ao = self.accum_out(st)
        ao.accumulate = 0
        capi.check(self.L.vrj_render_adaptive(hs.device_scene(0), C.byref(t), self.height, self.width, C.byref(p), C.byref(ap),
                                              C.byref(ao), self.ptr["y_sq_sum"], C.byref(ast)))
        self.started = True
        return st, ast

    def fetch(self):
        if self.memory == capi.MEM_DEVICE:
            for name, a in self.arr.items():
                capi.check(self.L.vrj_copy_to_host(0, a.ctypes.data, self.ptr[name], a.nbytes))
        return {k: v.copy() for k, v in self.arr.items()}


def assert_same_state(a, b, names=("colour",) + tuple(n for n, _ in STATE)):
    for name in names:
        assert np.array_equal(bits(a[name]), bits(b[name])), name


def spread_rel(hs, kw):
    """A rel_error whose adaptive render of the small tile ends with at least three counts, some below and some at MAX."""
    for rel in (0.5, 0.3, 0.2, 0.1, 0.05, 0.02):
        w = hs.render_adaptive(TILE, H, W, MIN, MAX, PASS, rel, want=("weight",), **kw)["weight"]
        counts = np.unique(w)
        if len(counts) >= 3 and counts.min() < MAX and counts.max() == MAX:
            return rel
    pytest.fail("no rel_error gave a spread of sample counts")


CASES = [pytest.param(whitted, precision, stride, offset, memory,
                      id="%s-%s-s%d-%s" % ("whitted" if whitted else "simple", "f64" if precision == capi.PRECISION_F64 else "f32fast",
                                           stride, "device" if memory == capi.MEM_DEVICE else "host"))
         for whitted in (False, True) for precision in (capi.PRECISION_F64, capi.PRECISION_F32_FAST)
         for stride, offset in ((1, 5), (2, 7)) for memory in (capi.MEM_HOST, capi.MEM_DEVICE)]


@pytest.mark.parametrize("whitted,precision,stride,offset,memory", CASES)
def test_fresh_call_equals_adaptive_and_one_pass_calls_reach_it(whitted, precision, stride, offset, memory):
    """(b) a fresh call with max_passes = 0 equals vrj_render_adaptive, every array and counter; (c) max_passes = 1 calls
    continuing one state end in that same state, and their passes and samples add up to the one-shot call's."""
    hs, kw = small_scene(whitted)
    kw.update(precision=precision, sample_stride=stride, sample_offset=offset)
    rel = spread_rel(hs, kw)
    with Frame(memory, TILE, H, W) as fa, Frame(memory, TILE, H, W) as fp, Frame(memory, TILE, H, W) as fl:
        sta, ast = fa.adaptive(hs, MIN, MAX, PASS, rel, **kw)
        stp, pst = fp.progressive(hs, MIN, MAX, PASS, rel, **kw)
        a, p = fa.fetch(), fp.fetch()
        assert_same_state(a, p, ("colour", "srgb8") + tuple(n for n, _ in STATE))
        assert (pst.passes, pst.samples, pst.pixels_converged, pst.pixels_at_max, pst.pixels_active) == \
            (ast.passes, ast.samples, ast.pixels_converged, ast.pixels_unconverged, 0)
        for name in ("primary_rays", "bounce_rays", "shadow_rays", "paths_missed", "paths_escaped", "paths_depth_limited"):
            assert getattr(stp, name) == getattr(sta, name), name
        passes = samples = 0
        for call in range(MAX):
            _, one = fl.progressive(hs, MIN, MAX, PASS, rel, max_passes=1, **kw)
            if one.passes == 0:
                break
            assert one.passes == 1
            passes, samples = passes + one.passes, samples + one.samples
        assert one.passes == 0 and one.samples == 0 and one.pixels_active == 0
        assert (passes, samples) == (pst.passes, pst.samples)
        assert (one.pixels_converged, one.pixels_at_max) == (pst.pixels_converged, pst.pixels_at_max)
        assert_same_state(fl.fetch(), p, ("colour", "srgb8") + tuple(n for n, _ in STATE))


@pytest.mark.parametrize("memory", [capi.MEM_HOST, capi.MEM_DEVICE], ids=["host", "device"])
def test_adaptive_state_continued_equals_the_longer_adaptive_render(memory):
    """(d) adaptive with max 16, then progressive with max 32, equals adaptive with max 32 (16 lies on the 4 + 4 j grid)."""
    hs, kw = small_scene(False)
    kw.update(sample_offset=3)
    rel = spread_rel(hs, kw)
    with Frame(memory, TILE, H, W) as f, Frame(memory, TILE, H, W) as ref:
        f.adaptive(hs, MIN, 16, PASS, rel, **kw)
        _, pst = f.progressive(hs, MIN, 32, PASS, rel, **kw)
        _, ast = ref.adaptive(hs, MIN, 32, PASS, rel, **kw)
        got, want = f.fetch(), ref.fetch()
        assert_same_state(got, want)
        assert (pst.pixels_converged, pst.pixels_at_max) == (ast.pixels_converged, ast.pixels_unconverged)
        assert pst.samples == int(want["weight"].sum()) - int(np.minimum(want["weight"], 16).sum())


def replay_schedule(Y, state, mn, mx, ps, rel, abs_floor=0.0, max_passes=0):
    """The header's schedule in numpy on the per-sample Y values Y[k, pixel], continuing `state` = (n, w, wb, s, b, q) (all
    modified in place; the Kahan updates of weight and colour_sum.y and q = q + y * y in sample order, binary64, numpy
    never fuses a multiply-add).  Returns the passes run and, per pass, the set of counts the active pixels took."""
    n, w, wb, s, b, q = state
    passes, counts = 0, []
    while not max_passes or passes < max_passes:
        with np.errstate(all="ignore"):
            m = s * (1.0 / w)
            v = (q - s * m) / (w - 1.0)
            v = np.where(v < 0.0, 0.0, v)
            t = rel * np.where(m > abs_floor, m, abs_floor)
            rule = v <= t * t * w
        c = np.where(n < mn, mn - n, np.where((n < mx) & ~rule, np.minimum(ps, mx - n), 0))
        if not c.any():
            break
        counts.append(set(np.unique(c[c > 0]).tolist()))
        for k in range(int(c.max())):
            sel = c > k
            y = Y[n[sel] + k, np.flatnonzero(sel)]
            wy = 1.0 - wb[sel]
            wt = w[sel] + wy
            wb[sel] = (wt - w[sel]) - wy
            w[sel] = wt
            yy = y * 1.0 - b[sel]
            ty = s[sel] + yy
            b[sel] = (ty - s[sel]) - yy
            s[sel] = ty
            q[sel] = q[sel] + y * y
        n += c
        passes += 1
    return passes, counts


def test_changing_the_rule_between_calls():
    """rel_error 0.3 -> 0.05, pass 4 -> 8, max 32 -> 40: the pixels of one pass take different counts.  Every pixel equals
    vrj_render_tile at its own count, its y_sq_sum equals vrj_render_adaptive(min = max = n)'s, and a numpy replay of the
    schedule predicts every count, every pass count and the final state's Y sums."""
    hs, kw = small_scene(False)
    kw.update(sample_offset=11, sample_stride=1)
    top = 40
    # a 1-spp render's colour_sum.y is that sample's Y exactly (0 + y)
    Y = np.stack([hs.render(TILE, H, W, spp=1, **dict(kw, sample_offset=11 + k))["colour_sum"].reshape(-1, 3)[:, 1] for k in range(top)])
    rs = (np.zeros(NPIX, np.int64),) + tuple(np.zeros(NPIX) for _ in range(5))
    with Frame(capi.MEM_HOST, TILE, H, W) as f:
        _, p1 = f.progressive(hs, MIN, 32, 4, 0.3, **kw)
        passes1, _ = replay_schedule(Y, rs, MIN, 32, 4, 0.3)
        _, p2 = f.progressive(hs, MIN, top, 8, 0.05, **kw)
        passes2, counts2 = replay_schedule(Y, rs, MIN, top, 8, 0.05)
        got = f.fetch()
    assert (p1.passes, p2.passes) == (passes1, passes2)
    assert any(len(c) > 1 for c in counts2), counts2  # a pass whose pixels took different counts
    n, w, wb, s, b, q = rs
    assert np.array_equal(n.astype(np.float64), got["weight"])
    assert np.array_equal(bits(s), bits(got["colour_sum"].reshape(-1, 3)[:, 1]))
    assert np.array_equal(bits(q), bits(got["y_sq_sum"]))
    assert p2.samples == int(got["weight"].sum()) - p1.samples
    assert p2.pixels_active == 0 and p2.pixels_converged + p2.pixels_at_max == NPIX
    for count in np.unique(got["weight"]):
        sel = got["weight"] == count
        u = hs.render(TILE, H, W, spp=int(count), **kw)
        for name, per in KAHAN + (("colour", 3),):
            assert np.array_equal(bits(got[name].reshape(-1, per)[sel]), bits(u[name].reshape(-1, per)[sel])), (name, count)
        a = hs.render_adaptive(TILE, H, W, int(count), int(count), 1, 0.1, want=("y_sq_sum",), **kw)
        assert np.array_equal(bits(got["y_sq_sum"][sel]), bits(a["y_sq_sum"][sel])), count


@pytest.mark.parametrize("memory", [capi.MEM_HOST, capi.MEM_DEVICE], ids=["host", "device"])
@pytest.mark.parametrize("whitted", [False, True], ids=["simple_random", "whitted_light"])
def test_uniform_progressive_frames(whitted, memory):
    """(e) calls with min = max = 4, 8, 12, 16 equal vrj_render_tile with spp 16 (the Kahan arrays, colour, srgb8) and
    vrj_render_adaptive with min = max = 16 (y_sq_sum)."""
    hs, kw = small_scene(whitted)
    kw.update(sample_offset=2)
    with Frame(memory, TILE, H, W) as f:
        for spp in (4, 8, 12, 16):
            _, pst = f.progressive(hs, spp, spp, 3, 0.01, **kw)
            assert pst.passes == 1 and pst.samples == 4 * NPIX and pst.pixels_active == 0
        got = f.fetch()
    u = hs.render(TILE, H, W, spp=16, want=("colour", "colour_sum", "colour_bias", "weight", "weight_bias", "srgb8"), **kw)
    a = hs.render_adaptive(TILE, H, W, 16, 16, 1, 0.01, want=("y_sq_sum",), **kw)
    assert_same_state(got, u, ("colour", "srgb8") + tuple(n for n, _ in KAHAN))
    assert np.array_equal(bits(got["y_sq_sum"]), bits(a["y_sq_sum"]))


def test_denoise_of_a_progressive_frame_equals_the_one_shot_frame():
    hs, kw = small_scene(False)
    rel = spread_rel(hs, kw)
    tw, th = TILE[1] - TILE[0], TILE[3] - TILE[2]
    one = hs.render_adaptive(TILE, H, W, MIN, MAX, PASS, rel, **kw)
    state = None
    for _ in range(MAX):
        state = hs.render_progressive(TILE, H, W, MIN, MAX, PASS, rel, max_passes=1, state=state, **kw)
        if state["progressive"].passes == 0:
            break
    aux = hs.render_aux(TILE, H, W, spp=MIN, **kw)
    d1 = host.denoise(one["colour_sum"], one["weight"], one["y_sq_sum"], aux, tw, th)
    d2 = host.denoise(state["colour_sum"], state["weight"], state["y_sq_sum"], aux, tw, th)
    for k in d1:
        if isinstance(d1[k], np.ndarray):
            assert np.array_equal(d1[k].view(np.uint8), d2[k].view(np.uint8)), k


def test_argument_errors_and_edge_cases():
    hs, kw = small_scene(False)
    L = capi.cuda()
    scene = hs.device_scene(0)
    t = capi.Tile(*TILE)
    base = hs.render_progressive(TILE, H, W, MIN, 8, 2, 0.1, **kw)

    def call(pp_kw=None, spp=0, weight=None, null=None, **ao_kw):
        p, keep = hs.make_params(spp=spp, **kw)
        pp = capi.ProgressiveParams(**dict(dict(min_samples=MIN, max_samples=8, pass_samples=2, rel_error=0.1), **(pp_kw or {})))
        arrs = {n: base[n].copy() for n, _ in STATE}
        if weight is not None:
            arrs["weight"][7] = weight
        ao = capi.AccumOut(memory=capi.MEM_HOST, accumulate=1, **ao_kw)
        for n, _ in KAHAN:
            setattr(ao, n, None if n == null else arrs[n].ctypes.data)
        ysq = None if null == "y_sq_sum" else arrs["y_sq_sum"].ctypes.data
        r = L.vrj_render_progressive(scene, C.byref(t), H, W, C.byref(p), C.byref(pp), C.byref(ao), ysq, None)
        return r, arrs

    assert call()[0] == capi.OK
    for bad in (float("nan"), -1.0, 2.5, float("inf"), 2.0 ** 32):
        r, arrs = call(weight=bad)
        assert r == 1 and b"weight" in L.vrj_last_error(), bad  # VRJ_ERR_INVALID_ARGUMENT
        assert_same_state(arrs, base, ("colour_sum", "colour_bias", "weight_bias", "y_sq_sum"))  # the state is left as it was
    for name, _ in STATE:
        assert call(null=name)[0] == 1, name
    for pp_kw, spp in [(dict(min_samples=1), 0), (dict(min_samples=8, max_samples=4), 0), (dict(pass_samples=0), 0),
                       (dict(rel_error=0.0), 0), (dict(rel_error=float("nan")), 0), (dict(abs_floor=-1.0), 0), ({}, 4)]:
        assert call(pp_kw, spp)[0] == 1, (pp_kw, spp)
    photons = np.zeros(NPIX * 64)
    assert call(photons=photons.ctypes.data)[0] == 3  # VRJ_ERR_UNSUPPORTED
    assert b"photons" in L.vrj_last_error()
    e = hs.render_progressive((4, 4, 0, H), H, W, MIN, 8, 2, 0.1, **kw)
    assert e["progressive"].passes == 0 and e["progressive"].samples == 0 and e["stats"].primary_rays == 0
    # nothing active: the state comes back bit for bit, with no pass and no ray
    done = hs.render_progressive(TILE, H, W, MIN, 8, 2, 0.1, state=base, **kw)
    assert done["progressive"].passes == 0 and done["progressive"].pixels_active == 0 and done["stats"].primary_rays == 0
    assert_same_state(done, base)


def test_c5_1080p_device_preview_loop_concurrent_with_a_uniform_render():
    """C5 at 1920x1080 in device memory: a max_passes = 1 preview loop, with a vrj_render_tile running from another thread,
    reaches the one-shot state; the uniform render gives its single-call result."""
    hs = V.build_scene(scenes.scene_main(variant="mixed"))
    W5, H5 = 1920, 1080
    full = (0, W5, 0, H5)
    kw = dict(max_depth=128, seed=5)
    args = (4, 16, 4, 0.25)
    u = hs.render(full, H5, W5, spp=8, want=("colour", "weight"), **dict(kw, sample_offset=1000))
    res = {}

    def run_uniform():
        res["u"] = hs.render(full, H5, W5, spp=8, want=("colour", "weight"), **dict(kw, sample_offset=1000))

    with Frame(capi.MEM_DEVICE, full, H5, W5) as one, Frame(capi.MEM_DEVICE, full, H5, W5) as loop:
        _, pst = one.progressive(hs, *args, **kw)
        th = threading.Thread(target=run_uniform)
        th.start()
        passes = 0
        for _ in range(16):
            _, p = loop.progressive(hs, *args, max_passes=1, **kw)
            if p.passes == 0:
                break
            passes += 1
        th.join()
        assert passes == pst.passes and pst.pixels_active == 0
        assert_same_state(loop.fetch(), one.fetch(), ("colour", "srgb8") + tuple(n for n, _ in STATE))
    for name in ("colour", "weight"):
        assert np.array_equal(bits(res["u"][name]), bits(u[name])), name


def test_vanrijn_cli_resident_rel_error_denoise(tmp_path):
    exe = os.path.join(ROOT, "build", "vanrijn")
    out = tmp_path / "preview.png"
    r = subprocess.run([exe, "--size", "96", "64", "--resident", "--rel-error", "0.1", "--min-spp", "4", "--max-spp", "16",
                        "--spp", "4", "--passes", "8", "--depth", "16", "--denoise", "--out", str(out)],
                       capture_output=True, text=True, timeout=600, env=dict(os.environ, VANRIJN_BUNNY_OBJ=""))
    assert r.returncode == 0, r.stdout + r.stderr
    assert out.exists() and out.read_bytes()[:8] == b"\x89PNG\r\n\x1a\n"
