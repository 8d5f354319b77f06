"""Per-pixel sample counts (vrj_render_counts) and the planner (vrj_plan_counts) on the GPU.  Run on the B200 box with `-m gpu`.

The bar is bit equality: a pixel that ends with N samples holds exactly what vrj_render_tile with spp = N gives it, and the
y_sq_sum of vrj_render_adaptive with min = max = N; the planner's counts and counters equal a numpy replay of the rule the
header states."""
import ctypes as C
import threading

import numpy as np
import pytest

import vanrijn_b200 as V
from vanrijn_b200 import capi, host, scenes

pytestmark = pytest.mark.gpu

KAHAN = (("colour_sum", 3), ("colour_bias", 3), ("weight", 1), ("weight_bias", 1))
STATE = KAHAN + (("y_sq_sum", 1),)
W, H = 37, 23                 # odd image
TILE = (5, 30, 3, 20)         # odd tile: 25 x 17 pixels
NPIX = (TILE[1] - TILE[0]) * (TILE[3] - TILE[2])


def bits(a):
    a = np.ascontiguousarray(a)
    return a.view(np.uint64) if a.dtype == np.float64 else a


def small_scene(whitted):
    spec = scenes.scene_main(subdivisions=2, obj=False)
    kw = dict(max_depth=6, seed=3)
    if whitted:
        light = spec.spectrum("grey", 1.0)
        kw.update(integrator=capi.INTEGRATOR_WHITTED, lights=[((1.0, 1.0, -1.0), light)])
    return V.build_scene(spec), kw


def random_map(seed, values=(0, 1, 2, 3, 5, 8), npix=NPIX):
    rng = np.random.default_rng(seed)
    c = rng.choice(np.array(values, np.uint32), npix)
    c[:len(values)] = values  # every value occurs
    return c


def assert_pixels_equal_tile(hs, got, total, kw, tile=TILE, height=H, width=W):
    """every pixel equals vrj_render_tile at its own count `total` (Kahan arrays and colour), and its y_sq_sum the one
    vrj_render_adaptive keeps at that count (y * y for a single sample); pixels with no sample hold zeros and NaN colour"""
    assert np.array_equal(got["weight"], total.astype(np.float64))
    for count in np.unique(total):
        sel = total == count
        if count == 0:
            for name, per in STATE:
                assert not got[name].reshape(-1, per)[sel].any(), name
            assert np.isnan(got["colour"].reshape(-1, 3)[sel]).all()
            continue
        u = hs.render(tile, height, width, spp=int(count), **kw)
        for name, per in KAHAN + (("colour", 3),):
            assert np.array_equal(bits(got[name].reshape(-1, per)[sel]), bits(u[name].reshape(-1, per)[sel])), (name, count)
        if count >= 2:
            a = hs.render_adaptive(tile, height, width, int(count), int(count), 1, 0.1, want=("y_sq_sum",), **kw)
            want = a["y_sq_sum"][sel]
        else:
            y = u["colour_sum"].reshape(-1, 3)[sel][:, 1]
            want = y * y
        assert np.array_equal(bits(got["y_sq_sum"][sel]), bits(want)), count


FRESH = [pytest.param(whitted, precision, stride, offset, filt, count,
                      id="%s-%s-s%d-o%d-f%d%s" % ("whitted" if whitted else "simple", "f64" if precision == capi.PRECISION_F64 else "f32fast",
                                                  stride, offset, filt, "-count" if count else ""))
         for whitted, precision, stride, offset, filt, count in [
             (False, capi.PRECISION_F64, 1, 0, capi.FILTER_F32, False),
             (False, capi.PRECISION_F64, 2, 7, capi.FILTER_F64, True),
             (False, capi.PRECISION_F64, 3, 2, capi.FILTER_Q16, False),
             (False, capi.PRECISION_F32_FAST, 1, 4, capi.FILTER_F32, False),
             (True, capi.PRECISION_F64, 1, 5, capi.FILTER_F32X4, False),
             (True, capi.PRECISION_F64, 2, 1, capi.FILTER_F32, True),
             (True, capi.PRECISION_F32_FAST, 2, 3, capi.FILTER_F32, False)]]


@pytest.mark.parametrize("whitted,precision,stride,offset,filt,count", FRESH)
def test_fresh_state_equals_tile_render_at_each_count(whitted, precision, stride, offset, filt, count):
    hs, kw = small_scene(whitted)
    kw.update(precision=precision, sample_stride=stride, sample_offset=offset, bvh_filter=filt, count_traversal=count)
    c = random_map(1 + stride + offset)
    got = hs.render_counts(TILE, H, W, c, **kw)
    cs = got["counts"]
    assert (cs.samples, cs.pixels, cs.batches) == (int(c.sum()), int((c > 0).sum()), 1)
    assert got["stats"].primary_rays == int(c.sum())
    if count:
        assert got["stats"].node_visits > 0
    assert_pixels_equal_tile(hs, got, c, kw)


def to_device(a):
    """a host array's bytes in device memory (a torch tensor: the library has no upload call of its own)"""
    import torch
    t = torch.from_numpy(np.ascontiguousarray(a).view(np.uint8).copy()).to("cuda:0")
    torch.cuda.synchronize()  # the library reads it on a stream of its own
    return t


class Frame:
    """A state, its colour and srgb8, in host or device memory; the count map goes in the same kind of memory."""

    def __init__(self, memory, npix):
        self.memory, self.npix = memory, npix
        self.L = capi.cuda()
        self.arr, self.ptr = {}, {}
        for name, per, dtype in [(n, p, np.float64) for n, p in STATE] + [("colour", 3, np.float64), ("srgb8", 3, np.uint8)]:
            self.arr[name] = np.zeros(npix * per, dtype)
            if memory == capi.MEM_DEVICE:
                self.ptr[name] = self.L.vrj_alloc_device(0, max(8, self.arr[name].nbytes))
                assert self.ptr[name]
            else:
                self.ptr[name] = self.arr[name].ctypes.data

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        if self.memory == capi.MEM_DEVICE:
            for p in self.ptr.values():
                self.L.vrj_free_device(p)

    def accum_out(self, st, accumulate):
        ao = capi.AccumOut(memory=self.memory, accumulate=1 if accumulate else 0)
        for name in ("colour", "colour_sum", "colour_bias", "weight", "weight_bias", "srgb8"):
            setattr(ao, name, self.ptr[name])
        ao.stats = C.pointer(st)
        return ao

    def counts(self, hs, tile, height, width, cmap, accumulate, **kw):
        cmap = np.ascontiguousarray(cmap, np.uint32)
        dev = to_device(cmap) if self.memory == capi.MEM_DEVICE else None
        p, keep = hs.make_params(spp=0, **kw)
        st, cst = capi.Stats(), capi.CountsStats()
        t = capi.Tile(*tile)
        r = self.L.vrj_render_counts(hs.device_scene(0), C.byref(t), height, width, C.byref(p),
                                     dev.data_ptr() if dev is not None else cmap.ctypes.data, C.byref(self.accum_out(st, accumulate)),
                                     self.ptr["y_sq_sum"], C.byref(cst))
        return r, st, cst

    def progressive(self, hs, tile, height, width, mn, mx, ps, rel, **kw):
        p, keep = hs.make_params(spp=0, **kw)
        pp = capi.ProgressiveParams(min_samples=mn, max_samples=mx, pass_samples=ps, rel_error=rel)
        st, pst = capi.Stats(), capi.ProgressiveStats()
        t = capi.Tile(*tile)
        capi.check(self.L.vrj_render_progressive(hs.device_scene(0), C.byref(t), height, width, C.byref(p), C.byref(pp),
                                                 C.byref(self.accum_out(st, False)), self.ptr["y_sq_sum"], C.byref(pst)))
        return pst

    def fetch(self):
        if self.memory == capi.MEM_DEVICE:
            for name, a in self.arr.items():
                capi.check(self.L.vrj_copy_to_host(0, a.ctypes.data, self.ptr[name], a.nbytes))
        return {k: v.copy() for k, v in self.arr.items()}


@pytest.mark.parametrize("memory", [capi.MEM_HOST, capi.MEM_DEVICE], ids=["host", "device"])
def test_continued_state_equals_tile_render_at_n_plus_c(memory):
    """A map added to a vrj_render_progressive state with mixed counts: every pixel equals the tile render at n + c, and
    colour and srgb8 are formed for every pixel."""
    hs, kw = small_scene(False)
    kw.update(sample_offset=9)
    c = random_map(7, values=(0, 1, 4, 7))
    with Frame(memory, NPIX) as f:
        pst = f.progressive(hs, TILE, H, W, 4, 24, 4, 0.2, **kw)
        n = f.fetch()["weight"].astype(np.int64)
        assert len(np.unique(n)) >= 2 and pst.samples == n.sum()
        r, st, cst = f.counts(hs, TILE, H, W, c, True, **kw)
        capi.check(r)
        got = f.fetch()
    assert cst.samples == int(c.sum()) and cst.pixels == int((c > 0).sum()) and cst.batches == 1
    total = n + c
    assert_pixels_equal_tile(hs, got, total, kw)
    assert np.array_equal(got["srgb8"], host.tone_map(got["colour"]).reshape(-1))


@pytest.mark.parametrize("memory", [capi.MEM_HOST, capi.MEM_DEVICE], ids=["host", "device"])
@pytest.mark.parametrize("whitted", [False, True], ids=["simple_random", "whitted_light"])
def test_uniform_map_equals_tile_render(whitted, memory):
    """c everywhere on a fresh state: every array, srgb8 and the ray counters of vrj_render_tile at spp = c"""
    hs, kw = small_scene(whitted)
    kw.update(sample_offset=4)
    with Frame(memory, NPIX) as f:
        r, st, cst = f.counts(hs, TILE, H, W, np.full(NPIX, 6, np.uint32), False, **kw)
        capi.check(r)
        got = f.fetch()
    u = hs.render(TILE, H, W, spp=6, want=("colour", "colour_sum", "colour_bias", "weight", "weight_bias", "srgb8"), **kw)
    for name in ("colour", "colour_sum", "colour_bias", "weight", "weight_bias", "srgb8"):
        assert np.array_equal(bits(got[name]), bits(u[name])), name
    for name in ("primary_rays", "bounce_rays", "shadow_rays", "paths_missed", "paths_escaped", "paths_depth_limited"):
        assert getattr(st, name) == getattr(u["stats"], name), name


def test_split_batches(monkeypatch):
    """With a path budget of 2^16 the map's 76k samples take two batches; a pixel's run straddles the boundary and every
    pixel still equals the tile render at its count."""
    monkeypatch.setenv("VRJ_PATH_BUDGET_LOG2", "16")
    hs, kw = small_scene(False)
    kw.update(sample_offset=1)
    c = random_map(3, values=(150, 170, 190, 210))
    off = np.concatenate([[0], np.cumsum(c.astype(np.int64))])
    assert off[-1] > 1 << 16 and ((off[:-1] < 1 << 16) & (off[1:] > 1 << 16)).any()
    got = hs.render_counts(TILE, H, W, c, **kw)
    assert got["counts"].batches == 2 and got["counts"].samples == off[-1]
    assert_pixels_equal_tile(hs, got, c.astype(np.int64), kw)


def replay_plan(n, s, q, mn, mx, ps, rel, floor):
    """the header's rule of vrj_plan_counts in numpy (binary64, same order; numpy never fuses a multiply-add)"""
    n = np.asarray(n, np.float64)
    with np.errstate(all="ignore"):
        m = s * (1.0 / n)
        v = (q - s * m) / (n - 1.0)
        v = np.where(v < 0.0, 0.0, v)
        t = rel * np.where(m > floor, m, floor)
        conv = v <= t * t * n
        need = v / (t * t)
        target = np.where(need < mx, np.ceil(need), float(mx))
        extra = target - n
        c = np.minimum(mx - n, np.where(extra > ps, extra, float(ps)))
    low = n < mn
    c = np.where(low, mn - n, np.where((n >= mx) | conv, 0.0, c)).astype(np.uint32)
    stats = (int(c.astype(np.int64).sum()), int((c > 0).sum()), int((~low & conv).sum()), int((~low & ~conv & (n >= mx)).sum()))
    return c, stats


@pytest.mark.parametrize("memory", [capi.MEM_HOST, capi.MEM_DEVICE], ids=["host", "device"])
def test_plan_equals_numpy_replay(memory):
    hs, kw = small_scene(False)
    mn, mx, ps, rel, floor = 4, 64, 4, 0.1, 0.01
    real = hs.render_progressive(TILE, H, W, 4, 16, 4, 0.3, **kw)  # a real state with mixed counts
    rng = np.random.default_rng(5)
    k = 600
    n = rng.choice(np.array([0, 1, mn - 1, mn, mn + 1, 17, mx - 1, mx, mx + 3], np.float64), k)
    mean = rng.uniform(0.0, 2.0, k)
    s = mean * n
    q = s * mean * rng.uniform(1.0, 3.0, k)
    q[::7] = s[::7] * mean[::7]        # zero variance (up to rounding)
    s[5::11] = np.nan                  # NaN estimates
    s[3::13], q[3::13] = 0.0, 0.0      # a black pixel: t from abs_floor
    weight = np.concatenate([real["weight"], n])
    sum3 = np.concatenate([real["colour_sum"].reshape(-1, 3), np.stack([s * 0.5, s, s * 2.0], 1)]).reshape(-1)
    ysq = np.concatenate([real["y_sq_sum"], q])
    want, want_stats = replay_plan(weight, sum3.reshape(-1, 3)[:, 1], ysq, mn, mx, ps, rel, floor)
    assert want_stats[1] and want_stats[2] and want_stats[3]
    rule = capi.AdaptiveParams(min_samples=mn, max_samples=mx, pass_samples=ps, rel_error=rel, abs_floor=floor)
    ins = [np.ascontiguousarray(a, np.float64) for a in (weight, sum3, ysq)]
    counts = np.full(weight.size, 77, np.uint32)
    L = capi.cuda()

    def plan(ins, counts):
        ps_ = capi.PlanStats()
        if memory == capi.MEM_HOST:
            r = L.vrj_plan_counts(0, memory, weight.size, *[a.ctypes.data for a in ins], C.byref(rule), counts.ctypes.data, C.byref(ps_))
            return r, counts, ps_
        dev = [to_device(a) for a in ins] + [to_device(counts)]
        r = L.vrj_plan_counts(0, memory, weight.size, *[d.data_ptr() for d in dev[:3]], C.byref(rule), dev[3].data_ptr(), C.byref(ps_))
        return r, dev[3].cpu().numpy().view(np.uint32).copy(), ps_

    r, got, pst = plan(ins, counts.copy())
    capi.check(r)
    assert np.array_equal(got, want)
    assert (pst.samples, pst.pixels_planned, pst.pixels_converged, pst.pixels_at_max) == want_stats
    assert pst.pixels_planned + pst.pixels_converged + pst.pixels_at_max == weight.size
    for bad in (float("nan"), -1.0, 2.5, float("inf"), 2.0 ** 32):
        w2 = ins[0].copy()
        w2[11] = bad
        r, got, _ = plan([w2, ins[1], ins[2]], counts.copy())
        assert r == 1 and b"weight" in L.vrj_last_error(), bad
        assert (got == 77).all()  # the counts are left as they were
    for rule_kw in (dict(min_samples=1), dict(max_samples=2), dict(pass_samples=0), dict(rel_error=0.0), dict(abs_floor=-1.0)):
        bad_rule = capi.AdaptiveParams(**dict(dict(min_samples=mn, max_samples=mx, pass_samples=ps, rel_error=rel), **rule_kw))
        assert L.vrj_plan_counts(0, capi.MEM_HOST, 1, ins[0].ctypes.data, ins[1].ctypes.data, ins[2].ctypes.data, C.byref(bad_rule),
                                 counts.ctypes.data, None) == 1, rule_kw
    assert L.vrj_plan_counts(0, capi.MEM_HOST, 0, None, None, None, C.byref(rule), None, None) == capi.OK


def test_plan_render_loop_ends_converged_or_at_max():
    hs, kw = small_scene(False)
    mn, mx, ps, rel = 4, 48, 4, 0.1
    res = hs.render_planned(TILE, H, W, mn, mx, ps, rel, **kw)
    assert res["rounds"] >= 2 and res["plan"].samples == 0
    assert res["plan"].pixels_converged + res["plan"].pixels_at_max == NPIX
    _, (samples, planned, conv, at_max) = replay_plan(res["weight"], res["colour_sum"].reshape(-1, 3)[:, 1], res["y_sq_sum"], mn, mx, ps, rel, 0.0)
    assert samples == 0 and planned == 0 and conv + at_max == NPIX
    assert res["samples"] == int(res["weight"].sum())
    # the rounds split differently (one round per call) end in the same bits
    state = None
    for _ in range(res["rounds"] + 1):
        state = hs.render_planned(TILE, H, W, mn, mx, ps, rel, rounds=1, state=state, **kw)
    for name, _ in STATE:
        assert np.array_equal(bits(state[name]), bits(res[name])), name
    assert_pixels_equal_tile(hs, res, res["weight"].astype(np.int64), kw)


def test_argument_errors_and_edge_cases():
    hs, kw = small_scene(False)
    L = capi.cuda()
    scene = hs.device_scene(0)
    t = capi.Tile(*TILE)
    base = hs.render_progressive(TILE, H, W, 4, 8, 2, 0.1, **kw)
    cmap = random_map(2)

    def call(c=cmap, spp=0, weight=None, null=None, accumulate=1, **ao_kw):
        p, keep = hs.make_params(spp=spp, **kw)
        arrs = {n: base[n].copy() for n, _ in STATE}
        if weight is not None:
            arrs["weight"][7] = weight
        ao = capi.AccumOut(memory=capi.MEM_HOST, accumulate=accumulate, **ao_kw)
        for n, _ in KAHAN:
            setattr(ao, n, None if n == null else arrs[n].ctypes.data)
        st, cst = capi.Stats(), capi.CountsStats()
        ao.stats = C.pointer(st)
        cc = None if c is None else np.ascontiguousarray(c, np.uint32)
        r = L.vrj_render_counts(scene, C.byref(t), H, W, C.byref(p), None if cc is None else cc.ctypes.data, C.byref(ao),
                                arrs["y_sq_sum"].ctypes.data, C.byref(cst))
        return r, arrs, st, cst

    assert call()[0] == capi.OK
    assert call(spp=4)[0] == 1
    assert call(c=None)[0] == 1
    for name, _ in KAHAN:
        assert call(null=name)[0] == 1, name
    photons = np.zeros(NPIX * 64)
    assert call(photons=photons.ctypes.data)[0] == 3 and b"photons" in L.vrj_last_error()
    for bad in (float("nan"), -1.0, 2.5, float("inf"), 2.0 ** 32):
        r, arrs, st, _ = call(weight=bad)
        assert r == 1 and b"weight" in L.vrj_last_error(), bad
        assert_same(arrs, base, ("colour_sum", "colour_bias", "weight_bias", "y_sq_sum"))
    # n + c >= 2^32: refused, state unchanged
    r, arrs, _, _ = call(weight=2.0 ** 32 - 3, c=np.where(np.arange(NPIX) == 7, 3, 0))
    assert r == 1 and b"2^32" in L.vrj_last_error()
    assert_same(arrs, base, ("colour_sum", "colour_bias", "weight_bias", "y_sq_sum"))
    # more than 2^32 - 1 samples in the call: unsupported, state unchanged
    r, arrs, st, _ = call(c=np.full(NPIX, 1 << 24, np.uint32))
    assert r == 3 and st.primary_rays == 0
    assert_same(arrs, base)
    # an all-zero map: the state comes back bit for bit, no ray, no batch
    r, arrs, st, cst = call(c=np.zeros(NPIX, np.uint32))
    assert r == capi.OK and st.primary_rays == 0 and (cst.samples, cst.pixels, cst.batches) == (0, 0, 0)
    assert_same(arrs, base)
    # an empty tile: no work
    e = hs.render_counts((4, 4, 0, H), H, W, np.zeros(0, np.uint32), **kw)
    assert e["counts"].samples == 0 and e["stats"].primary_rays == 0


def assert_same(a, b, names=tuple(n for n, _ in STATE)):
    for name in names:
        assert np.array_equal(bits(a[name]), bits(b[name])), name


def test_c5_1080p_alone_and_concurrent_with_a_tile_render():
    """C5 at 1920x1080: a count map in device memory, alone and with a vrj_render_tile running from another thread; both
    calls give their solo results bit for bit."""
    hs = V.build_scene(scenes.scene_main(variant="mixed"))
    W5, H5 = 1920, 1080
    full = (0, W5, 0, H5)
    kw = dict(max_depth=128, seed=5)
    c = random_map(11, values=(0, 1, 2, 4), npix=W5 * H5)
    u = hs.render(full, H5, W5, spp=4, want=("colour", "weight"), **dict(kw, sample_offset=1000))
    res = {}

    def run_uniform():
        res["u"] = hs.render(full, H5, W5, spp=4, want=("colour", "weight"), **dict(kw, sample_offset=1000))

    with Frame(capi.MEM_DEVICE, W5 * H5) as solo, Frame(capi.MEM_DEVICE, W5 * H5) as conc:
        capi.check(solo.counts(hs, full, H5, W5, c, False, **kw)[0])
        th = threading.Thread(target=run_uniform)
        th.start()
        capi.check(conc.counts(hs, full, H5, W5, c, False, **kw)[0])
        th.join()
        a, b = solo.fetch(), conc.fetch()
    assert_same(a, b, ("colour", "srgb8") + tuple(n for n, _ in STATE))
    assert np.array_equal(a["weight"], c.astype(np.float64))
    for name in ("colour", "weight"):
        assert np.array_equal(bits(res["u"][name]), bits(u[name])), name
