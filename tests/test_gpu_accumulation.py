"""Every resolve path's accumulators against a replay of update_pixel, bit for bit.  Run on the B200 box with `-m gpu`.

A render call ends in a resolve kernel that applies the batch's samples, in sample order, to the Kahan state of
AccumulationBuffer::update_pixel (colour_sum, colour_bias, weight, weight_bias; y_sq_sum too for the pass-based calls).
Here that state is recomputed on the host, independently of the kernels:
  * a fresh 1-spp call resolves one sample into a zero state, so its colour_sum is, bit for bit, the XYZ that sample adds
    in any call (samples are pure functions of seed, pixel and sample index);
  * test_accumulation_cpu.replay applies those values in binary64 in the kernels' order (it equals the oracle's
    PixelAccum::update bit for bit there).
The compensation terms, y_sq_sum and the colour are then compared by their bits: a resolve that dropped or mis-signed a
compensation, loaded a stale bias or copied a piece of the arrays from the wrong place fails here."""
import ctypes as C
import threading

import numpy as np
import pytest

import oraclelib as O
import vanrijn_b200 as V
from test_accumulation_cpu import OUTPUTS, STATE, cmf_xyz, replay
from test_gpu_parity import photons_close
from vanrijn_b200 import capi, scenes

pytestmark = pytest.mark.gpu

KAHAN = STATE[:4]
FIVE = OUTPUTS[:5]           # what vrj_render_tile returns
W, H = 37, 23                # odd image
TILE = (5, 30, 3, 20)        # odd tile: 25 x 17 pixels
NPIX = (TILE[1] - TILE[0]) * (TILE[3] - TILE[2])
U64 = 1 << 64
ERR_UNSUPPORTED = 3

# Per-sample XYZ against the oracle's colour matching functions on the device's own photons: the two differ only in the
# seven exponentials (CUDA's exp against glibc's).  Measured on an NVIDIA B200 (1000 W power limit): at most 4.0e-16 of the
# sample's largest component, on both scenes.
CMF_RTOL = 2e-15


def bits(a):
    a = np.ascontiguousarray(a)
    return a.view(np.uint64) if a.dtype == np.float64 else a


def assert_bits(got, want, names):
    for name in names:
        g, w = bits(got[name]), bits(want[name])
        bad = np.flatnonzero(g != w)
        assert bad.size == 0, (name, bad.size, bad[:4], got[name].reshape(-1)[bad[:4]], want[name].reshape(-1)[bad[:4]])


_SCENES = {}


def scene(variant="lambertian", subdivisions=2):
    """scene_main at `subdivisions` (6: the bench's C3 / C5), one per process, with a grey spectrum for a directional light
    (hs.light) added to it"""
    key = (variant, subdivisions)
    if key not in _SCENES:
        _SCENES[key] = build(variant, subdivisions)
    return _SCENES[key]


def build(variant="lambertian", subdivisions=2):
    spec = scenes.scene_main(subdivisions=subdivisions, obj=subdivisions >= 6, variant=variant)
    light = spec.spectrum("grey", 1.0)
    hs = V.build_scene(spec)
    hs.light = light
    return hs


def whitted_kw(hs):
    return dict(integrator=capi.INTEGRATOR_WHITTED, lights=[((1.0, 1.0, -1.0), hs.light)])


_SAMPLES = {}


def samples(hs, tile, height, width, indices, **kw):
    """The exact XYZ of sample `i` of every tile pixel, for each i of `indices` (taken mod 2^64): (len(indices), npix, 3).
    Each is the colour_sum of a fresh 1-spp call at sample_offset = i, whose weight must be 1 and whose compensation terms
    must be 0.  `kw`: the render parameters (sample_offset, sample_stride and spp excepted)."""
    npix = (tile[1] - tile[0]) * (tile[3] - tile[2])
    out = np.empty((len(indices), npix, 3))
    for j, i in enumerate(indices):
        key = (id(hs), tuple(tile), height, width, i % U64, repr(sorted(kw.items())))
        if key not in _SAMPLES:
            r = hs.render(tile, height, width, want=("colour_sum", "colour_bias", "weight", "weight_bias"), spp=1,
                          sample_offset=i % U64, **kw)
            assert (r["weight"] == 1.0).all() and not r["colour_bias"].any() and not r["weight_bias"].any(), i
            _SAMPLES[key] = (hs, r["colour_sum"].reshape(npix, 3))  # hs kept alive: its id stays its own
        out[j] = _SAMPLES[key][1]
    return out


def sample_indices(offset, stride, ks):
    return [(offset + k * stride) % U64 for k in ks]


def replay_tile(hs, tile, height, width, spp, sample_offset=0, sample_stride=1, state0=None, sampler=None, **kw):
    """what vrj_render_tile at spp leaves: the replay of samples offset + k * stride, k < spp, on state0 (None: zeros)"""
    c = samples(sampler or hs, tile, height, width, sample_indices(sample_offset, sample_stride, range(spp)), **kw)
    return replay(state0 or {}, c)


def replay_passes(hs, tile, height, width, n0, n1, sample_offset=0, sample_stride=1, state0=None, sampler=None, **kw):
    """a pass-based call's state: pixel p takes samples n0[p] .. n1[p] - 1 of its own, in order, on state0"""
    n0, n1 = np.asarray(n0, np.int64), np.asarray(n1, np.int64)
    assert (n1 >= n0).all()
    lo, hi = int(n0.min()), int(n1.max())
    c = samples(sampler or hs, tile, height, width, sample_indices(sample_offset, sample_stride, range(lo, hi)), **kw)
    ks = np.arange(lo, hi)[:, None]
    return replay(state0 or {}, c, active=(ks >= n0[None, :]) & (ks < n1[None, :]))


def random_state(seed, npix, integral):
    """a state with sums of a few scales, non-zero compensation terms and y_sq_sum above the mean's square; integral: the
    weights are sample counts 2..9 (what the pass-based calls accept), else any positive value"""
    rng = np.random.default_rng(seed)
    n = rng.integers(2, 10, npix).astype(np.float64) if integral else rng.uniform(0.25, 40.0, npix)
    mean = rng.uniform(0.05, 1.0, (npix, 3)) * 10.0 ** rng.uniform(-2, 1, (npix, 1))
    s = mean * n[:, None]
    b = rng.uniform(-1.0, 1.0, (npix, 3)) * np.spacing(s)
    wb = rng.uniform(-1.0, 1.0, npix) * np.spacing(n) * (0.0 if integral else 1.0)
    q = s[:, 1] * mean[:, 1] * rng.uniform(1.0, 1.5, npix)
    return {"colour_sum": s.reshape(-1), "colour_bias": b.reshape(-1), "weight": n, "weight_bias": wb, "y_sq_sum": q}


def render_into(hs, tile, height, width, ptrs, memory, accumulate, **kw):
    """vrj_render_tile into caller-owned arrays (`ptrs`: name -> address, absent = NULL); returns the stats"""
    p, keep = hs.make_params(**kw)
    ao = capi.AccumOut(memory=memory, accumulate=1 if accumulate else 0)
    for name, _ in FIVE:
        setattr(ao, name, ptrs.get(name))
    st = capi.Stats()
    ao.stats = C.pointer(st)
    t = capi.Tile(*tile)
    capi.check(capi.cuda().vrj_render_tile(hs.device_scene(0), C.byref(t), height, width, C.byref(p), C.byref(ao)))
    return st


# ------------------------------------------------------------------------------------------------ the samples themselves
@pytest.mark.parametrize("variant", ["lambertian", "mixed"])
def test_extracted_samples_equal_the_oracle_xyz_of_the_device_photons(variant):
    """c (the colour_sum of a 1-spp call) against orc_cmf_xyz(wavelength) * intensity of the same sample's photon: exactly
    zero where the intensity is +0, else within CMF_RTOL of the sample's largest component.  The 8-spp call's own arrays
    equal the replay of those c."""
    hs = scene(variant)
    kw = dict(max_depth=8, seed=7)
    spp = 8
    g = hs.render(TILE, H, W, spp=spp, want_photons=True, **kw)
    ph = g["photons"]
    c = samples(hs, TILE, H, W, range(spp), **kw)
    zero = bits(ph[..., 1]) == 0
    assert zero.any() and (~zero).sum() > spp * NPIX // 4
    assert not c[zero].any()
    ref = cmf_xyz(ph[..., 0][~zero]) * ph[..., 1][~zero][:, None]
    scale = np.abs(ref).max(axis=1)
    err = (np.abs(c[~zero] - ref).max(axis=1) / np.where(scale > 0, scale, 1.0))
    print("%s: worst per-sample relative difference from the oracle's XYZ %.3e over %d samples" % (variant, err.max(), err.size))
    assert err.max() <= CMF_RTOL, err.max()
    assert_bits(g, replay({}, c), [n for n, _ in FIVE])


# ------------------------------------------------------------------------------------------------ k_resolve (and k_resolve_multi)
RESOLVE = [pytest.param(whitted, precision, stride, offset, id="%s-%s-s%d-o%d" % ("whitted" if whitted else "simple",
                                                                                 "f64" if precision == capi.PRECISION_F64 else "f32fast", stride, offset))
           for whitted, precision, stride, offset in [(False, capi.PRECISION_F64, 1, 0), (False, capi.PRECISION_F64, 3, 5),
                                                      (False, capi.PRECISION_F32_FAST, 1, 11), (True, capi.PRECISION_F64, 3, 2),
                                                      (True, capi.PRECISION_F32_FAST, 1, 0)]]


@pytest.mark.parametrize("whitted,precision,stride,offset", RESOLVE)
def test_tile_render_equals_replay(whitted, precision, stride, offset):
    """vrj_render_tile in one batch at spp 1, 2, 7 and 32.  With srgb8 asked for the call never coalesces, so the 1- and
    2-spp calls run k_resolve; without it a simple-random 1..4-spp call may run k_resolve_multi: both are checked."""
    hs = scene()
    kw = dict(max_depth=6, seed=3, precision=precision)
    if whitted:
        kw.update(whitted_kw(hs))
    for spp in (1, 2, 7, 32):
        want = replay_tile(hs, TILE, H, W, spp, offset, stride, **kw)
        for extra in ((), ("srgb8",)):
            got = hs.render(TILE, H, W, spp=spp, sample_offset=offset, sample_stride=stride,
                            want=tuple(n for n, _ in FIVE) + extra, **kw)
            assert_bits(got, want, [n for n, _ in FIVE])


def test_split_batches_equal_replay(monkeypatch):
    """A path budget of 2^16 on a 95 x 73 tile: batches of 9 samples, so 37 spp (a prime) take batches that do not divide
    it.  vrj_render_tile, vrj_render_adaptive and vrj_render_counts all equal their replays."""
    monkeypatch.setenv("VRJ_PATH_BUDGET_LOG2", "16")
    hs = build()
    hs.device_scene(0)  # the budget is read when the device scene is created
    monkeypatch.delenv("VRJ_PATH_BUDGET_LOG2")
    sampler = scene()
    w2, h2, tile = 101, 77, (3, 98, 2, 75)
    npix = 95 * 73
    kw = dict(max_depth=6, seed=9, sample_offset=4)
    spp = 37
    got = hs.render(tile, h2, w2, spp=spp, **kw)
    assert 2 <= got["stats"].resolve_launches < spp
    assert_bits(got, replay_tile(hs, tile, h2, w2, spp, sampler=sampler, **kw), [n for n, _ in FIVE])

    a = hs.render_adaptive(tile, h2, w2, 6, 30, 8, 0.02, **kw)
    n1 = a["weight"].astype(np.int64)
    assert a["adaptive"].passes >= 2 and n1.max() > 6
    assert_bits(a, replay_passes(hs, tile, h2, w2, np.zeros(npix), n1, sampler=sampler, **kw), [n for n, _ in OUTPUTS])

    cmap = np.random.default_rng(2).integers(0, spp + 1, npix).astype(np.uint32)
    r = hs.render_counts(tile, h2, w2, cmap, **kw)
    assert r["counts"].batches >= 2
    assert_bits(r, replay_passes(hs, tile, h2, w2, np.zeros(npix), cmap, sampler=sampler, **kw), [n for n, _ in OUTPUTS])


# ------------------------------------------------------------------------------------------------ accumulate = 1
@pytest.mark.parametrize("memory,null", [(capi.MEM_HOST, None), (capi.MEM_DEVICE, None), (capi.MEM_HOST, "colour_bias"),
                                         (capi.MEM_DEVICE, "colour_bias")], ids=["host", "device", "host-null-bias", "device-null-bias"])
def test_continue_an_arbitrary_state(memory, null):
    """vrj_render_tile with accumulate = 1 from random sums, non-zero compensation terms and non-integer weights; a NULL
    colour_bias starts at zero (and is not written)."""
    hs = scene()
    kw = dict(max_depth=6, seed=5, sample_offset=3, sample_stride=2)
    st0 = random_state(17, NPIX, integral=False)
    arrs = {n: st0[n].copy() for n, _ in KAHAN}
    arrs["colour"] = np.zeros(NPIX * 3)
    if null:
        del arrs[null]
    if memory == capi.MEM_DEVICE:
        import torch
        dev = {n: torch.from_numpy(a).to("cuda:0") for n, a in arrs.items()}
        torch.cuda.synchronize()  # the library reads them on a stream of its own
        render_into(hs, TILE, H, W, {n: t.data_ptr() for n, t in dev.items()}, memory, True, spp=5, **kw)
        got = {n: t.cpu().numpy() for n, t in dev.items()}
    else:
        render_into(hs, TILE, H, W, {n: a.ctypes.data for n, a in arrs.items()}, memory, True, spp=5, **kw)
        got = arrs
    want = replay_tile(hs, TILE, H, W, 5, state0={n: st0[n] for n, _ in KAHAN if n != null}, **kw)
    assert_bits(got, want, [n for n, _ in FIVE if n != null])


# ------------------------------------------------------------------------------------------------ the pass-based calls
PASSES = [pytest.param(False, capi.PRECISION_F64, 1, 0, id="simple-f64"), pytest.param(True, capi.PRECISION_F64, 2, 3, id="whitted-f64-s2"),
          pytest.param(False, capi.PRECISION_F32_FAST, 3, 1, id="simple-f32fast-s3")]


def pass_kw(hs, whitted, precision, stride, offset):
    kw = dict(max_depth=6, seed=11, precision=precision, sample_stride=stride, sample_offset=offset)
    if whitted:
        kw.update(whitted_kw(hs))
    return kw


@pytest.mark.parametrize("whitted,precision,stride,offset", PASSES)
def test_adaptive_and_progressive_equal_replay(whitted, precision, stride, offset):
    """k_resolve_adaptive: vrj_render_adaptive and vrj_render_progressive from zero, and vrj_render_progressive continuing a
    random state (integral weights, non-zero colour_bias): every pixel is the replay of samples n0 .. n_final - 1 on its
    initial state, n_final being the weight the call returns."""
    hs = scene()
    kw = pass_kw(hs, whitted, precision, stride, offset)
    zero = np.zeros(NPIX)
    a = hs.render_adaptive(TILE, H, W, 4, 20, 4, 0.05, **kw)
    n1 = a["weight"].astype(np.int64)
    assert a["adaptive"].passes >= 2 and n1.max() > 4 and (n1 >= 4).all()
    assert_bits(a, replay_passes(hs, TILE, H, W, zero, n1, **kw), [n for n, _ in OUTPUTS])

    p = hs.render_progressive(TILE, H, W, 4, 20, 4, 0.05, max_passes=2, want=("colour",), **kw)
    n1 = p["weight"].astype(np.int64)
    assert p["progressive"].passes == 2 and n1.max() > 4
    assert_bits(p, replay_passes(hs, TILE, H, W, zero, n1, **kw), [n for n, _ in OUTPUTS])

    st0 = random_state(23, NPIX, integral=True)
    c = hs.render_progressive(TILE, H, W, 4, 16, 3, 0.02, state=st0, want=("colour",), **kw)
    n0, n1 = st0["weight"].astype(np.int64), c["weight"].astype(np.int64)
    assert (n1 > n0).any() and (n1 >= 4).all() and c["progressive"].passes >= 1
    assert_bits(c, replay_passes(hs, TILE, H, W, n0, n1, state0=st0, **kw), [n for n, _ in OUTPUTS])


@pytest.mark.parametrize("whitted,precision,stride,offset", PASSES)
def test_counts_equal_replay(whitted, precision, stride, offset):
    """k_resolve_counts: vrj_render_counts from zero and continuing a random state; pixel p ends at n0 + c[p]."""
    hs = scene()
    kw = pass_kw(hs, whitted, precision, stride, offset)
    cmap = np.random.default_rng(31).choice(np.array([0, 1, 2, 5, 9], np.uint32), NPIX)
    r = hs.render_counts(TILE, H, W, cmap, **kw)
    assert np.array_equal(r["weight"], cmap.astype(np.float64))
    assert_bits(r, replay_passes(hs, TILE, H, W, np.zeros(NPIX), cmap, **kw), [n for n, _ in OUTPUTS])

    st0 = random_state(37, NPIX, integral=True)
    r = hs.render_counts(TILE, H, W, cmap, state=st0, **kw)
    n0 = st0["weight"].astype(np.int64)
    assert_bits(r, replay_passes(hs, TILE, H, W, n0, n0 + cmap, state0=st0, **kw), [n for n, _ in OUTPUTS])


# ------------------------------------------------------------------------------------------------ the piecewise resolve
C3_W, C3_H = 600, 540
C3_TILE = (40, 552, 20, 532)  # 512 x 512 = 2^18 pixels: the smallest tile whose last batch resolves in pieces
C3_NPIX = 1 << 18
C3_KW = dict(max_depth=8, seed=21)  # depth <= 12: no drain check, so the launch count is the same from call to call


@pytest.fixture
def pinned(request):
    """pinned(names) -> a dict of page-locked float64 arrays (vrj_alloc_host) for the C3 tile, freed after the test"""
    L, ptrs = capi.cuda(), []

    def make(names=tuple(n for n, _ in FIVE)):
        out = {}
        for name, per in FIVE:
            if name in names:
                p = L.vrj_alloc_host(C3_NPIX * per * 8)
                assert p
                ptrs.append(p)
                out[name] = np.ctypeslib.as_array(C.cast(p, C.POINTER(C.c_double)), (C3_NPIX * per,))
        return out

    def free():
        for p in ptrs:
            L.vrj_free_host(p)

    request.addfinalizer(free)
    return make


def c3_replay(spp, offset=0, state0=None):
    return replay_tile(scene("lambertian", 6), C3_TILE, C3_H, C3_W, spp, offset, state0=state0, **C3_KW)


def test_piecewise_resolve_into_pinned_memory(pinned):
    """A 512 x 512 tile of C3 at 8 spp into vrj_alloc_host buffers: the last batch resolves in four pieces, each copied to
    the host behind its own event.  The arrays equal the replay and the same call into pageable arrays."""
    hs = scene("lambertian", 6)
    pageable = hs.render(C3_TILE, C3_H, C3_W, spp=8, **C3_KW)
    buf = pinned()
    got = hs.render(C3_TILE, C3_H, C3_W, spp=8, buffers=buf, **C3_KW)
    assert got["stats"].kernel_launches == pageable["stats"].kernel_launches + 3  # four resolve pieces instead of one
    want = c3_replay(8)
    assert_bits(got, want, [n for n, _ in FIVE])
    assert_bits(pageable, want, [n for n, _ in FIVE])

    # bench.py's end-to-end pattern: colour and weight only, the same pinned buffers call after call
    cw = pinned(("colour", "weight"))
    for offset in (0, 8):
        r = hs.render(C3_TILE, C3_H, C3_W, spp=8, sample_offset=offset, want=("colour", "weight"), buffers=cw, **C3_KW)
        assert r["stats"].kernel_launches == got["stats"].kernel_launches
        assert_bits(r, c3_replay(8, offset), ["colour", "weight"])
    # a pinned state continued by a second pinned call (accumulate = 1): samples 0 .. 15
    st = render_into(hs, C3_TILE, C3_H, C3_W, {n: a.ctypes.data for n, a in buf.items()}, capi.MEM_HOST, True, spp=8,
                     sample_offset=8, **C3_KW)
    assert st.kernel_launches == got["stats"].kernel_launches
    assert_bits(buf, c3_replay(16), [n for n, _ in FIVE])


def test_piecewise_resolve_of_a_partial_last_batch(monkeypatch, pinned):
    """A path budget of 2^21 splits 20 spp of the 2^18-pixel tile into batches of 8, 8 and 4; only the last resolves in
    pieces, with 4 samples."""
    monkeypatch.setenv("VRJ_PATH_BUDGET_LOG2", "21")
    hs = build("lambertian", 6)
    hs.device_scene(0)
    monkeypatch.delenv("VRJ_PATH_BUDGET_LOG2")
    pageable = hs.render(C3_TILE, C3_H, C3_W, spp=20, **C3_KW)
    got = hs.render(C3_TILE, C3_H, C3_W, spp=20, buffers=pinned(), **C3_KW)
    assert pageable["stats"].resolve_launches == 3
    assert got["stats"].kernel_launches == pageable["stats"].kernel_launches + 3
    want = c3_replay(20)
    assert_bits(got, want, [n for n, _ in FIVE])
    assert_bits(pageable, want, [n for n, _ in FIVE])


def test_piecewise_resolve_from_three_threads(pinned):
    """Three threads render into pinned buffers of their own at different offsets at the same time; each call's copies
    come from its own pieces."""
    hs = scene("lambertian", 6)
    offsets = (0, 8, 16)
    wants = {o: c3_replay(8, o) for o in offsets}
    bufs = {o: pinned() for o in offsets}
    res, errors = {}, []

    def work(o):
        try:
            res[o] = hs.render(C3_TILE, C3_H, C3_W, spp=8, sample_offset=o, buffers=bufs[o], **C3_KW)
        except Exception as e:  # noqa: BLE001 -- reported below, on the test's thread
            errors.append(e)

    threads = [threading.Thread(target=work, args=(o,)) for o in offsets]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    assert not errors, errors
    for o in offsets:
        assert_bits(res[o], wants[o], [n for n, _ in FIVE])


# ------------------------------------------------------------------------------------------------ 32-bit edges of the indices
EDGES = [pytest.param(dict(sample_offset=(1 << 32) - 2), 4, W, H, TILE, id="offset-2^32-2"),
         pytest.param(dict(sample_offset=U64 - 2), 4, W, H, TILE, id="offset-2^64-2"),
         pytest.param(dict(seed=(1 << 63) + 12345), 4, W, H, TILE, id="seed-2^63"),
         pytest.param(dict(sample_offset=5), 3, 65535, 65537, (65535 - 7, 65535, 65537 - 5, 65537), id="far-corner-2^32-1-pixels")]


@pytest.mark.parametrize("kw,spp,width,height,tile", EDGES)
def test_index_edges_match_the_oracle_and_the_replay(kw, spp, width, height, tile):
    """The device's photons equal the oracle's (relative 1e-12, Lambertian) and the tile render equals its replay where a
    sample index crosses into the Philox counter's high word, wraps mod 2^64, the seed has its top bit set, or the pixel
    index reaches 2^32 - 2 (the last pixel of a 65535 x 65537 image, the largest allowed)."""
    hs = scene()
    orc = O.OracleScene(hs.spec)
    kw = dict(dict(max_depth=6, seed=13), **kw)
    g = hs.render(tile, height, width, spp=spp, want_photons=True, **kw)
    r = orc.render(tile, height, width, spp=spp, want_photons=True, **kw)
    photons_close(g["photons"], r["photons"], 1e-12)
    assert (g["photons"][..., 1] != 0).any()
    assert_bits(g, replay_tile(hs, tile, height, width, spp, **kw), [n for n, _ in FIVE])


def test_stride_past_2_32_on_tile_adaptive_and_counts():
    """sample_stride = 2^31 + 1: sample k of a pixel is offset + k * stride, past 2^32 from k = 2, on the tile kernels
    (vrj_render_tile), the LIST kernels of a second adaptive pass and the slot bases of vrj_render_counts."""
    hs = scene()
    stride = (1 << 31) + 1
    kw = dict(max_depth=6, seed=17, sample_offset=7, sample_stride=stride)
    assert_bits(hs.render(TILE, H, W, spp=3, **kw), replay_tile(hs, TILE, H, W, 3, **kw), [n for n, _ in FIVE])
    a = hs.render_adaptive(TILE, H, W, 2, 3, 1, 1e-6, **kw)  # a pixel of non-zero variance takes a second pass: sample 2
    assert a["adaptive"].passes == 2 and (a["weight"] == 3).any()
    assert_bits(a, replay_passes(hs, TILE, H, W, np.zeros(NPIX), a["weight"], **kw), [n for n, _ in OUTPUTS])
    st0 = random_state(41, NPIX, integral=True)
    cmap = np.random.default_rng(43).integers(0, 4, NPIX).astype(np.uint32)
    r = hs.render_counts(TILE, H, W, cmap, state=st0, **kw)
    n0 = st0["weight"].astype(np.int64)
    assert_bits(r, replay_passes(hs, TILE, H, W, n0, n0 + cmap, state0=st0, **kw), [n for n, _ in OUTPUTS])


# ------------------------------------------------------------------------------------------------ image size limit
def five_statuses(hs, tile, height, width):
    """the status of vrj_render_tile, _adaptive, _progressive, _counts and vrj_render_aux on `tile`"""
    L = capi.cuda()
    sc = hs.device_scene(0)
    t = capi.Tile(*tile)
    npix = (tile[1] - tile[0]) * (tile[3] - tile[2])
    arrs = {n: np.zeros(npix * per) for n, per in OUTPUTS}

    def ao():
        o = capi.AccumOut(memory=capi.MEM_HOST, accumulate=0)
        for n, _ in FIVE:
            setattr(o, n, arrs[n].ctypes.data)
        return o

    p1, k1 = hs.make_params(spp=1, max_depth=4)
    p0, k0 = hs.make_params(spp=0, max_depth=4)
    ap = capi.AdaptiveParams(min_samples=2, max_samples=2, pass_samples=1, rel_error=0.1)
    pp = capi.ProgressiveParams(min_samples=2, max_samples=2, pass_samples=1, rel_error=0.1)
    cmap = np.ones(npix, np.uint32)
    depth = np.zeros(npix)
    aux = capi.AuxOut(memory=capi.MEM_HOST, depth=depth.ctypes.data)
    ysq = arrs["y_sq_sum"].ctypes.data
    return {"tile": L.vrj_render_tile(sc, C.byref(t), height, width, C.byref(p1), C.byref(ao())),
            "adaptive": L.vrj_render_adaptive(sc, C.byref(t), height, width, C.byref(p0), C.byref(ap), C.byref(ao()), ysq, None),
            "progressive": L.vrj_render_progressive(sc, C.byref(t), height, width, C.byref(p0), C.byref(pp), C.byref(ao()), ysq, None),
            "counts": L.vrj_render_counts(sc, C.byref(t), height, width, C.byref(p0), cmap.ctypes.data, C.byref(ao()), ysq, None),
            "aux": L.vrj_render_aux(sc, C.byref(t), height, width, C.byref(p1), C.byref(aux))}


def test_images_over_2_32_minus_1_pixels_are_refused_without_wrapping():
    """width * height wraps in 64 bits for 2^32 x 2^32 and 2^63 x 2; those images, and 65536 x 65536 (2^32 pixels), are
    VRJ_ERR_UNSUPPORTED on every render call, while 65535 x 65537 (2^32 - 1 pixels) renders."""
    hs = scene()
    for width, height in ((1 << 32, 1 << 32), (1 << 63, 2), (65536, 65536)):
        st = five_statuses(hs, (0, 1, 0, 1), height, width)
        assert st == dict.fromkeys(st, ERR_UNSUPPORTED), (width, height, st)
        assert b"2^32" in capi.cuda().vrj_last_error()
    st = five_statuses(hs, (65535 - 2, 65535, 65537 - 1, 65537), 65537, 65535)
    assert st == dict.fromkeys(st, capi.OK), st
