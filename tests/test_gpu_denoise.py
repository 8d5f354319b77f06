"""First-hit features (vrj_render_aux) and the variance-guided a-trous filter (vrj_denoise) on the GPU.  Run with `-m gpu`.

The bar is bit equality wherever the arithmetic allows it: the features against the CPU oracle's hits on the same camera
rays and against a numpy replay of the header's sums; the filter against a numpy replay of the header's filter (to the last
bits of exp / pow only)."""
import ctypes as C
import threading

import numpy as np
import pytest

import vanrijn_b200 as V
from vanrijn_b200 import capi, host, scenes

import oraclelib as O

pytestmark = pytest.mark.gpu

W, H = 37, 23                 # odd image
TILE = (5, 30, 3, 20)         # odd tile: 25 x 17 pixels
TW, TH = TILE[1] - TILE[0], TILE[3] - TILE[2]
NPIX = TW * TH
SEED = 3
KW = dict(max_depth=6, seed=SEED)
FEATURES = ("normal", "depth", "object_id", "material")
H5 = (1.0 / 16.0, 1.0 / 4.0, 3.0 / 8.0, 1.0 / 4.0, 1.0 / 16.0)


def bits(a):
    return np.ascontiguousarray(a).view(np.uint64)


@pytest.fixture(scope="module")
def small():
    spec = scenes.scene_main(subdivisions=2, obj=False)
    return spec, V.build_scene(spec), O.OracleScene(spec)


def np_normalize(v):
    """vrj_device.cuh's normalize: v * (1 / sqrt(((0 + x*x) + y*y) + z*z))."""
    n = np.sqrt(((0.0 + v[..., 0] * v[..., 0]) + v[..., 1] * v[..., 1]) + v[..., 2] * v[..., 2])
    return v * (1.0 / n)[..., None]


def camera_rays(tile, height, width, cam, seed, sample):
    """The render's camera rays of `sample` for the tile's pixels (camera.rs:45-66 with the oracle's Rng{seed, pixel, sample,
    0} draws), directions before Ray::new's normalisation: both the oracle and the kernels normalise (px, py, 1) once."""
    L = O.lib()
    sc, ec, sr, er = tile
    rows, cols = np.meshgrid(np.arange(sr, er), np.arange(sc, ec), indexing="ij")
    rows, cols = rows.ravel(), cols.ravel()
    ux = np.array([L.orc_rng_f64(seed, int(r * width + c), sample, 0) for r, c in zip(rows, cols)])
    uy = np.array([L.orc_rng_f64(seed, int(r * width + c), sample, 1) for r, c in zip(rows, cols)])
    fw, fh = (width / height, 1.0) if width > height else (1.0, width / height)
    px = (cols.astype(np.float64) + ux) * (fw * (1.0 / width)) - fw * 0.5
    py = ((height - (rows + 1)).astype(np.float64) + uy) * (fh * (1.0 / height)) - fh * 0.5
    d = np.stack([px, py, np.ones_like(px)], -1)
    return np.tile(np.asarray(cam, np.float64), (len(d), 1)), d


def oracle_hits(spec, orc, tile, height, width, seed, sample):
    """Per pixel: the oracle's (object_id, t), the unnormalised shading normal and material of the hit primitive
    (orc_{sphere,plane,triangle}_intersect), and whether the ray keeps clear of triangle edges (1e-6, as the id tests)."""
    o, d = camera_rays(tile, height, width, spec.camera, seed, sample)
    obj, prim, t, _ = orc.trace(o, d)
    clear = orc.edge_distance(o, d) > 1e-6
    normal = np.zeros((len(o), 3))
    material = np.full(len(o), -1, np.int32)
    L = O.lib()
    for i in np.flatnonzero(obj >= 0):
        kind, *rest = spec.objects[obj[i]]
        if kind == "list":
            p = rest[0][prim[i]]
            if p[0] == "sphere":
                h = O.hit16(L.orc_sphere_intersect, np.array(p[1], float), float(p[2]), o[i], d[i])
            elif p[0] == "plane":
                h = O.hit16(L.orc_plane_intersect, np.array(p[1], float), float(p[2]), o[i], d[i])
            else:
                h = O.hit16(L.orc_triangle_intersect, np.asarray(p[1], float), np.asarray(p[2], float), o[i], d[i])
            mat = p[3]
        else:  # mesh: prim is the triangle's row
            v, n, mat = rest
            h = O.hit16(L.orc_triangle_intersect, v.reshape(-1, 9)[prim[i]], n.reshape(-1, 9)[prim[i]], o[i], d[i])
        assert h is not None
        normal[i], material[i] = h["normal"], mat
    return dict(object_id=obj, t=t, normal=normal, material=material, clear=clear, origins=o, dirs=d)


# ---------------------------------------------------------------------------------------------------------- aux features
def test_aux_equals_the_oracle_bit_for_bit(small):
    spec, hs, orc = small
    a = hs.render_aux(TILE, H, W, spp=1, sample_offset=5, **KW)
    r = oracle_hits(spec, orc, TILE, H, W, SEED, 5)
    ok = r["clear"]
    assert ok.sum() >= NPIX - 10 and (r["object_id"][ok] >= 0).sum() > NPIX // 2 and (r["object_id"][ok] < 0).any()
    assert np.array_equal(a["object_id"][ok], r["object_id"][ok])
    miss = r["object_id"] < 0
    assert np.all(np.isinf(a["depth"][ok & miss])) and np.all(a["material"][ok & miss] == -1)
    assert np.all(a["normal"].reshape(-1, 3)[ok & miss] == 0.0)
    hit = ok & ~miss
    assert np.array_equal(bits(a["depth"][hit]), bits(r["t"][hit]))
    assert np.array_equal(bits(a["normal"].reshape(-1, 3)[hit]), bits(np_normalize(r["normal"][hit])))
    assert np.array_equal(a["material"][hit], r["material"][hit])
    # every ray, edges included, against the library's own closest-hit query on the same rays
    g_obj, _, g_t, _ = hs.trace(r["origins"], r["dirs"])
    assert np.array_equal(a["object_id"], g_obj) and np.array_equal(bits(a["depth"]), bits(g_t))
    st = a["stats"]
    assert st.primary_rays == NPIX and st.kernel_launches == 1 and st.device_ms > 0.0


def test_aux_aggregates_samples_as_the_header_states(small):
    spec, hs, orc = small
    K, G, OFF = 3, 3, 7
    a = hs.render_aux(TILE, H, W, spp=K, sample_offset=OFF, sample_stride=G, **KW)
    ones = [hs.render_aux(TILE, H, W, spp=1, sample_offset=OFF + k * G, **KW) for k in range(K)]
    raw = [oracle_hits(spec, orc, TILE, H, W, SEED, OFF + k * G) for k in range(K)]
    nsum, tsum = np.zeros((NPIX, 3)), np.zeros(NPIX)
    hits = np.zeros(NPIX, np.int64)
    obj, mat = np.full(NPIX, -1, np.int32), np.full(NPIX, -1, np.int32)
    for one, r in zip(ones, raw):
        h = one["object_id"] >= 0
        nsum[h] = nsum[h] + r["normal"][h]   # the unnormalised n_k (the 1-spp call returns normalize(n_k))
        tsum[h] = tsum[h] + one["depth"][h]  # a 1-spp depth is t_k exactly (t * (1.0 / 1))
        first = h & (hits == 0)
        obj[first], mat[first] = one["object_id"][first], one["material"][first]
        hits += h
    clear = np.logical_and.reduce([r["clear"] for r in raw])
    assert clear.sum() >= NPIX - 20 and ((hits > 0) & (hits < K)).any()
    with np.errstate(all="ignore"):
        depth = np.where(hits > 0, tsum * (1.0 / hits), np.inf)
        normal = np.where((hits > 0)[:, None], np_normalize(nsum), 0.0)
    assert np.array_equal(a["object_id"], obj) and np.array_equal(a["material"], mat)
    assert np.array_equal(bits(a["depth"]), bits(depth))
    assert np.array_equal(bits(a["normal"].reshape(-1, 3)[clear]), bits(normal[clear]))
    assert a["stats"].primary_rays == K * NPIX


def test_aux_rays_are_the_render_rays(small):
    spec, hs, orc = small
    SPP, OFF = 4, 11
    u = hs.render(TILE, H, W, spp=SPP, sample_offset=OFF, want=("colour",), want_photons=True, **KW)
    misses = 0
    for k in range(SPP):
        a = hs.render_aux(TILE, H, W, spp=1, sample_offset=OFF + k, want=("object_id",), **KW)
        m = a["object_id"] == -1
        assert np.all(u["photons"][k][m] == 0.0), k
        misses += int(m.sum())
    assert misses > 0 and misses == u["stats"].paths_missed


def test_aux_device_memory_and_precision_ignored(small):
    spec, hs, orc = small
    ref = hs.render_aux(TILE, H, W, spp=2, sample_offset=3, **KW)
    f32 = hs.render_aux(TILE, H, W, spp=2, sample_offset=3, precision=capi.PRECISION_F32_FAST, bvh_filter=capi.FILTER_Q16, **KW)
    dev = aux_device(hs, TILE, H, W, spp=2, sample_offset=3, **KW)
    for name in FEATURES:
        assert np.array_equal(f32[name].view(np.uint8), ref[name].view(np.uint8)), name
        assert np.array_equal(dev[name].view(np.uint8), ref[name].view(np.uint8)), name


# ---------------------------------------------------------------------------------------------------------- device plumbing
class DeviceArrays:
    """Pooled device blocks (vrj_alloc_device) freed on exit."""

    def __init__(self):
        self.L, self.ptrs = capi.cuda(), []

    def __enter__(self):
        return self

    def alloc(self, nbytes):
        p = self.L.vrj_alloc_device(0, max(nbytes, 8))
        assert p
        self.ptrs.append(p)
        return p

    def fetch(self, ptr, n, dtype):
        out = np.zeros(n, dtype)
        capi.check(self.L.vrj_copy_to_host(0, out.ctypes.data, ptr, out.nbytes))
        return out

    def __exit__(self, *exc):
        for p in self.ptrs:
            self.L.vrj_free_device(p)


def aux_device(hs, tile, height, width, spp=1, **kw):
    """vrj_render_aux into device memory, copied back (normal / depth as float64, ids as int32)."""
    npix = (tile[1] - tile[0]) * (tile[3] - tile[2])
    with DeviceArrays() as d:
        out = aux_device_ptrs(hs, d, tile, height, width, spp, **kw)
        return {n: d.fetch(out[n], npix * (3 if n == "normal" else 1), np.int32 if n in ("object_id", "material") else np.float64)
                for n in FEATURES}


def aux_device_ptrs(hs, d, tile, height, width, spp=1, **kw):
    npix = (tile[1] - tile[0]) * (tile[3] - tile[2])
    p, keep = hs.make_params(spp=spp, **kw)
    ao = capi.AuxOut(memory=capi.MEM_DEVICE)
    out = {}
    for n, nbytes in (("normal", 24), ("depth", 8), ("object_id", 4), ("material", 4)):
        out[n] = d.alloc(npix * nbytes)
        setattr(ao, n, out[n])
    st = capi.Stats()
    ao.stats = C.pointer(st)
    t = capi.Tile(*tile)
    capi.check(capi.cuda().vrj_render_aux(hs.device_scene(0), C.byref(t), height, width, C.byref(p), C.byref(ao)))
    out["stats"] = st
    return out


def adaptive_device_ptrs(hs, d, tile, height, width, spp, **kw):
    """vrj_render_adaptive with min == max == spp (the uniform frame) into device memory: colour_sum, weight, y_sq_sum."""
    npix = (tile[1] - tile[0]) * (tile[3] - tile[2])
    p, keep = hs.make_params(spp=0, **kw)
    ap = capi.AdaptiveParams(min_samples=spp, max_samples=spp, pass_samples=1, rel_error=0.01)
    ao = capi.AccumOut(memory=capi.MEM_DEVICE, accumulate=0)
    out = {"colour_sum": d.alloc(npix * 24), "weight": d.alloc(npix * 8), "y_sq_sum": d.alloc(npix * 8)}
    ao.colour_sum, ao.weight = out["colour_sum"], out["weight"]
    st = capi.Stats()
    ao.stats = C.pointer(st)
    t = capi.Tile(*tile)
    capi.check(capi.cuda().vrj_render_adaptive(hs.device_scene(0), C.byref(t), height, width, C.byref(p), C.byref(ap), C.byref(ao),
                                               out["y_sq_sum"], None))
    return out


def denoise_device(d, ins, tw, th, params, want_srgb8=False):
    npix = tw * th
    colour = d.alloc(npix * 24)
    srgb8 = d.alloc(npix * 3) if want_srgb8 else None
    ms = C.c_double(-1.0)
    capi.check(capi.cuda().vrj_denoise(0, capi.MEM_DEVICE, tw, th, ins["colour_sum"], ins["weight"], ins["y_sq_sum"], ins["normal"],
                                       ins["depth"], ins["material"], C.byref(params), colour, srgb8, C.byref(ms)))
    out = {"colour": d.fetch(colour, npix * 3, np.float64), "device_ms": ms.value}
    if want_srgb8:
        out["srgb8"] = d.fetch(srgb8, npix * 3, np.uint8)
    return out


# ---------------------------------------------------------------------------------------------------------- the filter
def replay(colour_sum, weight, y_sq_sum, normal, depth, material, tw, th, iterations, sl, sn, sz):
    """The header's filter in numpy, operation for operation (numpy never fuses a multiply-add)."""
    n, s, q = weight.reshape(th, tw), colour_sum.reshape(th, tw, 3), y_sq_sum.reshape(th, tw)
    N, Z, ID = normal.reshape(th, tw, 3), depth.reshape(th, tw), material.reshape(th, tw)
    with np.errstate(all="ignore"):
        inv = 1.0 / n
        c = s * inv[..., None]
        m = s[..., 1] * inv
        v = (q - s[..., 1] * m) / (n - 1.0)
        v = np.where(v < 0.0, 0.0, v)
        var = v * inv
        valid = (n >= 2.0) & np.all(np.isfinite(c), axis=-1) & np.isfinite(var)
        c0 = c.copy()
        for i in range(iterations):
            step = 1 << i
            Wt, Cs, Vs = np.zeros((th, tw)), np.zeros((th, tw, 3)), np.zeros((th, tw))
            lum_den = sl * np.sqrt(var) + 1e-10
            for dy in range(-2, 3):
                for dx in range(-2, 3):
                    ys, xs = np.arange(th) + step * dy, np.arange(tw) + step * dx
                    yin, xin = (ys >= 0) & (ys < th), (xs >= 0) & (xs < tw)
                    yc, xc = np.clip(ys, 0, th - 1), np.clip(xs, 0, tw - 1)
                    take = yin[:, None] & xin[None, :]
                    cq, vq, vq_ok = c[yc][:, xc], var[yc][:, xc], valid[yc][:, xc]
                    take = take & vq_ok
                    w = np.full((th, tw), H5[dx + 2] * H5[dy + 2])
                    if dx or dy:
                        idq, Nq, Zq = ID[yc][:, xc], N[yc][:, xc], Z[yc][:, xc]
                        take = take & (idq == ID)
                        dot = ((0.0 + N[..., 0] * Nq[..., 0]) + N[..., 1] * Nq[..., 1]) + N[..., 2] * Nq[..., 2]
                        geo = ID >= 0
                        dist = float(max(abs(dx), abs(dy)))
                        w = np.where(geo, w * np.power(np.maximum(0.0, dot), sn), w)
                        w = np.where(geo, w * np.exp(-np.abs(Z - Zq) / (((sz * Z) * float(step)) * dist)), w)
                        w = w * np.exp(-np.abs(c[..., 1] - cq[..., 1]) / lum_den)
                    w = np.where(take, w, 0.0)
                    Wt = np.where(take, Wt + w, Wt)
                    Cs = np.where(take[..., None], Cs + w[..., None] * cq, Cs)
                    Vs = np.where(take, Vs + (w * w) * vq, Vs)
            cn = Cs * (1.0 / Wt)[..., None]
            vn = Vs * (1.0 / (Wt * Wt))
            c = np.where(valid[..., None], cn, c0)
            var = np.where(valid, vn, var)
    return c.reshape(-1)


def small_inputs(hs, spp=8, offset=0):
    r = hs.render_adaptive(TILE, H, W, spp, spp, 1, 0.01, want=("colour", "colour_sum", "weight", "y_sq_sum"), sample_offset=offset, **KW)
    a = hs.render_aux(TILE, H, W, spp=1, sample_offset=offset, **KW)
    return r, a


DEFAULT = dict(sigma_luminance=host.DENOISE_SIGMA_LUMINANCE, sigma_normal=host.DENOISE_SIGMA_NORMAL, sigma_depth=host.DENOISE_SIGMA_DEPTH)


@pytest.mark.parametrize("memory", [capi.MEM_HOST, capi.MEM_DEVICE], ids=["host", "device"])
def test_filter_replayed_in_numpy(small, memory):
    spec, hs, orc = small
    r, a = small_inputs(hs)
    assert (a["material"] == -1).any() and len(np.unique(a["material"])) >= 3
    for it in range(6):
        if memory == capi.MEM_HOST:
            g = host.denoise(r["colour_sum"], r["weight"], r["y_sq_sum"], a, TW, TH, iterations=it, want_srgb8=True, **DEFAULT)
        else:
            with DeviceArrays() as d:
                ins = adaptive_device_ptrs(hs, d, TILE, H, W, 8, **KW)
                ins.update(aux_device_ptrs(hs, d, TILE, H, W, 1, **KW))
                g = denoise_device(d, ins, TW, TH, capi.DenoiseParams(iterations=it, **DEFAULT), want_srgb8=True)
        want = replay(r["colour_sum"], r["weight"], r["y_sq_sum"], a["normal"], a["depth"], a["material"], TW, TH, it,
                      DEFAULT["sigma_luminance"], DEFAULT["sigma_normal"], DEFAULT["sigma_depth"])
        if it == 0:
            assert np.array_equal(bits(g["colour"]), bits(r["colour"]))  # colour_sum * (1/weight)
        np.testing.assert_allclose(g["colour"], want, rtol=1e-12, atol=0.0, err_msg="iterations=%d" % it)
        assert np.array_equal(g["srgb8"], host.tone_map(g["colour"]).reshape(-1)), it
        assert g["device_ms"] > 0.0
        if it >= 3:
            assert not np.array_equal(g["colour"], r["colour"])


def synthetic(tw=40, th=30, seed=0):
    rng = np.random.default_rng(seed)
    npix = tw * th
    n = np.full(npix, 16.0)
    y = rng.uniform(0.1, 1.0, (npix, 16))
    s = np.stack([y.sum(1) * 0.9, y.sum(1), y.sum(1) * 1.1], 1).reshape(-1)
    q = (y * y).sum(1)
    nrm = np_normalize(rng.normal(size=(npix, 3)) + np.array([0.0, 3.0, 0.0]))
    aux = {"normal": nrm.reshape(-1), "depth": rng.uniform(4.0, 6.0, npix), "material": (rng.uniform(size=npix) < 0.5).astype(np.int32)}
    return s, n, q, aux


def test_constant_image_stays_constant():
    tw, th = 40, 30
    npix = tw * th
    c = np.array([0.5, 0.375, 0.25])
    n = np.full(npix, 16.0)
    s = np.tile(c * 16.0, npix)
    q = np.full(npix, 16.0 * 0.375 * 0.375 + 15 * 0.01)
    aux = {"normal": np.tile([0.0, 1.0, 0.0], npix), "depth": np.full(npix, 5.0), "material": np.zeros(npix, np.int32)}
    for it in (1, 5, 10):
        g = host.denoise(s, n, q, aux, tw, th, iterations=it)
        np.testing.assert_array_max_ulp(g["colour"], np.tile(c, npix), maxulp=1)


def test_materials_do_not_mix():
    tw, th = 40, 30
    s, n, q, aux = synthetic(tw, th)
    a = aux["material"] == 0
    g1 = host.denoise(s, n, q, aux, tw, th, iterations=5)
    s2, q2 = s.copy().reshape(-1, 3), q.copy()
    s2[a] *= 7.0
    q2[a] *= 49.0
    g2 = host.denoise(s2.reshape(-1), n, q2, aux, tw, th, iterations=5)
    b = ~a
    assert not np.array_equal(g1["colour"].reshape(-1, 3)[a], g2["colour"].reshape(-1, 3)[a])
    assert np.array_equal(bits(g1["colour"].reshape(-1, 3)[b]), bits(g2["colour"].reshape(-1, 3)[b]))


def test_invalid_pixels_pass_through_and_are_ignored():
    tw, th = 40, 30
    s, n, q, aux = synthetic(tw, th)
    aux["material"][:] = 0
    nan_px, one_px = 10 * tw + 12, 11 * tw + 14
    runs = []
    for variant in range(3):
        s2, n2, q2 = s.copy().reshape(-1, 3), n.copy(), q.copy()
        s2[nan_px, 1] = np.nan
        n2[one_px], s2[one_px], q2[one_px] = 1.0, [0.2, 0.3, 0.4], 0.09
        if variant == 1:  # other contents of the same invalid pixels
            s2[nan_px] = [np.nan, 5.0, np.nan]
            s2[one_px], q2[one_px] = [9.0, 9.0, 9.0], 81.0
        if variant == 2:  # the replay
            runs.append(replay(s2.reshape(-1), n2, q2, aux["normal"], aux["depth"], aux["material"], tw, th, 5,
                               DEFAULT["sigma_luminance"], DEFAULT["sigma_normal"], DEFAULT["sigma_depth"]).reshape(-1, 3))
            continue
        g = host.denoise(s2.reshape(-1), n2, q2, aux, tw, th, iterations=5)["colour"].reshape(-1, 3)
        assert np.array_equal(bits(g[one_px]), bits(s2[one_px] * (1.0 / 1.0)))
        assert np.array_equal(bits(g[nan_px]), bits(s2[nan_px] * (1.0 / 16.0)))
        runs.append(g)
    keep = np.ones(tw * th, bool)
    keep[[nan_px, one_px]] = False
    assert np.array_equal(bits(runs[0][keep]), bits(runs[1][keep]))
    np.testing.assert_allclose(runs[0][keep], runs[2][keep], rtol=1e-12, atol=0.0)


# With the default parameters the denoised 8-spp frame of the small scene was measured at 0.263 of the noisy frame's relative
# RMSE of Y (NVIDIA B200, 1000 W; the frame is deterministic); the assertion is that ratio rounded up to 0.3.
QUALITY_RATIO = 0.3


def test_denoising_lowers_the_error(small):
    spec, hs, orc = small
    w, h = 128, 96
    full = (0, w, 0, h)
    ref = hs.render(full, h, w, spp=1024, want=("colour",), **dict(KW, sample_offset=1 << 40))["colour"].reshape(-1, 3)[:, 1]
    r = hs.render_adaptive(full, h, w, 8, 8, 1, 0.01, want=("colour", "colour_sum", "weight", "y_sq_sum"), **KW)
    a = hs.render_aux(full, h, w, spp=1, **KW)
    g = host.denoise(r["colour_sum"], r["weight"], r["y_sq_sum"], a, w, h)

    def rel_rmse(y):
        return float(np.sqrt(np.mean((y - ref) ** 2) / np.mean(ref ** 2)))

    noisy, clean = rel_rmse(r["colour"].reshape(-1, 3)[:, 1]), rel_rmse(g["colour"].reshape(-1, 3)[:, 1])
    print("relative RMSE of Y: noisy %.4f, denoised %.4f (ratio %.3f)" % (noisy, clean, clean / noisy))
    assert clean < QUALITY_RATIO * noisy, (noisy, clean)


# ---------------------------------------------------------------------------------------------------------- errors
def test_argument_errors_and_empty_tiles(small):
    spec, hs, orc = small
    L = capi.cuda()
    scene = hs.device_scene(0)
    t = capi.Tile(*TILE)
    buf = np.zeros(NPIX * 4)

    def aux(spp=1, tile=t, memory=capi.MEM_HOST, out=True):
        p, keep = hs.make_params(spp=spp, **KW)
        ao = capi.AuxOut(memory=memory, depth=buf.ctypes.data)
        return L.vrj_render_aux(scene, C.byref(tile), H, W, C.byref(p), C.byref(ao) if out else None)

    assert aux() == capi.OK
    assert aux(spp=0) == 1 and b"spp" in L.vrj_last_error()
    assert aux(memory=2) == 1
    assert aux(out=False) == 1
    assert aux(tile=capi.Tile(0, W + 1, 0, H)) == 1
    st = capi.Stats()
    p, keep = hs.make_params(spp=1, **KW)
    ao = capi.AuxOut(memory=capi.MEM_HOST, stats=C.pointer(st))
    assert L.vrj_render_aux(scene, C.byref(capi.Tile(4, 4, 0, H)), H, W, C.byref(p), C.byref(ao)) == capi.OK
    assert st.primary_rays == 0 and st.kernel_launches == 0

    s, n, q, a = synthetic(8, 4)
    arrs = [s, n, q, a["normal"], a["depth"], a["material"]]
    col = np.zeros(8 * 4 * 3)

    def den(params=None, memory=capi.MEM_HOST, tw=8, th=4, null=None, **pkw):
        ptrs = [x.ctypes.data for x in arrs] + [col.ctypes.data]
        if null is not None:
            ptrs[null] = None
        dpar = capi.DenoiseParams(**dict(dict(iterations=2, **DEFAULT), **pkw)) if params is None else params
        return L.vrj_denoise(0, memory, tw, th, *ptrs[:6], C.byref(dpar) if dpar is not False else None, ptrs[6], None, None)

    assert den() == capi.OK
    for i in range(7):
        assert den(null=i) == 1, i
        assert b"NULL" in L.vrj_last_error()
    assert den(params=False) == 1
    assert den(memory=2) == 1
    assert den(iterations=11) == 1 and b"iterations" in L.vrj_last_error()
    assert den(iterations=10) == capi.OK
    for name, bad in (("sigma_luminance", [0.0, -1.0, np.nan, np.inf]), ("sigma_normal", [-1.0, np.nan, np.inf]),
                      ("sigma_depth", [0.0, -1.0, np.nan, np.inf])):
        for v in bad:
            assert den(**{name: v}) == 1, (name, v)
            assert name.encode() in L.vrj_last_error()
    assert den(sigma_normal=0.0) == capi.OK
    ms = C.c_double(-1.0)
    dpar = capi.DenoiseParams(iterations=2, **DEFAULT)
    for tw, th in ((0, 4), (8, 0)):
        assert L.vrj_denoise(0, capi.MEM_HOST, tw, th, None, None, None, None, None, None, C.byref(dpar), None, None, C.byref(ms)) == capi.OK
        assert ms.value == 0.0


# ---------------------------------------------------------------------------------------------------------- full size
def test_c3_1080p_device_buffers_and_concurrent_with_a_render():
    hs = V.build_scene(scenes.scene_main())
    w, h = 1920, 1080
    full = (0, w, 0, h)
    npix = w * h
    kw = dict(max_depth=8, seed=5)
    params = capi.DenoiseParams(iterations=host.DENOISE_ITERATIONS, **DEFAULT)

    def aux_and_denoise(d, ins):
        a = aux_device_ptrs(hs, d, full, h, w, 1, **kw)
        ins = dict(ins, **{k: a[k] for k in FEATURES})
        g = denoise_device(d, ins, w, h, params, want_srgb8=True)
        g["aux_ms"], g["depth"] = a["stats"].device_ms, d.fetch(a["depth"], npix, np.float64)
        return g

    with DeviceArrays() as d:
        ins = adaptive_device_ptrs(hs, d, full, h, w, 4, **kw)
        g = aux_and_denoise(d, ins)
        assert np.all(np.isfinite(g["colour"]))
        assert g["aux_ms"] > 0.0 and g["device_ms"] > 0.0
        print("C3 1080p: aux %.3f ms, denoise (%d iterations) %.3f ms" % (g["aux_ms"], params.iterations, g["device_ms"]))
        u = hs.render(full, h, w, spp=4, want=("colour", "weight"), **dict(kw, sample_offset=100))
        res = {}

        def run_uniform():
            res["u"] = hs.render(full, h, w, spp=4, want=("colour", "weight"), **dict(kw, sample_offset=100))

        th = threading.Thread(target=run_uniform)
        th.start()
        g2 = aux_and_denoise(d, ins)
        th.join()
        for name in ("colour", "srgb8", "depth"):
            assert np.array_equal(g2[name].view(np.uint8), g[name].view(np.uint8)), name
        for name in ("colour", "weight"):
            assert np.array_equal(bits(res["u"][name]), bits(u[name])), name
