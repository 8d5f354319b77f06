"""GPU parity on the generated scenes of scene_content.py: sampled spectra of 2 to 200 samples, rgb colours of every basis
branch, all four materials, 1 to 16 lights, spheres / planes / flat-list triangles / meshes of 1 to 3200 triangles in up to
three list objects, exact-distance ties between and inside objects, and rays that lie in the plane of a triangle or a
plane.  Run with `-m gpu`.

Bars, as in test_gpu_parity.py: hit ids and distances bit-exact; per-sample radiance to 1e-12 in all-Lambertian scenes and
1e-9 otherwise, with wavelengths bit-identical and ray counters equal; Phong scenes keep the allowance for samples whose
direction follows CUDA's sin / cos instead of glibc's by an ulp, and their ray counters may differ by what those paths
trace."""
import functools

import numpy as np
import pytest

import helpers
import oraclelib as O
import scene_content
import vanrijn_b200 as V
from test_gpu_parity import photons_close
from vanrijn_b200 import capi

pytestmark = pytest.mark.gpu

FILTERS = (capi.FILTER_F32, capi.FILTER_F64, capi.FILTER_F32X4, capi.FILTER_Q16)
W, H, SPP = 64, 40, 3
# of W * H * SPP = 7680 samples: test_path_traced_samples_phong's allowance for paths that diverge by a libm ulp
PHONG_DIVERGED = 12
COUNTERS = ("primary_rays", "bounce_rays", "paths_missed", "paths_escaped", "paths_depth_limited")


@functools.lru_cache(maxsize=None)
def content(seed):
    c = scene_content.generate(seed)
    return c, V.build_scene(c.spec), O.OracleScene(c.spec)


def same_hits(g, r):
    """(object, primitive, distance) equal; a NaN distance equals a NaN distance whatever its sign bit."""
    gt, rt = g[2], r[2]
    nan = np.isnan(gt) & np.isnan(rt)
    return (g[0] == r[0]) & (g[1] == r[1]) & ((gt.view(np.uint64) == rt.view(np.uint64)) | nan)


def tie_rays(c, n=200, seed=0):
    """Per tie set: rays from in front of the shared geometry to points well inside it (barycentrics >= 0.1), so the rays
    are neither degenerate nor near an edge."""
    rng = np.random.default_rng(seed)
    out = []
    for t in c.ties:
        if "tri" in t:
            b = rng.dirichlet((1.0, 1.0, 1.0), size=n) * 0.7 + 0.1
            target = b @ t["tri"]
        else:
            u = rng.normal(size=(n, 3))
            u[:, 2] = -np.abs(u[:, 2]) - 1.0
            u /= np.linalg.norm(u, axis=1, keepdims=True)
            target = t["centre"] + 0.8 * t["radius"] * u
        d = np.tile([0.0, 0.0, 1.0], (n, 1)) + rng.normal(size=(n, 3)) * 0.3
        d[:, 2] = np.abs(d[:, 2]) + 0.3
        o = target - d * rng.uniform(0.3, 1.0, size=(n, 1))
        out.append((t, o, d))
    return out


@pytest.mark.parametrize("seed", scene_content.SEEDS)
def test_hits_bit_exact_with_ties(seed):
    """Camera rays and random rays in all four filters against the oracle's reference traversal, bit for bit (with the
    usual exclusion of degenerate and near-edge rays); rays aimed at every tie set compared without any exclusion, each
    set hit by at least 100 rays and won by the oracle's winner: the earlier object between objects, the later DFS leaf
    inside a BVH."""
    c, hs, orc = content(seed)
    o1, d1 = helpers.camera_rays(W * 2, H * 2, c.spec.camera)
    o2, d2 = helpers.sphere_rays(20000, (0.0, 0.5, 4.0), 14.0, seed=seed)
    o, d = np.concatenate([o1, o2]), np.concatenate([d1, d2])
    keep = helpers.exclude_degenerate(d)
    o, d = o[keep], d[keep]
    ref = orc.trace(o, d, mode=O.TRAVERSE_REFERENCE)
    ok = orc.edge_distance(o, d) > 1e-6
    assert (ref[0][ok] >= 0).sum() > 5000
    ties = tie_rays(c, seed=seed)
    tref = [orc.trace(to, td, mode=O.TRAVERSE_REFERENCE) for _, to, td in ties]
    for (t, to, td), r in zip(ties, tref):
        assert helpers.exclude_degenerate(td).all()
        members = {m[0] for m in t["members"]}
        won = np.isin(r[0], list(members))
        assert won.sum() >= 100, (t["kind"], won.sum())
        # the oracle's winner is the earlier object, or the later triangle of a BVH holding the triangle more than once
        first = min(members)
        if t["kind"].startswith("mesh_dup"):
            assert np.all(r[1][won] == len(t["members"]) - 1), t["kind"]
        else:
            assert np.all(r[0][won] == first), t["kind"]
    for f in FILTERS:
        g = hs.trace(o, d, bvh_filter=f)
        eq = same_hits(g, ref)
        assert eq[ok].all(), (f, np.flatnonzero(~eq & ok)[:5])
        assert (~eq & ~ok).sum() <= max(2, int(1e-4 * len(o)))
        for (t, to, td), r in zip(ties, tref):
            eq = same_hits(hs.trace(to, td, bvh_filter=f), r)
            assert eq.all(), (f, t["kind"], np.flatnonzero(~eq)[:5])


def check_render(c, hs, orc, **kw):
    g = hs.render((0, W, 0, H), H, W, spp=SPP, want_photons=True, **kw)
    okw = dict(kw)
    if okw.pop("integrator", capi.INTEGRATOR_SIMPLE_RANDOM) == capi.INTEGRATOR_WHITTED:
        okw["integrator"] = O.WHITTED
    r = orc.render((0, W, 0, H), H, W, spp=SPP, want_photons=True, **okw)
    rtol = 1e-12 if c.lambertian else 1e-9
    diverged = photons_close(g["photons"], r["photons"], rtol, max_diverged=PHONG_DIVERGED if c.phong else 0)
    live = (g["photons"][..., 0] == r["photons"][..., 0]) & (r["photons"][..., 0] != 0)
    rel = np.abs(g["photons"][..., 1] - r["photons"][..., 1])[live] / np.maximum(np.abs(r["photons"][..., 1][live]), 1e-300)
    # the oracle's Whitted integrator counts no path ends
    counters = ("primary_rays", "bounce_rays", "shadow_rays") if "lights" in kw else COUNTERS
    # A path that follows CUDA's sin / cos instead of glibc's can also end with zero intensity on both sides (after a black
    # reflectance, or outside a sampled reflectance's range), where its photon cannot show the divergence.  In Phong scenes
    # the ray counts may therefore differ by what up to PHONG_DIVERGED paths trace: max_depth bounces each, and a shadow ray
    # per light per level.  Primary rays and primary misses never depend on a sampled direction.
    paths = PHONG_DIVERGED if c.phong else 0
    slack = {"primary_rays": 0, "paths_missed": 0, "bounce_rays": paths * kw["max_depth"],
             "shadow_rays": paths * kw["max_depth"] * len(kw.get("lights", ())),
             "paths_escaped": paths, "paths_depth_limited": paths}
    for k in counters:
        assert abs(int(getattr(g["stats"], k)) - int(getattr(r["stats"], k))) <= slack[k], (k, getattr(g["stats"], k), getattr(r["stats"], k))
    if diverged == 0:
        np.testing.assert_allclose(g["colour_sum"], r["colour_sum"], rtol=1e-9, atol=1e-25)
    print("seed %d %s: max rel err %.2e over %d live samples, %d diverged" % (c.seed, kw, np.nanmax(rel, initial=0.0), live.sum(), diverged))
    return g, r


@pytest.mark.parametrize("seed", scene_content.SEEDS)
def test_simple_random_samples(seed):
    """Per-sample photons at recursion limits 3, 8 and 128 (the last finishes in k_tail, whose walk meets the tie sets
    through bounces) and biases 1e-7 and 1e-3."""
    c, hs, orc = content(seed)
    for depth in (3, 8, 128):
        for bias in (1e-7, 1e-3):
            g, r = check_render(c, hs, orc, max_depth=depth, bias=bias, seed=11 + seed)
            assert (r["photons"][..., 0] != 0).sum() > 1000
            if depth == 128:
                assert g["stats"].tail_launches >= 1


@pytest.mark.parametrize("seed", scene_content.SEEDS)
def test_whitted_samples(seed):
    """Whitted at recursion limits 0, 1 and 3 with the scene's lights (1 to 16, some below the horizon, spectra of every
    kind and length) and ambient (none, grey, sampled over part of the band): photons and shadow-ray counts."""
    c, hs, orc = content(seed)
    for depth, bias in ((0, 1e-7), (1, 1e-7), (3, 1e-7), (3, 1e-3)):
        g, r = check_render(c, hs, orc, max_depth=depth, bias=bias, seed=5, integrator=capi.INTEGRATOR_WHITTED,
                            lights=c.lights, ambient=c.ambient)
        assert r["stats"].shadow_rays > 0
        assert (r["photons"][..., 1] != 0).sum() > 1000


@pytest.mark.parametrize("seed", scene_content.SEEDS)
def test_upload_build_and_kernel_variants_identical(seed, monkeypatch):
    """The tree built inside vrj_scene_create renders the same samples as the host-built one; for all-Lambertian scenes,
    so do the general material kernels and the queue-entry walk (VRJ_MATERIAL_MASK=15, VRJ_RECORDS=0)."""
    c, hs, _ = content(seed)
    kw = dict(spp=2, max_depth=128, seed=3, want_photons=True)
    ref = hs.render((0, W, 0, H), H, W, **kw)
    envs = [{}]
    if c.lambertian:
        envs += [{"VRJ_MATERIAL_MASK": "15"}, {"VRJ_RECORDS": "0"}, {"VRJ_MATERIAL_MASK": "15", "VRJ_RECORDS": "0"}]
    for env in envs:
        for k in ("VRJ_MATERIAL_MASK", "VRJ_RECORDS"):
            monkeypatch.delenv(k, raising=False)
        for k, v in env.items():
            monkeypatch.setenv(k, v)          # read by vrj_scene_create
        for builder in ((False, "upload") if env else ("upload",)):
            g = V.build_scene(c.spec, device_builder=builder).render((0, W, 0, H), H, W, **kw)
            assert np.array_equal(g["photons"], ref["photons"]), (env, builder)
            assert np.array_equal(g["colour_sum"], ref["colour_sum"]), (env, builder)
            assert g["stats"].rays == ref["stats"].rays


def edge_on_rays(e, n, rng):
    """Origins exactly on the plane of `e`, directions with an exactly zero component along its normal."""
    axis, lo, hi = e["axis"], e["lo"], e["hi"]
    o = lo + rng.random((n, 3)) * (hi - lo)
    o[:, axis] = e["level"]
    d = rng.normal(size=(n, 3))
    d[:, axis] = 0.0
    # helpers.exclude_degenerate: the signed-largest component must be positive
    other = [a for a in range(3) if a != axis]
    d[:, other[0]] = np.abs(d[:, other[0]]) + 0.05
    return o, d


@pytest.mark.parametrize("seed", scene_content.SEEDS)
def test_edge_on_rays(seed):
    """Rays lying in the plane of axis-aligned flat-list triangles, of the flat floor mesh and of an axis plane.  All three
    edge functions of most in-plane triangle tests are zero with equal sign bits, so the depth is 0 * inf = NaN and its sign
    bit decides hit or miss: on x86-64 the NaN has it set and the ray misses, and the device has to agree (measured on a
    B200: it does, with no special case in triangle_test).  Hit ids and distances must equal the oracle's in all four
    filters, a NaN distance matching a NaN.  A ray in the plane of a plane object hits it at 0 / 0 = NaN:
    where that NaN then meets other hits, which one is kept depends on the order of the comparisons (DESIGN 3.2, deviation
    ii): the reference keeps the NaN as its list object's closest hit, so that list's finite hits behind it never compete
    with the other objects, while the device compares every analytic primitive on its own.  For those rays a difference is
    allowed only where one side's distance is NaN, or where the device's winner is in the plane's list object and the
    reference's is not."""
    c, hs, orc = content(seed)
    rng = np.random.default_rng(100 + seed)
    for e in c.edge_on:
        o, d = edge_on_rays(e, 4000, rng)
        assert helpers.exclude_degenerate(d).all()
        r = orc.trace(o, d, mode=O.TRAVERSE_REFERENCE)
        for f in FILTERS:
            g = hs.trace(o, d, bvh_filter=f)
            eq = same_hits(g, r)
            if e["kind"] == "plane":
                eq |= np.isnan(g[2]) | np.isnan(r[2]) | ((g[0] == e["object"]) & (r[0] != e["object"]))
            else:
                assert not np.isnan(r[2]).any()
            assert eq.all(), (e["kind"], f, np.flatnonzero(~eq)[:5], g[0][~eq][:5], r[0][~eq][:5], g[2][~eq][:5], r[2][~eq][:5])
