"""CPU checks of the generated scene content (scene_content.py): the fixed list of seeds covers every spectrum, material,
object, tie and light configuration the GPU parity tests of test_gpu_scene_content.py rely on.  Everything is read back
from the SceneSpecs themselves, not from what the generator says it built.  Also: a light spectrum longer than 64 samples
reaches the render parameters whole."""
from collections import Counter

import numpy as np
import pytest

import scene_content
import vanrijn_b200 as V
from vanrijn_b200 import capi
from vanrijn_b200.scenes import MAT_DIELECTRIC, MAT_LAMBERTIAN, MAT_PHONG, MAT_REFLECTIVE

LO, HI = scene_content.BAND
CONTENT = [scene_content.generate(s) for s in scene_content.SEEDS]


def rgb_branch(r, g, b):
    """The branch of rgb_basis_split (vrj_device.cuh) / spectrum.rs:81-165 a colour takes, 0..5."""
    if r <= g and r <= b:
        return 0 if g <= b else 1
    if g <= r and g < b:
        return 2 if r <= b else 3
    return 4 if r <= g else 5


def spectra_of(c, ids):
    return [c.spec.spectra[i] for i in ids]


def used_spectra(c):
    """(reflectance / eta spectra of the materials, spectra of the lights, the ambient spectrum or None)"""
    return ([c.spec.spectra[m.spectrum] for m in c.spec.materials], spectra_of(c, [s for _, s in c.lights]),
            c.spec.spectra[c.ambient] if c.ambient >= 0 else None)


def list_prims(c):
    return [(oi, pi, p) for oi, o in enumerate(c.spec.objects) if o[0] == "list" for pi, p in enumerate(o[1])]


def meshes(c):
    return [(oi, o) for oi, o in enumerate(c.spec.objects) if o[0] == "mesh"]


def test_the_same_seed_gives_the_same_scene():
    a, b = scene_content.generate(3), scene_content.generate(3)
    assert len(a.spec.objects) == len(b.spec.objects) and a.lights == b.lights
    for x, y in zip(a.spec.objects, b.spec.objects):
        if x[0] == "mesh":
            assert np.array_equal(x[1], y[1]) and np.array_equal(x[2], y[2]) and x[3] == y[3]


def test_scenes_are_small_enough_for_the_oracle():
    for c in CONTENT:
        assert sum(o[1].size // 9 for _, o in meshes(c)) <= 5000


def test_spectra_coverage():
    counts, ranges, branches, rgbs, grey = set(), set(), set(), set(), False
    for c in CONTENT:
        mats, lights, amb = used_spectra(c)
        for sp in mats + lights + ([amb] if amb else []):
            if sp[0] == "samples":
                counts.add(len(sp[3]))
                lo, hi = sp[1], sp[2]
                ranges.add("inside" if LO < lo and hi < HI else "enclosing" if lo < LO and hi > HI else
                           "overlapping" if (lo < LO < hi < HI) or (LO < lo < HI < hi) else "other")
                if lo == LO or hi == HI:
                    ranges.add("ends on %g" % (LO if lo == LO else HI))
                if lo == LO and hi == HI:
                    ranges.add("the band")
            elif sp[0] == "rgb":
                branches.add(rgb_branch(*sp[1]))
                rgbs.add(tuple(sp[1]))
            grey |= sp[0] == "grey"
    assert set(scene_content.SAMPLE_COUNTS) <= counts
    assert {"inside", "enclosing", "overlapping", "ends on 380", "ends on 740", "the band"} <= ranges
    assert branches == set(range(6))
    patterns = set()
    for r, g, b in rgbs:
        for name, hit in (("r=g=b", r == g == b), ("r=g<b", r == g < b), ("r=g>b", r == g > b), ("g=b>r", g == b > r),
                          ("g=b<r", g == b < r), ("r=b<g", r == b < g), ("r=b>g", r == b > g)):
            if hit:
                patterns.add(name)
    assert len(patterns) == 7, patterns
    assert grey


def test_material_coverage():
    kinds, smooth, etas = Counter(), [], set()
    for c in CONTENT:
        for m in c.spec.materials:
            kinds[m.kind] += 1
            if m.kind == MAT_PHONG:
                smooth.append(m.p2)
            if m.kind == MAT_DIELECTRIC:
                sp = c.spec.spectra[m.spectrum]
                if sp[0] == "diamond":
                    etas.add("diamond")
                    continue
                assert sp[0] == "samples" and sp[1] <= LO and sp[2] >= HI, sp[:3]   # eta covers every wavelength drawn
                v = np.asarray(sp[3])
                etas.add("constant 1.5" if np.all(v == 1.5) else "below 1" if v.max() < 1.0 else
                         "dispersive around 1.5" if abs(v.mean() - 1.5) < 0.1 and v.min() < v.max() else "other")
        lam = all(m.kind == MAT_LAMBERTIAN for m in c.spec.materials)
        assert lam == c.lambertian and c.phong == any(m.kind == MAT_PHONG for m in c.spec.materials)
    assert all(kinds[k] >= 4 for k in (MAT_LAMBERTIAN, MAT_PHONG, MAT_REFLECTIVE, MAT_DIELECTRIC))
    assert min(smooth) == 1.0 and max(smooth) == 200.0 and len(set(smooth)) >= 5
    assert {"constant 1.5", "dispersive around 1.5", "below 1"} <= etas
    assert sum(c.lambertian for c in CONTENT) >= 2 and sum(not c.lambertian for c in CONTENT) >= 2


def test_object_coverage():
    radii, overlap, around, normals, random_planes = [], 0, 0, set(), 0
    flipped = nonunit = 0
    mesh_sizes, flat_floor, list_counts, mesh_between = set(), 0, set(), 0
    for c in CONTENT:
        cam = np.asarray(c.spec.camera)
        spheres = [(np.asarray(p[1]), p[2]) for _, _, p in list_prims(c) if p[0] == "sphere"]
        for i, (ci, ri) in enumerate(spheres):
            radii.append(ri)
            around += np.linalg.norm(ci - cam) < ri
            overlap += any(0 < np.linalg.norm(ci - cj) < ri + rj for cj, rj in spheres[i + 1:])
        for _, _, p in list_prims(c):
            if p[0] == "plane":
                n = np.asarray(p[1])
                assert abs(np.linalg.norm(n) - 1.0) < 1e-12
                if np.count_nonzero(n) == 1:
                    normals.add(tuple(n))
                else:
                    random_planes += 1
            if p[0] == "triangle":
                t = np.asarray(p[1]).reshape(3, 3)
                g = np.cross(t[1] - t[0], t[2] - t[0])
                nv = np.asarray(p[2]).reshape(3, 3)
                lens = np.linalg.norm(nv, axis=1)
                assert lens.min() > 0
                flipped += np.all(nv @ g < 0)
                nonunit += np.all(np.abs(lens - 1.0) > 0.1)
        for oi, o in meshes(c):
            n = o[1].size // 9
            mesh_sizes.add(n if n <= 3 else "hundreds" if n < 1000 else "thousands")
            flat_floor += n >= 100 and np.all(o[1].reshape(-1, 3)[:, 1] == scene_content.FLOOR_Y)
        kinds = [o[0] for o in c.spec.objects]
        lists = [i for i, k in enumerate(kinds) if k == "list"]
        list_counts.add(len(lists))
        mesh_between += any(k == "mesh" for k in kinds[lists[0]:lists[-1]])
    assert min(radii) <= 0.05 and max(radii) >= 5.0
    assert overlap >= 8 and around >= 2
    assert normals == {tuple(float(x) for x in v) for v in np.vstack([np.eye(3), -np.eye(3)])} and random_planes >= 8
    assert flipped >= 8 and nonunit >= 8
    assert {1, 2, 3, "hundreds", "thousands"} <= mesh_sizes and flat_floor == len(CONTENT)
    assert list_counts == {2, 3} and mesh_between == len(CONTENT)


def test_tie_coverage():
    """Exact-distance ties with different materials: a sphere in two list objects, a triangle in two meshes, a triangle
    as a flat-list triangle and in a mesh in both orders, the same triangle 2 and 50 times in one mesh."""
    found = Counter()
    for c in CONTENT:
        spheres, list_tris, mesh_tris = {}, {}, {}
        for oi, pi, p in list_prims(c):
            if p[0] == "sphere":
                spheres.setdefault((tuple(p[1]), p[2]), []).append((oi, p[3]))
            if p[0] == "triangle":
                list_tris.setdefault(np.asarray(p[1]).tobytes(), []).append((oi, p[3]))
        for oi, o in meshes(c):
            v, n = o[1].reshape(-1, 9), o[2].reshape(-1, 9)
            keys = Counter(t.tobytes() for t in v)
            for key, cnt in keys.items():
                mesh_tris.setdefault(key, []).append((oi, o[3]))
                if cnt in (2, 50):
                    same = [i for i in range(len(v)) if v[i].tobytes() == key]
                    # copies inside one mesh share its material: they differ in their vertex normals
                    assert len({n[i].tobytes() for i in same}) == cnt
                    found["mesh holds a triangle %d times" % cnt] += 1
        for where in spheres.values():
            if len({o for o, _ in where}) >= 2 and len({m for _, m in where}) >= 2:
                found["sphere in two lists"] += 1
        for key, where in mesh_tris.items():
            if len(where) >= 2 and len({m for _, m in where}) >= 2:
                found["triangle in two meshes"] += 1
            for lo, lm in list_tris.get(key, []):
                for mo, mm in where:
                    if lm != mm:
                        found["list triangle before mesh" if lo < mo else "mesh before list triangle"] += 1
    for k in ("sphere in two lists", "triangle in two meshes", "list triangle before mesh", "mesh before list triangle",
              "mesh holds a triangle 2 times", "mesh holds a triangle 50 times"):
        assert found[k] >= len(CONTENT), (k, found[k])


def test_light_coverage():
    n_lights, lengths, below, kinds, long, ambient = set(), [], 0, set(), 0, set()
    for c in CONTENT:
        n_lights.add(len(c.lights))
        for d, sid in c.lights:
            lengths.append(np.linalg.norm(d))
            below += d[1] < 0
            sp = c.spec.spectra[sid]
            kinds.add(sp[0])
            long += sp[0] == "samples" and len(sp[3]) > 64
        if c.ambient < 0:
            ambient.add("none")
        else:
            sp = c.spec.spectra[c.ambient]
            ambient.add("grey" if sp[0] == "grey" else "part of the band" if sp[0] == "samples" and LO < sp[1] and sp[2] < HI else "other")
    assert min(n_lights) == 1 and max(n_lights) == 16 and len(n_lights) >= 6
    assert min(lengths) == pytest.approx(0.1) and max(lengths) == pytest.approx(10.0)
    assert below >= 8 and long >= len(CONTENT)
    assert {"grey", "rgb", "samples"} <= kinds
    assert {"none", "grey", "part of the band"} <= ambient


def test_long_light_spectrum_reaches_the_render_parameters():
    """HostScene.spectrum_data hands the library every sample of a spectrum (it once read at most 64 of them but passed the
    full count, so stage_lights copied past the buffer): 200- and 65-sample light and ambient spectra arrive whole."""
    c = scene_content.generate(0)
    vals = np.linspace(0.1, 2.0, 200)
    s200 = c.spec.spectrum("samples", 300.0, 800.0, vals)
    s65 = c.spec.spectrum("samples", 380.0, 740.0, vals[:65] * 3)
    hs = V.build_scene(c.spec)
    for sid, want in ((s200, vals), (s65, vals[:65] * 3)):
        sd, keep = hs.spectrum_data(sid)
        assert sd.n_samples == len(want) and (sd.shortest_wavelength, sd.longest_wavelength) == c.spec.spectra[sid][1:3]
        assert np.array_equal(np.ctypeslib.as_array(sd.samples, (sd.n_samples,)), want)
    p, keep = hs.make_params(lights=[((0.0, 1.0, 0.0), s200), ((1.0, 1.0, 0.0), s65)], ambient=s200,
                             integrator=capi.INTEGRATOR_WHITTED)
    for sd, want in ((p.lights[0].spectrum, vals), (p.lights[1].spectrum, vals[:65] * 3), (p.ambient_light.contents, vals)):
        assert sd.n_samples == len(want)
        assert np.array_equal(np.ctypeslib.as_array(sd.samples, (sd.n_samples,)), want)
    # a grey spectrum (2 samples) and the 32-sample rgb basis still come back whole
    for sid, n in ((c.spec.spectrum("grey", 0.5), 2), (c.spec.spectrum("rgb", (0.1, 0.2, 0.3)), 32)):
        hs = V.build_scene(c.spec)
        assert hs.spectrum_data(sid)[0].n_samples == n
    with pytest.raises(capi.VrjError):
        hs.spectrum_data(len(c.spec.spectra))
