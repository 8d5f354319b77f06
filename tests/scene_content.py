"""Seeded scene content for the parity tests: generate(seed) builds a SceneSpec (plus Whitted lights and ambient) that
exercises what the fixed scenes of vanrijn_b200.scenes never do -- sampled spectra of many lengths and ranges, every
branch of the rgb basis split, all four materials, spheres / planes / flat-list triangles / meshes of 1 to thousands of
triangles in several list objects, exact-distance ties between and inside objects, and 1 to 16 lights.

Every scene lays out the same skeleton at seed-dependent scales and materials:
  * a row of tie sets in front of the camera (z = 2), each set of identical geometry with DIFFERENT materials (or, inside
    one mesh, different vertex normals), so that a wrong winner changes the radiance as well as the hit id;
  * axis-aligned flat-list triangles and a flat floor mesh whose planes hold exact binary fractions, for edge-on rays;
  * random spheres, meshes and planes behind the tie row (z >= 4), and in some scenes a sphere around the camera.
The content stays small enough for the CPU oracle (a few thousand triangles).  SEEDS is the fixed list the tests use;
tests/test_scene_content_cpu.py checks that it covers every item above."""
from dataclasses import dataclass, field

import numpy as np

from vanrijn_b200 import scenes
from vanrijn_b200.scenes import MAT_DIELECTRIC, MAT_LAMBERTIAN, MAT_PHONG, MAT_REFLECTIVE, SceneSpec

SEEDS = tuple(range(8))

# photon.rs:18-24 draws wavelengths in [380, 740) nm
BAND = (380.0, 740.0)
SAMPLE_COUNTS = (2, 3, 7, 33, 65, 200)
# inside, overlapping below / above, enclosing, ending on 380, ending on 740, exactly the band
RANGES = ((450.0, 650.0), (300.0, 500.0), (600.0, 800.0), (300.0, 800.0), (380.0, 600.0), (500.0, 740.0), (380.0, 740.0))
# every branch of spectrum.rs:81-165 (rgb_basis_split), with and without ties between channels
RGBS = ((0.2, 0.5, 0.8), (0.2, 0.8, 0.5), (0.5, 0.2, 0.8), (0.8, 0.2, 0.5), (0.5, 0.8, 0.2), (0.8, 0.5, 0.2),
        (0.4, 0.4, 0.4), (0.3, 0.3, 0.7), (0.6, 0.6, 0.2), (0.2, 0.6, 0.6), (0.7, 0.3, 0.3), (0.3, 0.7, 0.3), (0.6, 0.2, 0.6),
        (0.0, 0.0, 0.0), (1.0, 1.0, 1.0))
CAMERA = (0.0, 0.5, -8.0)
# planes of the axis-aligned flat-list triangles (exact in binary), the flat floor mesh, and the axis planes: (axis, level)
FLAT_TRIANGLE_PLANES = ((1, 1.25), (0, -5.5), (2, 6.5))
FLOOR_Y = -2.5
AXIS_PLANES = (((1.0, 0.0, 0.0), 7.0), ((-1.0, 0.0, 0.0), 7.0), ((0.0, 1.0, 0.0), -4.0), ((0.0, -1.0, 0.0), -6.0),
               ((0.0, 0.0, 1.0), 25.0), ((0.0, 0.0, -1.0), 25.0))


@dataclass
class Content:
    seed: int
    spec: SceneSpec
    lights: list                 # Whitted lights: [(direction, spectrum id)]
    ambient: int                 # spectrum id, -1: none
    lambertian: bool             # every material is Lambertian (the 1e-12 bar; the Lambertian-only kernels)
    phong: bool                  # some material is Phong (libm sin / cos feed the sampled direction)
    # tie sets: dict(kind, members=[(object, primitive)], and tri=(3, 3) vertices of the shared triangle, or centre and
    # radius of the shared sphere)
    ties: list = field(default_factory=list)
    # edge-on targets: dict(kind "list_triangle" / "floor_mesh" / "plane", axis, level, lo=(3,), hi=(3,)) -- origins on the
    # plane `axis` = level inside [lo, hi] on the other two axes; a plane's also names its list object (`object`)
    edge_on: list = field(default_factory=list)


def _sampled(rng, n, rng_range, lo=0.05, hi=0.95):
    return ("samples", float(rng_range[0]), float(rng_range[1]), rng.uniform(lo, hi, n))


def _tri_normals(rng, geometric, flip, count=3):
    """`count` vertex normals in the hemisphere of +-geometric, of length 0.3 to 3 (never zero, never unit)."""
    g = np.asarray(geometric, np.float64)
    g = g / np.linalg.norm(g)
    s = -1.0 if flip else 1.0
    out = []
    for _ in range(count):
        v = s * g + rng.normal(size=3) * 0.3
        if np.dot(v, s * g) <= 0.1:
            v = s * g
        v = v / np.linalg.norm(v) * rng.choice([0.3, 0.7, 1.9, 3.0])
        out.append(v)
    return np.concatenate(out)


def _geo_normal(tri):
    t = np.asarray(tri).reshape(3, 3)
    return np.cross(t[1] - t[0], t[2] - t[0])


def _mesh(tris, normals, material):
    return ("mesh", np.ascontiguousarray(np.asarray(tris, np.float64).reshape(-1, 9)),
            np.ascontiguousarray(np.asarray(normals, np.float64).reshape(-1, 9)), material)


def _tie_triangle(centre, size, rng):
    """A triangle around `centre` tilted toward the camera; its vertices are binary64 values used verbatim by every copy."""
    c = np.asarray(centre, np.float64)
    a = rng.uniform(0, 2 * np.pi)
    pts = [c + size * np.array([np.cos(a + k * 2.1), np.sin(a + k * 2.1), 0.25 * np.cos(a + k)]) for k in range(3)]
    return np.concatenate(pts)


def generate(seed):
    rng = np.random.default_rng(7919 + seed)
    s = SceneSpec(camera=CAMERA)
    lambertian = seed % 3 == 0
    k = seed

    # ---- spectra: sampled (two lengths, two ranges per scene, rotating), rgb (two branches per scene), grey
    sampled = [s.spectrum(*_sampled(rng, SAMPLE_COUNTS[(k + j) % 6], RANGES[(k + 3 * j) % 7])) for j in range(3)]
    rgbs = [s.spectrum("rgb", RGBS[(2 * k + j) % len(RGBS)]) for j in range(2)]
    grey = s.spectrum("grey", float(rng.uniform(0.3, 0.9)))
    reflectances = sampled + rgbs + [grey]

    # ---- materials
    def lam(i):
        return s.material(MAT_LAMBERTIAN, reflectances[i % len(reflectances)], rng.uniform(0.05, 1.0))

    mats = [lam(i) for i in range(len(reflectances))]
    if not lambertian:
        if k % 4 != 3:
            # one mixed scene without Phong keeps mirrors, glass and ties under the exact ray counts
            smooth = (1.0, 200.0, 5.0, 40.0, 12.0)[k % 5]
            mats.append(s.material(MAT_PHONG, reflectances[(k + 1) % len(reflectances)], rng.uniform(0.1, 0.6), rng.uniform(0.1, 0.6), smooth))
            mats.append(s.material(MAT_PHONG, reflectances[(k + 4) % len(reflectances)], 0.3, 0.5, (200.0, 1.0, 80.0)[k % 3]))
        mirror = len(mats) + 1
        mats.append(s.material(MAT_REFLECTIVE, reflectances[(k + 2) % len(reflectances)], rng.uniform(0.0, 0.2), rng.uniform(0.5, 1.0)))
        mats.append(s.material(MAT_REFLECTIVE, reflectances[(k + 5) % len(reflectances)], 0.01, 0.99))
        # eta spectra cover the whole band: constant 1.5, dispersive around 1.5, below 1 (total internal reflection outside)
        etas = [s.spectrum("samples", 370.0, 750.0, np.array([1.5, 1.5])),
                s.spectrum("samples", BAND[0], BAND[1], np.linspace(1.56, 1.44, SAMPLE_COUNTS[(k + 2) % 6])),
                s.spectrum("samples", 300.0, 800.0, rng.uniform(0.6, 0.9, 5))]
        glass = [s.material(MAT_DIELECTRIC, e) for e in etas]
        mats += glass
        if k % 4 == 1:
            mats.append(s.dielectric_diamond())
    pick = lambda: int(rng.integers(len(mats)))  # noqa: E731
    # two materials guaranteed to differ, for the members of a tie set
    def two():
        a = pick()
        b = (a + 1 + int(rng.integers(len(mats) - 1))) % len(mats)
        return a, b

    objects = s.objects
    ties, edge_on = [], []
    scale = (0.5, 1.0, 2.0)[k % 3]

    # ---- list object 0: random spheres (overlapping pairs), random and axis-aligned flat-list triangles, tie members
    l0 = []
    for _ in range(4):
        c = np.array([rng.uniform(-6, 6), rng.uniform(-2, 4), rng.uniform(6, 14)])
        r = float(np.exp(rng.uniform(np.log(0.05), np.log(2.0))))
        l0.append(("sphere", tuple(c), r, pick()))
        l0.append(("sphere", tuple(c + rng.normal(size=3) * r * 0.5), r * rng.uniform(0.5, 1.2), pick()))
    # a large sphere behind everything; a mirror where the scene has one, so bounces come back to the tie row
    mirror = mats[mirror] if not lambertian else pick()
    l0.append(("sphere", (rng.uniform(-6, 6), rng.uniform(0, 4), 18.0), 5.0, mirror))
    for _ in range(3):
        c = np.array([rng.uniform(-6, 6), rng.uniform(-1, 5), rng.uniform(5, 12)])
        tri = np.concatenate([c + rng.normal(size=3) * scale for _ in range(3)])
        l0.append(("triangle", tri, _tri_normals(rng, _geo_normal(tri), bool(rng.integers(2))), pick()))
    for axis, level in FLAT_TRIANGLE_PLANES:
        # an axis-aligned triangle: the coordinate `axis` of every vertex is exactly `level`
        centre = {1: (4.5, 1.25, 3.0), 0: (-5.5, 1.0, 4.0), 2: (0.5, 3.5, 6.5)}[axis]
        v = []
        for j in range(3):
            p = np.array(centre, np.float64) + rng.normal(size=3) * 1.2
            p[axis] = level
            v.append(p)
        tri = np.concatenate(v)
        g = np.zeros(3)
        g[axis] = 1.0
        l0.append(("triangle", tri, _tri_normals(rng, g, axis != 1), pick()))
        lo, hi = np.min(v, 0) - 0.5, np.max(v, 0) + 0.5
        lo[axis] = hi[axis] = level
        edge_on.append(dict(kind="list_triangle", axis=axis, level=level, lo=lo, hi=hi))
    # tie: one sphere in list objects 0 and 1
    ms = two()
    sph_c, sph_r = np.array([-3.0, 0.0, 2.0]), 0.6 * min(scale, 1.0)
    l0.append(("sphere", tuple(sph_c), sph_r, ms[0]))
    sphere_members = [(0, len(l0) - 1)]
    # tie: a triangle in list object 0 and, after it, in a mesh
    mc = two()
    tri_c = _tie_triangle((1.0, 0.0, 2.0), 0.7, rng)
    l0.append(("triangle", tri_c, _tri_normals(rng, _geo_normal(tri_c), False), mc[0]))
    list_then_mesh = [(0, len(l0) - 1)]
    objects.append(("list", l0))

    objects.append(_mesh(tri_c, _tri_normals(rng, _geo_normal(tri_c), True), mc[1]))
    list_then_mesh.append((len(objects) - 1, 0))
    ties.append(dict(kind="list_then_mesh", members=list_then_mesh, tri=tri_c.reshape(3, 3)))

    # tie: a triangle in a mesh and, after it, in list object 1 (the mesh is written first)
    md = two()
    tri_d = _tie_triangle((3.0, 0.0, 2.0), 0.7, rng)
    other = tri_d + np.tile(rng.normal(size=3) * 0.5 + np.array([0.0, 0.0, 2.0]), 3)
    objects.append(_mesh(np.concatenate([other, tri_d]), np.concatenate([_tri_normals(rng, _geo_normal(other), False),
                                                                         _tri_normals(rng, _geo_normal(tri_d), False)]), md[0]))
    mesh_then_list = [(len(objects) - 1, 1)]

    # ---- list object 1: the second copy of the tie sphere and the tie triangle, planes, more spheres
    l1 = [("sphere", tuple(sph_c), sph_r, ms[1])]
    sphere_members.append((len(objects), 0))
    l1.append(("triangle", tri_d, _tri_normals(rng, _geo_normal(tri_d), True), md[1]))
    mesh_then_list.append((len(objects), 1))
    an, ad = AXIS_PLANES[k % 6]
    l1.append(("plane", an, ad, pick()))
    axis = int(np.argmax(np.abs(an)))
    level = ad * an[axis]
    lo, hi = np.array([-6.0, -3.0, -2.0]), np.array([6.0, 5.0, 14.0])
    lo[axis] = hi[axis] = level
    edge_on.append(dict(kind="plane", axis=axis, level=level, lo=lo, hi=hi, object=len(objects)))
    n = rng.normal(size=3)
    n /= np.linalg.norm(n)
    l1.append(("plane", tuple(n), float(np.dot(n, np.array([0.0, 0.0, 4.0]) + 11.0 * n)), pick()))
    if not lambertian and k % 2 == 0:
        # a glass sphere around the camera: every camera ray leaves through it
        l1.append(("sphere", (0.3, 0.2, -8.5), 3.0, glass[k % 3]))
    objects.append(("list", l1))
    ties.append(dict(kind="sphere_in_two_lists", members=sphere_members, centre=sph_c, radius=sph_r))
    ties.append(dict(kind="mesh_then_list", members=mesh_then_list, tri=tri_d.reshape(3, 3)))

    # ---- meshes of 1, 2 and 3 triangles, the same triangle in two meshes, the same triangle 2 and 50 times in one mesh
    mb = two()
    tri_b = _tie_triangle((-1.0, 0.0, 2.0), 0.7, rng)
    objects.append(_mesh(tri_b, _tri_normals(rng, _geo_normal(tri_b), False), mb[0]))
    two_meshes = [(len(objects) - 1, 0)]
    extra = tri_b + np.tile(np.array([0.3, 1.0, 1.5]), 3)
    objects.append(_mesh(np.concatenate([extra, tri_b]), np.concatenate([_tri_normals(rng, _geo_normal(extra), True),
                                                                         _tri_normals(rng, _geo_normal(tri_b), True)]), mb[1]))
    two_meshes.append((len(objects) - 1, 1))
    ties.append(dict(kind="two_meshes", members=two_meshes, tri=tri_b.reshape(3, 3)))

    c3 = np.array([rng.uniform(-5, 5), rng.uniform(2, 4), rng.uniform(5, 9)])
    t3 = np.concatenate([np.concatenate([c3 + rng.normal(size=3) * scale * 0.5 for _ in range(3)]) for _ in range(3)])
    objects.append(_mesh(t3, np.concatenate([_tri_normals(rng, _geo_normal(t3[9 * j:9 * j + 9]), j == 1) for j in range(3)]), pick()))

    for copies, centre in ((2, (-2.0, 2.0, 2.0)), (50, (2.0, 2.0, 2.0))):
        tri = _tie_triangle(centre, 0.8, rng)
        g = _geo_normal(tri)
        nrm = np.concatenate([_tri_normals(rng, g, j % 3 == 1) for j in range(copies)])
        objects.append(_mesh(np.tile(tri, copies), nrm, pick()))
        ties.append(dict(kind="mesh_dup%d" % copies, members=[(len(objects) - 1, j) for j in range(copies)], tri=tri.reshape(3, 3)))

    # ---- a displaced icosphere (320 triangles) at this scene's scale, and a flat floor grid (3200 triangles)
    pos, nrm, faces = scenes.bunny_proxy(2, radius=0.8 * scale, centre=(rng.uniform(-4, 4), rng.uniform(-1, 2), 9.0))
    v, nn = scenes.mesh_arrays(pos, nrm, faces)
    objects.append(("mesh", v, nn * rng.choice([1.0, -2.0]), pick()))
    # grid lines off the binary fractions the camera rays are made of: a ray through a shared edge can slip between the two
    # triangles, and the reference's exact box test then decides which object it reports (no near-edge exclusion sees it)
    g = 40
    xs = np.linspace(-20.0, 20.0, g + 1) + 0.3183098861837907
    zs = np.linspace(-6.0, 26.0, g + 1) + 0.1591549430918953
    quads = []
    for i in range(g):
        for j in range(g):
            a, b = (xs[i], zs[j]), (xs[i + 1], zs[j])
            c, d = (xs[i + 1], zs[j + 1]), (xs[i], zs[j + 1])
            quads.append([a[0], FLOOR_Y, a[1], b[0], FLOOR_Y, b[1], c[0], FLOOR_Y, c[1]])
            quads.append([a[0], FLOOR_Y, a[1], c[0], FLOOR_Y, c[1], d[0], FLOOR_Y, d[1]])
    floor = np.array(quads)
    objects.append(_mesh(floor, np.tile([0.0, 1.0, 0.0], (len(floor), 3)) * (1.0 + 0.5 * (k % 2)), pick()))
    edge_on.append(dict(kind="floor_mesh", axis=1, level=FLOOR_Y, lo=np.array([-18.0, FLOOR_Y, -4.0]), hi=np.array([18.0, FLOOR_Y, 24.0])))

    # ---- list object 2 in some scenes: spheres of the extreme radii
    if k % 2 == 1:
        objects.append(("list", [("sphere", (rng.uniform(-3, 3), rng.uniform(-1, 1), 4.5), 0.05, pick()),
                                 ("sphere", (rng.uniform(-6, 6), 1.0, 12.0), 2.5, pick())]))

    # ---- Whitted: 1 to 16 lights of every spectrum kind, directions of length 0.1 to 10, some below the horizon
    n_lights = 1 + (5 * k) % 16
    kinds = [lambda j: s.spectrum("grey", float(rng.uniform(0.2, 2.0))),
             lambda j: s.spectrum("rgb", RGBS[(k + j) % len(RGBS)]),
             lambda j: s.spectrum(*_sampled(rng, SAMPLE_COUNTS[(k + j) % 6], RANGES[(k + 2 * j) % 7], 0.1, 2.0))]
    lights = []
    for j in range(n_lights):
        d = rng.normal(size=3)
        if j == 0:
            d[1] = abs(d[1]) + 0.5
        elif j % 3 == 2:
            d[1] = -abs(d[1]) - 0.1       # below the horizon
        length = (0.1, 10.0)[j % 2] if j < 2 else float(np.exp(rng.uniform(np.log(0.1), np.log(10.0))))
        lights.append((tuple(d / np.linalg.norm(d) * length), kinds[(j + k) % 3](j)))
    # a light with more than 64 samples in every scene
    lights[-1] = (lights[-1][0], s.spectrum(*_sampled(rng, (65, 200)[k % 2], RANGES[k % 7], 0.1, 2.0)))
    ambient = (-1, s.spectrum("grey", 0.05), s.spectrum("samples", 450.0, 650.0, rng.uniform(0.01, 0.1, 7)))[k % 3]

    phong = any(m.kind == MAT_PHONG for m in s.materials)
    return Content(seed, s, lights, ambient, lambertian, phong, ties, edge_on)
