"""Scene descriptions for the configurations of BASELINE.json / SURVEY.md section 8(d).

A SceneSpec is a neutral, plain-data description (camera, spectra, materials, objects in
`Scene.objects` order).  The product turns it into host-builder calls
(vanrijn_b200.host.build_scene); the tests additionally hand the same spec to the oracle.

Also holds the deterministic bunny proxy: /root/reference/test_data/stanford_bunny.obj is
a Git-LFS pointer in the reference snapshot, so until the real 4.86 MB file is dropped in
(path given by $VANRIJN_BUNNY_OBJ) every "bunny" configuration uses the displaced
icosphere of SURVEY.md 8(d): 6 subdivisions = 81 920 triangles / 40 962 vertices.
"""
import atexit
import os
import shutil
import tempfile
from dataclasses import dataclass, field

import numpy as np

MAT_LAMBERTIAN, MAT_PHONG, MAT_REFLECTIVE, MAT_DIELECTRIC = 0, 1, 2, 3

# colour/colour_rgb.rs:17-35
NAMED = {"Yellow": (1.0, 1.0, 0.0), "Green": (0.0, 0.5, 0.0), "Blue": (0.0, 0.0, 1.0), "Red": (1.0, 0.0, 0.0)}


@dataclass
class Mat:
    kind: int
    spectrum: int
    p0: float = 0.0
    p1: float = 0.0
    p2: float = 0.0


@dataclass
class SceneSpec:
    camera: tuple = (0.0, 0.0, 0.0)
    spectra: list = field(default_factory=list)
    materials: list = field(default_factory=list)
    objects: list = field(default_factory=list)

    def spectrum(self, *desc):
        self.spectra.append(tuple(desc))
        return len(self.spectra) - 1

    def material(self, kind, spectrum, p0=0.0, p1=0.0, p2=0.0):
        self.materials.append(Mat(kind, spectrum, float(p0), float(p1), float(p2)))
        return len(self.materials) - 1

    def lambertian_rgb(self, rgb, diffuse):
        return self.material(MAT_LAMBERTIAN, self.spectrum("rgb", tuple(rgb)), diffuse)

    def reflective_rgb(self, rgb, diffuse, reflection):
        return self.material(MAT_REFLECTIVE, self.spectrum("rgb", tuple(rgb)), diffuse, reflection)

    def phong_rgb(self, rgb, diffuse, specular, smoothness):
        return self.material(MAT_PHONG, self.spectrum("rgb", tuple(rgb)), diffuse, specular, smoothness)

    def dielectric_diamond(self):
        return self.material(MAT_DIELECTRIC, self.spectrum("diamond"))


# ----------------------------------------------------------------------------- proxy mesh
def icosphere(subdivisions):
    """Unit icosphere: (vertices (V,3) f64, faces (F,3) int64). Deterministic."""
    t = (1.0 + 5.0 ** 0.5) / 2.0
    v = np.array([[-1, t, 0], [1, t, 0], [-1, -t, 0], [1, -t, 0], [0, -1, t], [0, 1, t], [0, -1, -t], [0, 1, -t],
                  [t, 0, -1], [t, 0, 1], [-t, 0, -1], [-t, 0, 1]], dtype=np.float64)
    v /= np.linalg.norm(v, axis=1, keepdims=True)
    f = np.array([[0, 11, 5], [0, 5, 1], [0, 1, 7], [0, 7, 10], [0, 10, 11], [1, 5, 9], [5, 11, 4], [11, 10, 2],
                  [10, 7, 6], [7, 1, 8], [3, 9, 4], [3, 4, 2], [3, 2, 6], [3, 6, 8], [3, 8, 9], [4, 9, 5], [2, 4, 11],
                  [6, 2, 10], [8, 6, 7], [9, 8, 1]], dtype=np.int64)
    for _ in range(subdivisions):
        nv = len(v)
        edges = np.concatenate([f[:, [0, 1]], f[:, [1, 2]], f[:, [2, 0]]], axis=0)
        edges.sort(axis=1)
        key = edges[:, 0] * nv + edges[:, 1]
        uniq, inverse = np.unique(key, return_inverse=True)
        a, b = uniq // nv, uniq % nv
        mid = v[a] + v[b]
        mid /= np.linalg.norm(mid, axis=1, keepdims=True)
        v = np.concatenate([v, mid], axis=0)
        nf = len(f)
        m01, m12, m20 = nv + inverse[:nf], nv + inverse[nf:2 * nf], nv + inverse[2 * nf:]
        f = np.concatenate([np.stack([f[:, 0], m01, m20], 1), np.stack([f[:, 1], m12, m01], 1),
                            np.stack([f[:, 2], m20, m12], 1), np.stack([m01, m12, m20], 1)], axis=0)
    return v, f


def bunny_proxy(subdivisions=6, radius=1.5, centre=(0.0, -0.5, 0.0)):
    """Displaced icosphere (SURVEY.md 8d): r(u) = radius*(1 + 0.15 sin(3x) sin(5y) sin(4z)) with
    (x,y,z) = radius*u; smooth normals = normalised gradient of the implicit surface.
    Returns (positions (V,3) f32, normals (V,3) f32, faces (F,3) int64)."""
    u, f = icosphere(subdivisions)
    q = radius * u
    sx, sy, sz = np.sin(3 * q[:, 0]), np.sin(5 * q[:, 1]), np.sin(4 * q[:, 2])
    cx, cy, cz = np.cos(3 * q[:, 0]), np.cos(5 * q[:, 1]), np.cos(4 * q[:, 2])
    g = 1.0 + 0.15 * sx * sy * sz
    pos = u * (radius * g)[:, None]
    grad_g = 0.15 * np.stack([3 * cx * sy * sz, 5 * sx * cy * sz, 4 * sx * sy * cz], axis=1)
    tangential = grad_g - u * np.sum(grad_g * u, axis=1, keepdims=True)
    n = u - (radius * radius / (radius * g))[:, None] * tangential
    n /= np.linalg.norm(n, axis=1, keepdims=True)
    pos = pos + np.asarray(centre, dtype=np.float64)[None, :]
    return pos.astype(np.float32), n.astype(np.float32), f


def write_obj(path, pos, nrm, faces):
    """`v`, `vn`, `f a//a` text, floats printed so that an f32 parse reproduces them exactly."""
    with open(path, "w") as fh:
        fh.write("# vanrijn-b200 bunny proxy: displaced icosphere (not the Stanford bunny)\n")
        np.savetxt(fh, pos, fmt="v %.9g %.9g %.9g")
        np.savetxt(fh, nrm, fmt="vn %.9g %.9g %.9g")
        idx = faces + 1
        np.savetxt(fh, np.stack([idx[:, 0], idx[:, 0], idx[:, 1], idx[:, 1], idx[:, 2], idx[:, 2]], 1),
                   fmt="f %d//%d %d//%d %d//%d")


_MESH_DIR = None


def _mesh_dir():
    """A temporary directory of this process for generated meshes, removed at exit: the source tree may be read-only."""
    global _MESH_DIR
    if _MESH_DIR is None:
        _MESH_DIR = tempfile.mkdtemp(prefix="vanrijn_b200_meshes_")
        atexit.register(shutil.rmtree, _MESH_DIR, True)
    return _MESH_DIR


def bunny_obj_path(cache_dir=None, subdivisions=6):
    """Path of the bunny OBJ: the real file when $VANRIJN_BUNNY_OBJ points at one, else the proxy
    (generated once into cache_dir, by default a temporary directory of this process)."""
    real = os.environ.get("VANRIJN_BUNNY_OBJ")
    if real and os.path.exists(real) and os.path.getsize(real) > 1000:
        return real, "stanford_bunny"
    cache_dir = cache_dir or _mesh_dir()
    os.makedirs(cache_dir, exist_ok=True)
    path = os.path.join(cache_dir, "bunny_proxy_s%d.obj" % subdivisions)
    if not os.path.exists(path):
        tmp = path + ".tmp%d" % os.getpid()
        write_obj(tmp, *bunny_proxy(subdivisions))
        os.replace(tmp, path)
    return path, "bunny_proxy_%dtri" % (20 * 4 ** subdivisions)


def mesh_arrays(pos, nrm, faces):
    """(F,9) f64 vertex and normal arrays, as mesh.rs widens f32 -> f64."""
    p = pos.astype(np.float64)[faces].reshape(-1, 9)
    n = nrm.astype(np.float64)[faces].reshape(-1, 9)
    return np.ascontiguousarray(p), np.ascontiguousarray(n)


# ----------------------------------------------------------------------------- configs
CAMERA = (-2.0, 1.0, -5.0)  # main.rs:139, benches/simple_scene.rs:24


def _add_bunny(spec, material, subdivisions, obj=True):
    if obj:
        path, name = bunny_obj_path(subdivisions=subdivisions)
        spec.objects.append(("obj", path, material))
        return name
    v, n = mesh_arrays(*bunny_proxy(subdivisions))
    spec.objects.append(("mesh", v, n, material))
    return "bunny_proxy_%dtri" % len(v)


def scene_bench(subdivisions=6, obj=True):
    """C1a -- benches/simple_scene.rs:16-37 (with the Spectrum conversion the stale bench lacks):
    one object, the bunny BVH, ReflectiveMaterial(Yellow, 0.05, 0.9)."""
    s = SceneSpec(camera=CAMERA)
    m = s.reflective_rgb(NAMED["Yellow"], 0.05, 0.9)
    _add_bunny(s, m, subdivisions, obj)
    return s


def scene_main(subdivisions=6, obj=True, variant="lambertian"):
    """C1b -- src/main.rs:123-189: objects[0] = [plane, 3 spheres], objects[1] = bunny BVH.
    variant "mixed" is C5 (mirror sphere, diamond sphere, reflective bunny; main.rs:170-171,182-183)."""
    s = SceneSpec(camera=CAMERA)
    ground = s.lambertian_rgb((0.55, 0.27, 0.04), 0.1)
    green = s.lambertian_rgb(NAMED["Green"], 0.1)
    if variant == "mixed":
        blue = s.reflective_rgb(NAMED["Blue"], 0.01, 0.99)
        red = s.dielectric_diamond()
        bunny = s.reflective_rgb(NAMED["Yellow"], 0.05, 0.9)
    else:
        blue = s.lambertian_rgb(NAMED["Blue"], 0.1)
        red = s.lambertian_rgb(NAMED["Red"], 0.05)
        bunny = s.lambertian_rgb(NAMED["Yellow"], 0.05)
    s.objects.append(("list", [("plane", (0.0, 1.0, 0.0), -2.0, ground),
                               ("sphere", (-6.25, -0.5, 1.0), 1.0, green),
                               ("sphere", (-4.25, -0.5, 2.0), 1.0, blue),
                               ("sphere", (-5.0, 1.5, 1.0), 1.0, red)]))
    _add_bunny(s, bunny, subdivisions, obj)
    return s


def scene_direct(subdivisions=6, obj=True, reflective=False):
    """C2 -- bunny BVH only; Whitted, one DirectionalLight (1,1,-1) grey(1), ambient grey(0.05)."""
    s = SceneSpec(camera=CAMERA)
    m = s.reflective_rgb(NAMED["Yellow"], 0.05, 0.9) if reflective else s.lambertian_rgb(NAMED["Yellow"], 0.05)
    _add_bunny(s, m, subdivisions, obj)
    light = s.spectrum("grey", 1.0)
    ambient = s.spectrum("grey", 0.05)
    return s, [((1.0, 1.0, -1.0), light)], ambient


def scene_grid(copies=11, subdivisions=6, pitch=4.0):
    """C4 -- copies x copies bunny copies on an XZ grid + ground plane; camera (-2, 6, -12)."""
    s = SceneSpec(camera=(-2.0, 6.0, -12.0))
    ground = s.lambertian_rgb((0.55, 0.27, 0.04), 0.1)
    bunny = s.lambertian_rgb(NAMED["Yellow"], 0.05)
    s.objects.append(("list", [("plane", (0.0, 1.0, 0.0), -2.0, ground)]))
    pos, nrm, faces = bunny_proxy(subdivisions)
    v0, n0 = mesh_arrays(pos, nrm, faces)
    vs = []
    for ix in range(copies):
        for iz in range(copies):
            off = np.array([-2.0 + (ix - (copies - 1) / 2.0) * pitch, 0.0, iz * pitch])
            # offsets are applied in f64 then rounded through f32, as an OBJ holding the grid would be
            vs.append((v0.reshape(-1, 3, 3) + off[None, None, :]).astype(np.float32).astype(np.float64).reshape(-1, 9))
    s.objects.append(("mesh", np.concatenate(vs, 0), np.tile(n0, (copies * copies, 1)), bunny))
    return s


def tiny_mesh_scene(subdivisions=2, variant="lambertian"):
    """Small version of C1b for CPU-speed parity tests (320 triangles at subdivisions=2)."""
    return scene_main(subdivisions=subdivisions, obj=False, variant=variant)
