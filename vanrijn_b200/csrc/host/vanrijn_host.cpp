// vanrijn_host.cpp -- host side of the drop-in: scene types, OBJ loading, the reference-topology
// BVH build, flattening to the SoA layout of include/vanrijn_cuda.h, and partial_render_scene.
// No ray is ever traced on the host: everything below either prepares data or calls the C ABI.
// Reference paths are relative to /root/reference/src/.
#include "../../../include/vanrijn.hpp"

#include <algorithm>
#if defined(__x86_64__)
#include <immintrin.h>
#endif
#include <atomic>
#include <chrono>
#include <cmath>
#include <condition_variable>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <functional>
#include <limits>
#include <mutex>
#include <numeric>
#include <thread>

namespace vanrijn {

namespace {
const double kRgbBasis[7][32] = {
#include "../rgb_basis_tables.inc"
};
enum { B_WHITE = 0, B_CYAN, B_MAGENTA, B_YELLOW, B_RED, B_GREEN, B_BLUE };

inline Vec3 sub(Vec3 a, Vec3 b) { return Vec3(a.x - b.x, a.y - b.y, a.z - b.z); }
inline double dot(Vec3 a, Vec3 b) { return ((0.0 + a.x * b.x) + a.y * b.y) + a.z * b.z; }
inline Vec3 cross(Vec3 a, Vec3 b) { return Vec3(a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x); }
inline Vec3 normalize(Vec3 a) {
    double inv = 1.0 / std::sqrt(dot(a, a));
    return Vec3(a.x * inv, a.y * inv, a.z * inv);
}
} // namespace

// ------------------------------------------------------------------------------ colour
ColourRgbF ColourRgbF::from_named(NamedColour name) {
    switch (name) {
    case NamedColour::Black: return {0.0, 0.0, 0.0};
    case NamedColour::White: return {1.0, 1.0, 1.0};
    case NamedColour::Red: return {1.0, 0.0, 0.0};
    case NamedColour::Lime: return {0.0, 1.0, 0.0};
    case NamedColour::Blue: return {0.0, 0.0, 1.0};
    case NamedColour::Yellow: return {1.0, 1.0, 0.0};
    case NamedColour::Cyan: return {0.0, 1.0, 1.0};
    case NamedColour::Magenta: return {1.0, 0.0, 1.0};
    case NamedColour::Gray: return {0.5, 0.5, 0.5};
    case NamedColour::Maroon: return {0.5, 0.0, 0.0};
    case NamedColour::Olive: return {0.5, 0.5, 0.0};
    case NamedColour::Green: return {0.0, 0.5, 0.0};
    case NamedColour::Purple: return {0.5, 0.0, 0.5};
    case NamedColour::Teal: return {0.0, 0.5, 0.5};
    case NamedColour::Navy: return {0.0, 0.0, 0.5};
    }
    return {};
}

Spectrum Spectrum::black() { return grey(0.0); }
Spectrum Spectrum::grey(double brightness) {
    Spectrum s;
    s.samples = {brightness, brightness};
    return s;
}
Spectrum Spectrum::diamond_index_of_refraction() { // spectrum.rs:29-48
    Spectrum s;
    s.shortest_wavelength = 326.27, s.longest_wavelength = 774.9;
    s.samples = {2.505813241, 2.487866556, 2.473323675, 2.464986815, 2.455051934, 2.441251728,
                 2.431478974, 2.427076431, 2.420857286, 2.411429037, 2.406543164, 2.406202402};
    return s;
}
Spectrum Spectrum::reflection_from_linear_rgb(const ColourRgbF &c) { // spectrum.rs:81-165
    const double r = c.red, g = c.green, b = c.blue;
    int mid, last;
    double k0, k1, k2;
    if (r <= g && r <= b) {
        mid = B_CYAN, k0 = r;
        if (g <= b) last = B_BLUE, k1 = g - r, k2 = b - g;
        else last = B_GREEN, k1 = b - r, k2 = g - b;
    } else if (g <= r && g < b) {
        mid = B_MAGENTA, k0 = g;
        if (r <= b) last = B_BLUE, k1 = r - g, k2 = b - r;
        else last = B_RED, k1 = b - g, k2 = r - b;
    } else {
        mid = B_YELLOW, k0 = b;
        if (r <= g) last = B_GREEN, k1 = r - b, k2 = g - r;
        else last = B_RED, k1 = g - b, k2 = r - g;
    }
    Spectrum s;
    s.shortest_wavelength = 380.0, s.longest_wavelength = 720.0;
    s.samples.resize(32);
    for (int i = 0; i < 32; i++) s.samples[i] = k0 * kRgbBasis[B_WHITE][i] + k1 * kRgbBasis[mid][i] + k2 * kRgbBasis[last][i];
    return s;
}

// ------------------------------------------------------------------------------ materials
uint32_t LambertianMaterial::flatten(FlatSceneBuilder &out) const {
    return out.add_material(VRJ_MAT_LAMBERTIAN, out.add_spectrum(colour), diffuse_strength, 0.0, 0.0);
}
uint32_t PhongMaterial::flatten(FlatSceneBuilder &out) const {
    return out.add_material(VRJ_MAT_PHONG, out.add_spectrum(colour), diffuse_strength, specular_strength, smoothness);
}
uint32_t ReflectiveMaterial::flatten(FlatSceneBuilder &out) const {
    return out.add_material(VRJ_MAT_REFLECTIVE, out.add_spectrum(colour), diffuse_strength, reflection_strength, 0.0);
}
uint32_t SmoothTransparentDialectric::flatten(FlatSceneBuilder &out) const {
    return out.add_material(VRJ_MAT_DIELECTRIC, out.add_spectrum(eta), 0.0, 0.0, 0.0);
}

// ------------------------------------------------------------------------------ primitives
Plane::Plane(Vec3 n, double d, std::shared_ptr<Material> m) : distance_from_origin(d), material(std::move(m)) {
    normal = normalize(n);
    // vec3.rs:112-127 smallest_coord
    double ax = std::fabs(normal.x), ay = std::fabs(normal.y), az = std::fabs(normal.z);
    int smallest = ax < ay ? (ax < az ? 0 : 2) : (ay < az ? 1 : 2);
    Vec3 axis(smallest == 0 ? 1.0 : 0.0, smallest == 1 ? 1.0 : 0.0, smallest == 2 ? 1.0 : 0.0);
    cotangent = normalize(cross(normal, axis));
    tangent = cross(normal, cotangent);
}
void Sphere::flatten(FlatSceneBuilder &out, uint32_t object_id, uint32_t prim_id) const {
    out.add_sphere(*this, out.material_index(material.get()), object_id, prim_id);
}
void Plane::flatten(FlatSceneBuilder &out, uint32_t object_id, uint32_t prim_id) const {
    out.add_plane(*this, out.material_index(material.get()), object_id, prim_id);
}
void Triangle::flatten(FlatSceneBuilder &out, uint32_t object_id, uint32_t prim_id) const {
    out.add_triangle(*this, out.material_index(material.get()), object_id, prim_id);
}
void PrimitiveList::flatten(FlatSceneBuilder &out, uint32_t object_id) const {
    for (size_t i = 0; i < primitives.size(); i++) primitives[i]->flatten(out, object_id, (uint32_t)i);
}

// ------------------------------------------------------------------------------ BVH build
namespace {
struct BuildCtx {
    const std::vector<double> *v;  // 9 per triangle (input order)
    std::vector<double> lo, hi, centre; // 3 per triangle
    std::vector<uint32_t> order;
    std::vector<double> node_min, node_max;
    std::vector<int32_t> node_child;

    // util/axis_aligned_bounding_box.rs:76-99: first strictly-largest extent; degenerate extents count as -1
    static int largest_dimension(const double lo[3], const double hi[3]) {
        int dim = 0;
        double best = 0.0;
        for (int k = 0; k < 3; k++) {
            double extent = (lo[k] == hi[k]) ? -1.0 : hi[k] - lo[k];
            if (extent > best) dim = k, best = extent;
        }
        return dim;
    }
    // bounding_volume_hierarchy.rs:49-75.  Node `me` covers order[begin, end).  A median-split tree over n
    // primitives has exactly 2n-1 nodes, so DFS pre-order indices are known up front (left = me+1,
    // right = me + 2*n_left) and the big subtrees can be built on separate threads.  Node boxes are unions of
    // triangle boxes (min/max are exact, so this equals the reference's fold over the slice).
    uint32_t build(size_t begin, size_t end, uint32_t level, size_t me) {
        double blo[3], bhi[3];
        for (int k = 0; k < 3; k++) blo[k] = std::numeric_limits<double>::infinity(), bhi[k] = -blo[k];
        for (size_t i = begin; i < end; i++) {
            uint32_t t = order[i];
            for (int k = 0; k < 3; k++) blo[k] = std::fmin(blo[k], lo[3 * t + k]), bhi[k] = std::fmax(bhi[k], hi[3 * t + k]);
        }
        for (int k = 0; k < 3; k++) node_min[3 * me + k] = blo[k], node_max[3 * me + k] = bhi[k];
        if (end - begin <= 1) {
            node_child[2 * me] = ~(int32_t)begin; // leaf: ~first triangle (BVH-local, leaf order)
            node_child[2 * me + 1] = (int32_t)(end - begin);
            return level + 1;
        }
        int axis = largest_dimension(blo, bhi);
        // bounding_volume_hierarchy.rs:38-46: sort by box centre on that axis.  The reference uses
        // sort_unstable_by (order among equal keys unspecified); a stable sort makes the tree deterministic.
        std::stable_sort(order.begin() + begin, order.begin() + end,
                         [this, axis](uint32_t a, uint32_t b) { return centre[3 * a + axis] < centre[3 * b + axis]; });
        size_t pivot = begin + (end - begin) / 2;
        size_t l = me + 1, r = me + 2 * (pivot - begin);
        node_child[2 * me] = (int32_t)l, node_child[2 * me + 1] = (int32_t)r;
        uint32_t dl, dr;
        if (level < 4 && end - begin > 65536) {
            std::thread left([&] { dl = build(begin, pivot, level + 1, l); });
            dr = build(pivot, end, level + 1, r);
            left.join();
        } else {
            dl = build(begin, pivot, level + 1, l);
            dr = build(pivot, end, level + 1, r);
        }
        return std::max(dl, dr);
    }
};
} // namespace

// the recursion (or its device twin) over triangle arrays; fills every member but tri_material_ and returns the leaf order
std::vector<uint32_t> BoundingVolumeHierarchy::build_arrays(const std::vector<double> &v, const std::vector<double> &nr, Builder builder, int device) {
    BoundingVolumeHierarchy *bvh = this;
    const size_t n = v.size() / 9;
    const size_t n_nodes = n ? 2 * n - 1 : 1;
    std::vector<uint32_t> order;
    if (builder == Builder::AtUpload) {
        order.resize(n);
        std::iota(order.begin(), order.end(), 0u);
        uint32_t depth = 1;
        for (size_t m = n; m > 1; m = m - m / 2) depth++;
        bvh->depth_ = depth; // node arrays stay empty: flatten() emits VrjBvh.n_nodes == 0
    } else if (builder == Builder::Device) {
        // the same recursion on the GPU (csrc/vrj_bvh_build.cu); 4 doubles per node box there, 3 here
        std::vector<double> mn(4 * n_nodes), mx(4 * n_nodes);
        order.resize(n);
        bvh->node_child_.assign(2 * n_nodes, 0);
        if (vrj_bvh_build(device, n, v.data(), order.data(), mn.data(), mx.data(), bvh->node_child_.data(), &bvh->depth_, nullptr) != VRJ_OK)
            throw std::runtime_error(std::string("vrj_bvh_build: ") + vrj_last_error());
        bvh->node_min_.resize(3 * n_nodes), bvh->node_max_.resize(3 * n_nodes);
        for (size_t i = 0; i < n_nodes; i++)
            for (int k = 0; k < 3; k++) bvh->node_min_[3 * i + k] = mn[4 * i + k], bvh->node_max_[3 * i + k] = mx[4 * i + k];
    } else {
        BuildCtx cx;
        cx.v = &v;
        cx.lo.resize(3 * n), cx.hi.resize(3 * n), cx.centre.resize(3 * n);
        for (size_t i = 0; i < n; i++)
            for (int k = 0; k < 3; k++) {
                double a = v[i * 9 + k], b = v[i * 9 + 3 + k], c = v[i * 9 + 6 + k];
                double mn = std::fmin(std::fmin(a, b), c), mx = std::fmax(std::fmax(a, b), c);
                cx.lo[3 * i + k] = mn, cx.hi[3 * i + k] = mx;
                cx.centre[3 * i + k] = (mn + mx) / 2.0; // bounding_volume_hierarchy.rs:30-36
            }
        cx.order.resize(n);
        std::iota(cx.order.begin(), cx.order.end(), 0u);
        cx.node_child.assign(2 * n_nodes, 0);
        cx.node_min.assign(3 * n_nodes, 0.0), cx.node_max.assign(3 * n_nodes, 0.0);
        bvh->depth_ = cx.build(0, n, 0, 0);
        bvh->node_min_ = std::move(cx.node_min), bvh->node_max_ = std::move(cx.node_max), bvh->node_child_ = std::move(cx.node_child);
        order = std::move(cx.order);
    }
    bvh->tri_v_.resize(n * 9), bvh->tri_n_.resize(n * 9), bvh->tri_prim_id_.resize(n);
    for (size_t i = 0; i < n; i++) {
        uint32_t src = order[i];
        std::memcpy(&bvh->tri_v_[i * 9], &v[(size_t)src * 9], 72);
        std::memcpy(&bvh->tri_n_[i * 9], &nr[(size_t)src * 9], 72);
        bvh->tri_prim_id_[i] = src;
    }
    return order;
}

std::unique_ptr<BoundingVolumeHierarchy> BoundingVolumeHierarchy::build(std::vector<std::shared_ptr<Primitive>> &primitives,
                                                                        Builder builder, int device) {
    std::unique_ptr<BoundingVolumeHierarchy> bvh(new BoundingVolumeHierarchy());
    const size_t n = primitives.size();
    std::vector<double> v(n * 9), nr(n * 9);
    for (size_t i = 0; i < n; i++) {
        const Triangle *t = dynamic_cast<const Triangle *>(primitives[i].get());
        if (!t) throw std::runtime_error("BoundingVolumeHierarchy::build: only Triangle primitives can be stored on the device BVH");
        for (int k = 0; k < 3; k++) {
            v[i * 9 + 3 * k] = t->vertices[k].x, v[i * 9 + 3 * k + 1] = t->vertices[k].y, v[i * 9 + 3 * k + 2] = t->vertices[k].z;
            nr[i * 9 + 3 * k] = t->normals[k].x, nr[i * 9 + 3 * k + 1] = t->normals[k].y, nr[i * 9 + 3 * k + 2] = t->normals[k].z;
        }
    }
    std::vector<uint32_t> order = bvh->build_arrays(v, nr, builder, device);
    bvh->tri_material_.resize(n);
    std::vector<std::shared_ptr<Primitive>> reordered(n);
    for (size_t i = 0; i < n; i++) {
        bvh->tri_material_[i] = static_cast<const Triangle *>(primitives[order[i]].get())->material;
        reordered[i] = primitives[order[i]];
    }
    if (builder != Builder::AtUpload) primitives.swap(reordered); // the reference sorts the caller's slice in place
    return bvh;
}

std::unique_ptr<BoundingVolumeHierarchy> BoundingVolumeHierarchy::build(const TriangleMesh &mesh, std::shared_ptr<Material> material,
                                                                        Builder builder, int device) {
    if (mesh.vertices.size() != mesh.normals.size() || mesh.vertices.size() % 9) throw std::runtime_error("TriangleMesh: 9 doubles per triangle, vertices and normals");
    std::unique_ptr<BoundingVolumeHierarchy> bvh(new BoundingVolumeHierarchy());
    bvh->build_arrays(mesh.vertices, mesh.normals, builder, device);
    bvh->tri_material_.assign(mesh.vertices.size() / 9, material);
    return bvh;
}
void BoundingVolumeHierarchy::flatten(FlatSceneBuilder &out, uint32_t object_id) const { out.add_bvh(*this, object_id); }

// ------------------------------------------------------------------------------ flattening
uint32_t FlatSceneBuilder::add_spectrum(const Spectrum &s) {
    VrjSpectrum d;
    d.shortest_wavelength = s.shortest_wavelength, d.longest_wavelength = s.longest_wavelength;
    d.first_sample = (uint32_t)samples_.size(), d.n_samples = (uint32_t)s.samples.size();
    samples_.insert(samples_.end(), s.samples.begin(), s.samples.end());
    spectra_.push_back(d);
    return (uint32_t)spectra_.size() - 1;
}
uint32_t FlatSceneBuilder::add_material(uint32_t kind, uint32_t spectrum, double p0, double p1, double p2) {
    materials_.push_back(VrjMaterial{kind, spectrum, p0, p1, p2});
    return (uint32_t)materials_.size() - 1;
}
uint32_t FlatSceneBuilder::material_index(const Material *m) {
    if (!m) throw std::runtime_error("primitive without a material");
    for (auto &e : material_cache_)
        if (e.first == m) return e.second;
    uint32_t id = m->flatten(*this);
    material_cache_.push_back({m, id});
    return id;
}
void FlatSceneBuilder::add_sphere(const Sphere &s, uint32_t material, uint32_t object_id, uint32_t prim_id) {
    spheres_.push_back(VrjSphere{{s.centre.x, s.centre.y, s.centre.z}, s.radius, material, 0});
    items_.push_back(VrjItem{VRJ_ITEM_SPHERE, (uint32_t)spheres_.size() - 1, object_id, prim_id});
}
void FlatSceneBuilder::add_plane(const Plane &p, uint32_t material, uint32_t object_id, uint32_t prim_id) {
    VrjPlane d{};
    d.normal[0] = p.normal.x, d.normal[1] = p.normal.y, d.normal[2] = p.normal.z;
    d.tangent[0] = p.tangent.x, d.tangent[1] = p.tangent.y, d.tangent[2] = p.tangent.z;
    d.cotangent[0] = p.cotangent.x, d.cotangent[1] = p.cotangent.y, d.cotangent[2] = p.cotangent.z;
    d.distance_from_origin = p.distance_from_origin, d.material = material;
    planes_.push_back(d);
    items_.push_back(VrjItem{VRJ_ITEM_PLANE, (uint32_t)planes_.size() - 1, object_id, prim_id});
}
void FlatSceneBuilder::add_triangle(const Triangle &t, uint32_t material, uint32_t object_id, uint32_t prim_id) {
    for (int k = 0; k < 3; k++) {
        const Vec3 &v = t.vertices[k], &n = t.normals[k];
        tri_[k].insert(tri_[k].end(), {v.x, v.y, v.z, 0.0});
        tri_[3 + k].insert(tri_[3 + k].end(), {n.x, n.y, n.z, 0.0});
    }
    tri_material_.push_back(material), tri_prim_id_.push_back(prim_id);
    items_.push_back(VrjItem{VRJ_ITEM_TRIANGLE, (uint32_t)tri_material_.size() - 1, object_id, prim_id});
}
void FlatSceneBuilder::add_bvh(const BoundingVolumeHierarchy &b, uint32_t object_id) {
    VrjBvh d{};
    d.first_node = node_child_.size() / 2, d.n_nodes = b.node_child_.size() / 2;
    d.first_triangle = tri_material_.size(), d.n_triangles = b.triangle_count();
    d.depth = b.depth_;
    const size_t nt = b.triangle_count();
    for (int k = 0; k < 6; k++) tri_[k].reserve(tri_[k].size() + 4 * nt);
    tri_material_.reserve(tri_material_.size() + nt), tri_prim_id_.reserve(tri_prim_id_.size() + nt);
    node_min_.reserve(node_min_.size() + 4 * d.n_nodes), node_max_.reserve(node_max_.size() + 4 * d.n_nodes);
    node_child_.reserve(node_child_.size() + 2 * d.n_nodes);
    for (size_t i = 0; i < nt; i++) {
        for (int k = 0; k < 3; k++) {
            const double *v = &b.tri_v_[i * 9 + 3 * k], *n = &b.tri_n_[i * 9 + 3 * k];
            tri_[k].insert(tri_[k].end(), {v[0], v[1], v[2], 0.0});
            tri_[3 + k].insert(tri_[3 + k].end(), {n[0], n[1], n[2], 0.0});
        }
        tri_material_.push_back(material_index(b.tri_material_[i].get()));
        tri_prim_id_.push_back(b.tri_prim_id_[i]);
    }
    for (size_t n = 0; n < d.n_nodes; n++) {
        for (int k = 0; k < 3; k++) node_min_.push_back(b.node_min_[3 * n + k]), node_max_.push_back(b.node_max_[3 * n + k]);
        node_min_.push_back(0.0), node_max_.push_back(0.0);
        int32_t l = b.node_child_[2 * n], r = b.node_child_[2 * n + 1];
        if (l >= 0) {
            node_child_.push_back(l + (int32_t)d.first_node), node_child_.push_back(r + (int32_t)d.first_node);
        } else {
            node_child_.push_back(~((~l) + (int32_t)d.first_triangle)), node_child_.push_back(r);
        }
    }
    bvhs_.push_back(d);
    items_.push_back(VrjItem{VRJ_ITEM_BVH, (uint32_t)bvhs_.size() - 1, object_id, 0});
}
const VrjSceneDesc &FlatSceneBuilder::desc(const Vec3 &camera) {
    VrjSceneDesc &d = desc_;
    d = VrjSceneDesc{};
    d.abi_version = VRJ_ABI_VERSION;
    d.camera_location[0] = camera.x, d.camera_location[1] = camera.y, d.camera_location[2] = camera.z;
    d.n_spectra = (uint32_t)spectra_.size(), d.n_spectrum_samples = (uint32_t)samples_.size();
    d.spectra = spectra_.data(), d.spectrum_samples = samples_.data();
    d.n_materials = (uint32_t)materials_.size(), d.materials = materials_.data();
    d.n_spheres = (uint32_t)spheres_.size(), d.spheres = spheres_.data();
    d.n_planes = (uint32_t)planes_.size(), d.planes = planes_.data();
    d.n_bvhs = (uint32_t)bvhs_.size(), d.bvhs = bvhs_.data();
    d.n_triangles = tri_material_.size();
    d.tri_v0 = tri_[0].data(), d.tri_v1 = tri_[1].data(), d.tri_v2 = tri_[2].data();
    d.tri_n0 = tri_[3].data(), d.tri_n1 = tri_[4].data(), d.tri_n2 = tri_[5].data();
    d.tri_material = tri_material_.data(), d.tri_prim_id = tri_prim_id_.data();
    d.n_nodes = node_child_.size() / 2;
    d.node_min = node_min_.data(), d.node_max = node_max_.data(), d.node_child = node_child_.data();
    d.n_items = (uint32_t)items_.size(), d.items = items_.data();
    return d;
}

// ------------------------------------------------------------------------------ OBJ loading
// mesh.rs:13-88 over the behaviour of obj 0.9's Obj::<SimplePolygon>::load: `v`, `vn`, `f`
// (a, a/b, a//c, a/b/c; 1-based, negative = relative to the end), f32 parse then widen,
// fan triangulation around the polygon's first vertex, zero normal when a vertex has none.
std::vector<std::shared_ptr<Primitive>> load_obj(const std::string &filename, std::shared_ptr<Material> material) {
    const TriangleMesh mesh = load_obj_mesh(filename);
    const size_t n = mesh.triangle_count();
    std::vector<std::shared_ptr<Primitive>> out(n);
    for (size_t i = 0; i < n; i++) {
        const double *v = &mesh.vertices[9 * i], *m = &mesh.normals[9 * i];
        out[i] = std::make_shared<Triangle>(std::array<Vec3, 3>{Vec3(v[0], v[1], v[2]), Vec3(v[3], v[4], v[5]), Vec3(v[6], v[7], v[8])},
                                            std::array<Vec3, 3>{Vec3(m[0], m[1], m[2]), Vec3(m[3], m[4], m[5]), Vec3(m[6], m[7], m[8])}, material);
    }
    return out;
}
TriangleMesh load_obj_mesh(const std::string &filename) {
    FILE *f = std::fopen(filename.c_str(), "r");
    if (!f) throw std::runtime_error("load_obj: cannot open " + filename);
    std::vector<float> positions, normals;
    TriangleMesh out;
    std::vector<long> vi, ni;
    char line[8192];
    auto is_space = [](char c) { return c == ' ' || c == '\t'; };
    while (std::fgets(line, sizeof line, f)) {
        const char *p = line;
        while (is_space(*p)) p++;
        if (p[0] == 'v' && is_space(p[1])) {
            char *q = const_cast<char *>(p + 1);
            for (int k = 0; k < 3; k++) positions.push_back(std::strtof(q, &q));
        } else if (p[0] == 'v' && p[1] == 'n' && is_space(p[2])) {
            char *q = const_cast<char *>(p + 2);
            for (int k = 0; k < 3; k++) normals.push_back(std::strtof(q, &q));
        } else if (p[0] == 'f' && is_space(p[1])) {
            vi.clear(), ni.clear();
            char *q = const_cast<char *>(p + 1);
            const long np = (long)positions.size() / 3, nn = (long)normals.size() / 3;
            while (true) {
                while (is_space(*q)) q++;
                if (*q == '\0' || *q == '\n' || *q == '\r' || *q == '#') break;
                long v = std::strtol(q, &q, 10), n = 0;
                bool has_normal = false;
                if (*q == '/') {
                    q++;
                    if (*q != '/') (void)std::strtol(q, &q, 10);
                    if (*q == '/') {
                        q++;
                        n = std::strtol(q, &q, 10);
                        has_normal = true;
                    }
                }
                vi.push_back(v < 0 ? np + v : v - 1);
                ni.push_back(has_normal ? (n < 0 ? nn + n : n - 1) : -1);
            }
            auto vertex = [&](size_t k) { return Vec3(positions[3 * vi[k]], positions[3 * vi[k] + 1], positions[3 * vi[k] + 2]); };
            auto normal = [&](size_t k) {
                return ni[k] < 0 ? Vec3() : Vec3(normals[3 * ni[k]], normals[3 * ni[k] + 1], normals[3 * ni[k] + 2]);
            };
            for (size_t k = 1; k + 1 < vi.size(); k++) {
                const Vec3 tv[3] = {vertex(0), vertex(k), vertex(k + 1)}, tn[3] = {normal(0), normal(k), normal(k + 1)};
                for (int c = 0; c < 3; c++) {
                    out.vertices.insert(out.vertices.end(), {tv[c].x, tv[c].y, tv[c].z});
                    out.normals.insert(out.normals.end(), {tn[c].x, tn[c].y, tn[c].z});
                }
            }
        }
    }
    std::fclose(f);
    return out;
}

// ------------------------------------------------------------------------------ tiles, accumulation buffer
TileIterator::TileIterator(size_t total_width, size_t total_height, size_t tile_size)
    : tile_size_(tile_size), total_height_(total_height), total_width_(total_width) {
    if (!(tile_size > 0 && tile_size * 2 < std::numeric_limits<size_t>::max())) throw std::runtime_error("TileIterator: bad tile size");
}
bool TileIterator::next(Tile &tile) { // tile_iterator.rs:41-66
    if (current_row_ >= total_height_) return false;
    tile.start_column = current_column_, tile.end_column = std::min(total_width_, current_column_ + tile_size_);
    tile.start_row = current_row_, tile.end_row = std::min(total_height_, current_row_ + tile_size_);
    current_column_ += tile_size_;
    if (current_column_ >= total_width_) current_row_ += tile_size_, current_column_ = 0;
    return true;
}

AccumulationBuffer::AccumulationBuffer(size_t width, size_t height)
    : colour(3 * width * height, 0.0), colour_sum(3 * width * height, 0.0), colour_bias(3 * width * height, 0.0),
      weight(width * height, 0.0), weight_bias(width * height, 0.0), width_(width), height_(height) {}

AccumulationBuffer::AccumulationBuffer(size_t width, size_t height, Uninitialized, bool kahan_state)
    : colour(3 * width * height), colour_sum(kahan_state ? 3 * width * height : 0), colour_bias(kahan_state ? 3 * width * height : 0),
      weight(kahan_state ? width * height : 0), weight_bias(kahan_state ? width * height : 0), width_(width), height_(height) {}

ImageRgbU8 AccumulationBuffer::to_image_rgb_u8(int device) const {
    ImageRgbU8 image(width_, height_);
    if (vrj_tone_map(device, VRJ_MEM_HOST, VRJ_TONEMAP_XYZ, colour.data(), width_ * height_, image.pixel_data().data()) != VRJ_OK)
        throw std::runtime_error(std::string("vrj_tone_map: ") + vrj_last_error());
    return image;
}

// ------------------------------------------------------------------------------ PNG (image.rs:52-66)
namespace {
struct Crc32 {
    uint32_t table[256];
    Crc32() {
        for (uint32_t n = 0; n < 256; n++) {
            uint32_t c = n;
            for (int k = 0; k < 8; k++) c = (c & 1) ? 0xedb88320u ^ (c >> 1) : c >> 1;
            table[n] = c;
        }
    }
    uint32_t update(uint32_t crc, const uint8_t *p, size_t n) const {
        for (size_t i = 0; i < n; i++) crc = table[(crc ^ p[i]) & 0xff] ^ (crc >> 8);
        return crc;
    }
};
void put_be32(std::vector<uint8_t> &v, uint32_t x) {
    v.push_back((uint8_t)(x >> 24)), v.push_back((uint8_t)(x >> 16)), v.push_back((uint8_t)(x >> 8)), v.push_back((uint8_t)x);
}
void put_chunk(std::vector<uint8_t> &file, const char type[4], const std::vector<uint8_t> &data) {
    static const Crc32 crc;
    put_be32(file, (uint32_t)data.size());
    const size_t start = file.size();
    file.insert(file.end(), type, type + 4);
    file.insert(file.end(), data.begin(), data.end());
    put_be32(file, crc.update(0xffffffffu, file.data() + start, file.size() - start) ^ 0xffffffffu);
}
} // namespace

void ImageRgbU8::write_png(const std::string &filename) const {
    if (width_ == 0 || height_ == 0 || width_ > 0x7fffffff || height_ > 0x7fffffff) throw std::runtime_error("write_png: bad image size");
    // raw scanlines: filter byte 0 + RGB bytes
    const size_t stride = 3 * width_ + 1;
    std::vector<uint8_t> raw(stride * height_);
    for (size_t r = 0; r < height_; r++) {
        raw[r * stride] = 0;
        std::memcpy(&raw[r * stride + 1], &pixel_data_[r * 3 * width_], 3 * width_);
    }
    // zlib stream of stored blocks (RFC 1950 / 1951) + Adler-32
    std::vector<uint8_t> z;
    z.reserve(raw.size() + raw.size() / 65535 * 5 + 16);
    z.push_back(0x78), z.push_back(0x01);
    uint32_t a = 1, b = 0;
    for (size_t off = 0; off < raw.size() || off == 0;) {
        const size_t n = std::min<size_t>(65535, raw.size() - off);
        const bool last = off + n >= raw.size();
        z.push_back(last ? 1 : 0);
        z.push_back((uint8_t)(n & 0xff)), z.push_back((uint8_t)(n >> 8));
        z.push_back((uint8_t)(~n & 0xff)), z.push_back((uint8_t)((~n >> 8) & 0xff));
        z.insert(z.end(), raw.begin() + off, raw.begin() + off + n);
        for (size_t i = 0; i < n; i++) {
            a += raw[off + i];
            if (a >= 65521) a -= 65521;
            b += a;
            if (b >= 65521) b -= 65521;
        }
        off += n;
        if (last) break;
    }
    put_be32(z, (b << 16) | a);
    std::vector<uint8_t> file = {0x89, 'P', 'N', 'G', 0x0d, 0x0a, 0x1a, 0x0a};
    std::vector<uint8_t> ihdr;
    put_be32(ihdr, (uint32_t)width_), put_be32(ihdr, (uint32_t)height_);
    ihdr.insert(ihdr.end(), {8, 2, 0, 0, 0}); // 8 bits, colour type 2 (RGB), deflate, adaptive filtering, no interlace
    put_chunk(file, "IHDR", ihdr);
    put_chunk(file, "IDAT", z);
    put_chunk(file, "IEND", {});
    FILE *f = std::fopen(filename.c_str(), "wb");
    if (!f) throw std::runtime_error("write_png: cannot open " + filename);
    const bool ok = std::fwrite(file.data(), 1, file.size(), f) == file.size();
    if (std::fclose(f) != 0 || !ok) throw std::runtime_error("write_png: write failed: " + filename);
}

namespace {
// A few resident threads for merge_tile: a whole 1080p frame is 200 MB of reads and writes per merge, and the reference's
// loop (main.rs:215-217) merges on ONE thread once per partial_render_scene call -- with the rendering on the GPU that
// single thread is what bounds the loop, so big tiles are split by rows over a pool that lives as long as the process
// (starting threads per call cost as much as a quarter of the merge).
class RowPool {
  public:
    static RowPool &instance() {
        static RowPool pool;
        return pool;
    }
    // runs fn(r0, r1) over [0, rows) in pieces of a few rows that the pool's threads and the caller take one after another;
    // returns when all are done.  Small pieces, handed out on demand: the threads do not run at the same speed (a sibling
    // hyper-thread may be busy feeding the GPU), and with one fixed share per thread the slowest one set the time of the pass.
    void run(size_t rows, const std::function<void(size_t, size_t)> &fn) {
        std::lock_guard<std::mutex> serial(serial_); // one merge at a time owns the pool
        if (rows == 0) return;
        uint64_t gen;
        {
            std::lock_guard<std::mutex> g(m_);
            fn_ = &fn, rows_ = rows, per_ = std::max<size_t>(1, rows / ((workers_.size() + 1) * 8));
            pieces_ = (rows + per_ - 1) / per_, next_ = 0, finished_ = 0, gen = ++generation_;
        }
        wake_.notify_all();
        work(gen);
        std::unique_lock<std::mutex> g(m_);
        done_.wait(g, [&] { return finished_ == pieces_; });
        fn_ = nullptr;
    }

  private:
    RowPool() {
        const unsigned hw = std::max(1u, std::thread::hardware_concurrency());
        // + the calling thread = half the cores: a 1080p merge runs at 180 GB/s with 8 threads and gains nothing from 16
        // (build/merge_bench), and the other half stays free for the workers that enqueue the device's kernels -- a worker
        // that loses its core while it launches a wavefront leaves the GPU idle
        unsigned n = std::min(15u, hw > 3 ? hw / 2 - 1 : 1u);
        if (const char *e = std::getenv("VRJ_MERGE_THREADS")) n = (unsigned)std::max(0, std::atoi(e) - 1); // experiments
        for (unsigned i = 0; i < n; i++) workers_.emplace_back([this] { loop(); });
    }
    ~RowPool() {
        {
            std::lock_guard<std::mutex> g(m_);
            stop_ = true;
        }
        wake_.notify_all();
        for (auto &t : workers_) t.join();
    }
    // take pieces of generation `gen` until none is left (or the pool has moved on)
    void work(uint64_t gen) {
        for (;;) {
            size_t piece, rows, per;
            const std::function<void(size_t, size_t)> *fn;
            {
                std::lock_guard<std::mutex> g(m_);
                if (generation_ != gen || !fn_ || next_ >= pieces_) return;
                piece = next_++, rows = rows_, per = per_, fn = fn_;
            }
            (*fn)(piece * per, std::min(rows, (piece + 1) * per)); // run() cannot return before this piece is counted below
            std::lock_guard<std::mutex> g(m_);
            if (++finished_ == pieces_) done_.notify_one();
        }
    }
    void loop() {
        uint64_t seen = 0;
        for (;;) {
            uint64_t gen;
            {
                std::unique_lock<std::mutex> g(m_);
                wake_.wait(g, [&] { return stop_ || (generation_ != seen && fn_); });
                if (stop_) return;
                gen = seen = generation_;
            }
            work(gen);
        }
    }
    std::vector<std::thread> workers_;
    std::mutex m_, serial_;
    std::condition_variable wake_, done_;
    const std::function<void(size_t, size_t)> *fn_ = nullptr;
    size_t rows_ = 0, per_ = 1, pieces_ = 0, next_ = 0, finished_ = 0;
    uint64_t generation_ = 0;
    bool stop_ = false;
};
} // namespace

// One row of merge_tile (accumulation_buffer.rs:62-85) for `ns` source buffers applied in order: per pixel and buffer
// inv = 1/(w1+w2); c = (c*w1 + s*w2)*inv per channel; w = w1+w2.  The destination's colour and weight are read and written
// once whatever `ns` is.  On AVX2 hosts four pixels go through the same operations at once: the weights are expanded to one
// value per channel with lane permutes, which turns the interleaved XYZ triples into three flat vectors.  Every lane performs
// the same IEEE binary64 operation on the same operands as the scalar form (separate multiply and add: no FMA), so the result
// is bit-identical (tests/test_host_cpu.py compares both paths with the oracle's blend).
struct MergeSource {
    const double *colour; // first pixel of the row
    const double *weight; // NULL: `uniform`
    double uniform;
};
static void merge_row_scalar(double *colour, double *weight, const MergeSource *src, size_t ns, size_t j0, size_t n) {
    for (size_t j = j0; j < n; j++) {
        double w1 = weight[j], c0 = colour[3 * j], c1 = colour[3 * j + 1], c2 = colour[3 * j + 2];
        for (size_t k = 0; k < ns; k++) {
            const double w2 = src[k].weight ? src[k].weight[j] : src[k].uniform;
            const double inv = 1.0 / (w1 + w2); // accumulation_buffer.rs:81-85
            const double *sc = src[k].colour + 3 * j;
            c0 = (c0 * w1 + sc[0] * w2) * inv, c1 = (c1 * w1 + sc[1] * w2) * inv, c2 = (c2 * w1 + sc[2] * w2) * inv;
            w1 += w2;
        }
        colour[3 * j] = c0, colour[3 * j + 1] = c1, colour[3 * j + 2] = c2, weight[j] = w1;
    }
}
#if defined(__x86_64__)
__attribute__((target("avx2")))
static void merge_row_avx2(double *colour, double *weight, const MergeSource *src, size_t ns, size_t n) {
    const __m256d one = _mm256_set1_pd(1.0);
    size_t j = 0;
    for (; j + 4 <= n; j += 4) {
        __m256d w1 = _mm256_loadu_pd(weight + j);
        __m256d c0 = _mm256_loadu_pd(colour + 3 * j), c1 = _mm256_loadu_pd(colour + 3 * j + 4), c2 = _mm256_loadu_pd(colour + 3 * j + 8);
        for (size_t k = 0; k < ns; k++) {
            const __m256d w2 = src[k].weight ? _mm256_loadu_pd(src[k].weight + j) : _mm256_set1_pd(src[k].uniform);
            const __m256d sum = _mm256_add_pd(w1, w2), inv = _mm256_div_pd(one, sum);
            const double *sc = src[k].colour + 3 * j;
            // pixels a b c d -> channel vectors [a a a b] [b b c c] [c d d d]
#define VRJ_BLEND(c, off, imm)                                                                                                   \
    c = _mm256_mul_pd(_mm256_add_pd(_mm256_mul_pd(c, _mm256_permute4x64_pd(w1, imm)),                                            \
                                    _mm256_mul_pd(_mm256_loadu_pd(sc + off), _mm256_permute4x64_pd(w2, imm))),                   \
                      _mm256_permute4x64_pd(inv, imm))
            VRJ_BLEND(c0, 0, 0x40);
            VRJ_BLEND(c1, 4, 0xA5);
            VRJ_BLEND(c2, 8, 0xFE);
#undef VRJ_BLEND
            w1 = sum;
        }
        _mm256_storeu_pd(weight + j, w1);
        _mm256_storeu_pd(colour + 3 * j, c0), _mm256_storeu_pd(colour + 3 * j + 4, c1), _mm256_storeu_pd(colour + 3 * j + 8, c2);
    }
    merge_row_scalar(colour, weight, src, ns, j, n);
}
#endif
static void merge_row(double *colour, double *weight, const MergeSource *src, size_t ns, size_t n) {
#if defined(__x86_64__)
    static const bool avx2 = __builtin_cpu_supports("avx2") && !std::getenv("VRJ_MERGE_SCALAR");
    if (avx2) return merge_row_avx2(colour, weight, src, ns, n);
#endif
    merge_row_scalar(colour, weight, src, ns, 0, n);
}

void AccumulationBuffer::merge_tile(const Tile &tile, const AccumulationBuffer &src) { merge_tiles(tile, {&src}); }

void AccumulationBuffer::merge_tiles(const Tile &tile, const std::vector<const AccumulationBuffer *> &srcs) {
    for (const AccumulationBuffer *src : srcs)
        if (tile.width() != src->width() || tile.height() != src->height()) throw std::runtime_error("merge_tile: tile and source sizes differ");
    if (tile.end_row > height_ || tile.end_column > width_) throw std::runtime_error("merge_tile: tile outside the buffer");
    if (weight.empty()) throw std::runtime_error("merge_tile: the destination needs per-pixel weights");
    if (srcs.empty()) return;
    auto rows = [&](size_t r0, size_t r1) {
        std::vector<MergeSource> ms(srcs.size());
        for (size_t i = r0; i < r1; i++) {
            const size_t d = (tile.start_row + i) * width_ + tile.start_column, s = i * tile.width();
            for (size_t k = 0; k < srcs.size(); k++) // a colour-only tile carries one weight for all its pixels
                ms[k] = MergeSource{srcs[k]->colour.data() + 3 * s, srcs[k]->weight.empty() ? nullptr : srcs[k]->weight.data() + s, srcs[k]->uniform_weight};
            merge_row(colour.data() + 3 * d, weight.data() + d, ms.data(), ms.size(), tile.width());
        }
    };
    // pixels are independent: big tiles are merged by the resident row pool
    if (tile.width() * tile.height() < (size_t(1) << 18)) return rows(0, tile.height());
    RowPool::instance().run(tile.height(), rows);
}

// ------------------------------------------------------------------------------ scene cache (SURVEY 8f N3)
namespace {
const char kCacheMagic[8] = {'V', 'R', 'J', 'S', 'C', 'N', '1', 0};
template <typename T>
void put_array(std::vector<uint8_t> &out, const std::vector<T> &v) {
    const uint64_t n = v.size();
    const uint8_t *pn = reinterpret_cast<const uint8_t *>(&n);
    out.insert(out.end(), pn, pn + 8);
    const uint8_t *p = reinterpret_cast<const uint8_t *>(v.data());
    out.insert(out.end(), p, p + n * sizeof(T));
}
template <typename T>
void get_array(const std::vector<uint8_t> &in, size_t &pos, std::vector<T> &v) {
    if (pos + 8 > in.size()) throw std::runtime_error("scene cache: truncated");
    uint64_t n;
    std::memcpy(&n, &in[pos], 8);
    pos += 8;
    if (n > (in.size() - pos) / sizeof(T)) throw std::runtime_error("scene cache: truncated");
    v.resize(n);
    if (n) std::memcpy(v.data(), &in[pos], n * sizeof(T));
    pos += n * sizeof(T);
}
} // namespace

FlatScene::FlatScene(const VrjSceneDesc &d) {
    desc_ = d;
    spectra_.assign(d.spectra, d.spectra + d.n_spectra), samples_.assign(d.spectrum_samples, d.spectrum_samples + d.n_spectrum_samples);
    materials_.assign(d.materials, d.materials + d.n_materials), spheres_.assign(d.spheres, d.spheres + d.n_spheres);
    planes_.assign(d.planes, d.planes + d.n_planes), bvhs_.assign(d.bvhs, d.bvhs + d.n_bvhs), items_.assign(d.items, d.items + d.n_items);
    const double *tri[6] = {d.tri_v0, d.tri_v1, d.tri_v2, d.tri_n0, d.tri_n1, d.tri_n2};
    for (int k = 0; k < 6; k++) tri_[k].assign(tri[k], tri[k] + 4 * d.n_triangles);
    tri_material_.assign(d.tri_material, d.tri_material + d.n_triangles), tri_prim_id_.assign(d.tri_prim_id, d.tri_prim_id + d.n_triangles);
    node_min_.assign(d.node_min, d.node_min + 4 * d.n_nodes), node_max_.assign(d.node_max, d.node_max + 4 * d.n_nodes);
    node_child_.assign(d.node_child, d.node_child + 2 * d.n_nodes);
    bind();
}
void FlatScene::bind() {
    VrjSceneDesc &d = desc_;
    d.n_spectra = (uint32_t)spectra_.size(), d.n_spectrum_samples = (uint32_t)samples_.size();
    d.spectra = spectra_.data(), d.spectrum_samples = samples_.data();
    d.n_materials = (uint32_t)materials_.size(), d.materials = materials_.data();
    d.n_spheres = (uint32_t)spheres_.size(), d.spheres = spheres_.data();
    d.n_planes = (uint32_t)planes_.size(), d.planes = planes_.data();
    d.n_bvhs = (uint32_t)bvhs_.size(), d.bvhs = bvhs_.data();
    d.n_triangles = tri_material_.size();
    d.tri_v0 = tri_[0].data(), d.tri_v1 = tri_[1].data(), d.tri_v2 = tri_[2].data();
    d.tri_n0 = tri_[3].data(), d.tri_n1 = tri_[4].data(), d.tri_n2 = tri_[5].data();
    d.tri_material = tri_material_.data(), d.tri_prim_id = tri_prim_id_.data();
    d.n_nodes = node_child_.size() / 2;
    d.node_min = node_min_.data(), d.node_max = node_max_.data(), d.node_child = node_child_.data();
    d.n_items = (uint32_t)items_.size(), d.items = items_.data();
}
void FlatScene::save(const std::string &filename) const {
    std::vector<uint8_t> out(kCacheMagic, kCacheMagic + 8);
    const uint32_t head[2] = {VRJ_ABI_VERSION, 0};
    out.insert(out.end(), reinterpret_cast<const uint8_t *>(head), reinterpret_cast<const uint8_t *>(head) + 8);
    out.insert(out.end(), reinterpret_cast<const uint8_t *>(desc_.camera_location), reinterpret_cast<const uint8_t *>(desc_.camera_location) + 24);
    put_array(out, spectra_), put_array(out, samples_), put_array(out, materials_), put_array(out, spheres_), put_array(out, planes_);
    put_array(out, bvhs_), put_array(out, items_);
    for (int k = 0; k < 6; k++) put_array(out, tri_[k]);
    put_array(out, tri_material_), put_array(out, tri_prim_id_), put_array(out, node_min_), put_array(out, node_max_), put_array(out, node_child_);
    static const Crc32 crc;
    const uint32_t sum = crc.update(0xffffffffu, out.data(), out.size()) ^ 0xffffffffu;
    out.insert(out.end(), reinterpret_cast<const uint8_t *>(&sum), reinterpret_cast<const uint8_t *>(&sum) + 4);
    FILE *f = std::fopen(filename.c_str(), "wb");
    if (!f) throw std::runtime_error("scene cache: cannot open " + filename);
    const bool ok = std::fwrite(out.data(), 1, out.size(), f) == out.size();
    if (std::fclose(f) != 0 || !ok) throw std::runtime_error("scene cache: write failed: " + filename);
}
FlatScene FlatScene::load(const std::string &filename) {
    FILE *f = std::fopen(filename.c_str(), "rb");
    if (!f) throw std::runtime_error("scene cache: cannot open " + filename);
    std::vector<uint8_t> in;
    uint8_t buf[1 << 16];
    for (size_t n; (n = std::fread(buf, 1, sizeof buf, f)) > 0;) in.insert(in.end(), buf, buf + n);
    std::fclose(f);
    if (in.size() < 8 + 8 + 24 + 4 || std::memcmp(in.data(), kCacheMagic, 8) != 0) throw std::runtime_error("scene cache: not a scene cache file: " + filename);
    static const Crc32 crc;
    uint32_t stored;
    std::memcpy(&stored, &in[in.size() - 4], 4);
    if ((crc.update(0xffffffffu, in.data(), in.size() - 4) ^ 0xffffffffu) != stored) throw std::runtime_error("scene cache: checksum mismatch: " + filename);
    in.resize(in.size() - 4);
    uint32_t head[2];
    std::memcpy(head, &in[8], 8);
    if (head[0] != VRJ_ABI_VERSION) throw std::runtime_error("scene cache: written for another ABI version");
    FlatScene s;
    s.desc_.abi_version = VRJ_ABI_VERSION;
    std::memcpy(s.desc_.camera_location, &in[16], 24);
    size_t pos = 40;
    get_array(in, pos, s.spectra_), get_array(in, pos, s.samples_), get_array(in, pos, s.materials_), get_array(in, pos, s.spheres_);
    get_array(in, pos, s.planes_), get_array(in, pos, s.bvhs_), get_array(in, pos, s.items_);
    for (int k = 0; k < 6; k++) get_array(in, pos, s.tri_[k]);
    get_array(in, pos, s.tri_material_), get_array(in, pos, s.tri_prim_id_), get_array(in, pos, s.node_min_), get_array(in, pos, s.node_max_);
    get_array(in, pos, s.node_child_);
    const size_t nt = s.tri_material_.size();
    for (int k = 0; k < 6; k++)
        if (s.tri_[k].size() != 4 * nt) throw std::runtime_error("scene cache: inconsistent triangle arrays");
    if (s.tri_prim_id_.size() != nt || s.node_min_.size() != 2 * s.node_child_.size() || s.node_max_.size() != s.node_min_.size() || pos != in.size())
        throw std::runtime_error("scene cache: inconsistent arrays");
    s.bind();
    return s;
}
void save_scene_cache(const Scene &scene, const std::string &filename) {
    if (scene.flattened) return scene.flattened->save(filename);
    FlatSceneBuilder fb;
    for (size_t i = 0; i < scene.objects.size(); i++) scene.objects[i]->flatten(fb, (uint32_t)i);
    FlatScene(fb.desc(scene.camera_location)).save(filename);
}
Scene load_scene_cache(const std::string &filename) {
    Scene scene;
    auto flat = std::make_shared<FlatScene>(FlatScene::load(filename));
    scene.camera_location = Vec3(flat->desc().camera_location[0], flat->desc().camera_location[1], flat->desc().camera_location[2]);
    scene.flattened = std::move(flat);
    return scene;
}

// ------------------------------------------------------------------------------ device scene + render
struct Scene::DeviceCache {
    std::mutex mutex;
    std::vector<std::pair<int, VrjScene *>> scenes;
    ~DeviceCache() {
        for (auto &e : scenes) vrj_scene_destroy(e.second);
    }
};
Scene::~Scene() = default;

const VrjScene *device_scene(const Scene &scene, int device) {
    static std::mutex create_mutex;
    {
        std::lock_guard<std::mutex> g(create_mutex);
        if (!scene.device_cache) scene.device_cache = std::make_shared<Scene::DeviceCache>();
    }
    std::lock_guard<std::mutex> g(scene.device_cache->mutex);
    for (auto &e : scene.device_cache->scenes)
        if (e.first == device) return e.second;
    FlatSceneBuilder fb;
    const VrjSceneDesc *desc = nullptr;
    if (scene.flattened) {
        desc = &scene.flattened->desc();
    } else {
        for (size_t i = 0; i < scene.objects.size(); i++) scene.objects[i]->flatten(fb, (uint32_t)i);
        desc = &fb.desc(scene.camera_location);
    }
    VrjScene *dev = nullptr;
    if (vrj_scene_create(desc, device, &dev) != VRJ_OK)
        throw std::runtime_error(std::string("vrj_scene_create: ") + vrj_last_error());
    scene.device_cache->scenes.push_back({device, dev});
    return dev;
}

// The reference draws fresh `rand` values on every call (camera.rs:47-48, photon.rs:18-24), and main.rs:199-217 relies on
// that: it calls partial_render_scene over and over and merge_tile()s the results so the image converges.  The
// counter-based generator here is a pure function of (seed, pixel, sample index), so "fresh" means a sample index no
// earlier call of this process has used: the same-signature overload takes its indices from one process-wide counter.
// Reproducible renders go through the RenderOptions overload, which says which indices to use.
uint64_t next_sample_index(uint64_t count) {
    static std::atomic<uint64_t> counter{0};
    return counter.fetch_add(count, std::memory_order_relaxed);
}

AccumulationBuffer partial_render_scene(const Scene &scene, Tile tile, size_t height, size_t width) {
    RenderOptions o;
    o.sample_offset = next_sample_index(o.spp);
    return partial_render_scene(scene, tile, height, width, o);
}

AccumulationBuffer partial_render_scene(const Scene &scene, Tile tile, size_t height, size_t width, const RenderOptions &o) {
    // every element is overwritten by the copies out of vrj_render_tile (which returns early, writing nothing, for 0 spp)
    AccumulationBuffer buffer = o.spp ? AccumulationBuffer(tile.width(), tile.height(), AccumulationBuffer::Uninitialized{}, o.kahan_state)
                                      : AccumulationBuffer(tile.width(), tile.height());
    VrjRenderParams p{};
    p.spp = o.spp, p.max_depth = o.max_depth, p.sample_offset = o.sample_offset, p.seed = o.seed;
    p.integrator = o.integrator, p.bvh_filter = o.bvh_filter, p.bias = 0.0000001, p.sample_stride = o.sample_stride;
    auto as_data = [](const Spectrum &s) {
        return VrjSpectrumData{s.shortest_wavelength, s.longest_wavelength, (uint32_t)s.samples.size(), 0u, s.samples.data()};
    };
    std::vector<VrjLight> lights;
    VrjSpectrumData ambient = as_data(o.ambient_light);
    if (o.integrator == VRJ_INTEGRATOR_WHITTED) { // WhittedIntegrator { ambient_light, lights }
        for (const DirectionalLight &l : o.lights) {
            VrjLight d{};
            d.direction[0] = l.direction.x, d.direction[1] = l.direction.y, d.direction[2] = l.direction.z;
            d.spectrum = as_data(l.spectrum);
            lights.push_back(d);
        }
        p.lights = lights.data(), p.n_lights = (uint32_t)lights.size(), p.ambient_light = &ambient;
    }
    const VrjScene *dev = device_scene(scene, o.device);
    VrjTile t{tile.start_column, tile.end_column, tile.start_row, tile.end_row};
    VrjAccumOut out{};
    out.memory = VRJ_MEM_HOST;
    out.colour = buffer.colour.data();
    const bool full_state = !buffer.colour_sum.empty();
    if (full_state) out.weight = buffer.weight.data(), out.colour_sum = buffer.colour_sum.data(), out.colour_bias = buffer.colour_bias.data(), out.weight_bias = buffer.weight_bias.data();
    out.stats = o.stats;
    if (vrj_render_tile(dev, &t, height, width, &p, &out) != VRJ_OK) throw std::runtime_error(std::string("vrj_render_tile: ") + vrj_last_error());
    // A fresh buffer's weight is known without asking the device: every sample, hit or miss, enters update_pixel with weight
    // 1.0 (camera.rs:121-127) and a sum of spp ones is exact, so the colour-only buffer brings back the colours alone
    if (!full_state) buffer.uniform_weight = (double)o.spp;
    return buffer;
}

// ------------------------------------------------------------------------------ main.rs:192-217
MainLoopStats render_like_main(const Scene &scene, size_t width, size_t height, size_t tile_size, uint64_t calls, unsigned workers,
                               const RenderOptions &options, bool fresh_samples, AccumulationBuffer &rendered_image) {
    if (rendered_image.width() != width || rendered_image.height() != height) throw std::runtime_error("render_like_main: image size mismatch");
    std::vector<Tile> tiles;
    {
        TileIterator it(width, height, tile_size);
        Tile t;
        while (it.next(t)) tiles.push_back(t);
    }
    MainLoopStats total;
    if (tiles.empty() || calls == 0) return total;
    workers = std::max(1u, workers);
    device_scene(scene, options.device); // flatten + upload before the clock starts (main.rs builds the scene first)
    {
        // The buffers partial_render_scene returns live in pooled page-locked memory.  Up to three per worker exist at the same
        // moment (being rendered, waiting in the channel, being merged); growing the pool costs ~40 ms of cudaMallocHost per
        // buffer during which the device cannot be fed, so the pool is brought to that size once, before the loop starts.
        std::vector<AccumulationBuffer> warm;
        const size_t want = (size_t)std::min<uint64_t>(calls, 3ull * workers);
        for (size_t i = 0; i < want; i++) warm.push_back(AccumulationBuffer(tiles[0].width(), tiles[0].height(), AccumulationBuffer::Uninitialized{}, options.kahan_state));
    }
    struct Item {
        Tile tile;
        AccumulationBuffer buffer;
    };
    std::mutex m;
    std::condition_variable ready, room;
    std::vector<std::unique_ptr<Item>> queue; // the mpsc channel of main.rs:195, bounded so finished tiles cannot pile up
    std::atomic<uint64_t> next{0};
    std::string error;
    unsigned live = workers;
    uint64_t pending = 0; // calls a worker has started and not yet delivered (guarded by m)
    const auto t0 = std::chrono::steady_clock::now();
    auto seconds = [](std::chrono::steady_clock::time_point a) { return std::chrono::duration<double>(std::chrono::steady_clock::now() - a).count(); };
    std::vector<std::thread> pool;
    for (unsigned w = 0; w < workers; w++) {
        pool.emplace_back([&]() {
            double my_call = 0, my_ms = 0;
            uint64_t my_rays = 0, my_calls = 0, my_bytes = 0, my_shared = 0;
            try {
                for (;;) {
                    const uint64_t k = next.fetch_add(1);
                    if (k >= calls) break;
                    {
                        std::lock_guard<std::mutex> lock(m);
                        pending++;
                    }
                    const Tile tile = tiles[k % tiles.size()]; // .cycle()
                    RenderOptions o = options;
                    VrjStats stats{};
                    o.stats = &stats;
                    o.sample_offset = fresh_samples ? next_sample_index(o.spp) : options.sample_offset + (k / tiles.size()) * (uint64_t)o.spp * o.sample_stride;
                    const auto tc = std::chrono::steady_clock::now();
                    std::unique_ptr<Item> item(new Item{tile, partial_render_scene(scene, tile, height, width, o)});
                    my_call += seconds(tc);
                    my_rays += stats.primary_rays + stats.bounce_rays + stats.shadow_rays, my_ms += stats.device_ms, my_calls++, my_shared += stats.coalesced_calls;
                    // what crossed PCIe: all five arrays, or the colours alone (the weights of a colour-and-weight-only buffer are written on the host)
                    my_bytes += 8 * (item->buffer.colour_sum.empty() ? item->buffer.colour.size()
                                                                      : item->buffer.colour.size() + item->buffer.colour_sum.size() + item->buffer.colour_bias.size() +
                                                                            item->buffer.weight.size() + item->buffer.weight_bias.size());
                    std::unique_lock<std::mutex> lock(m);
                    room.wait(lock, [&] { return queue.size() < workers || !error.empty(); });
                    pending--;
                    if (!error.empty()) break;
                    queue.push_back(std::move(item));
                    ready.notify_one();
                }
            } catch (const std::exception &e) { // partial_render_scene threw: its call was counted in `pending`
                std::lock_guard<std::mutex> lock(m);
                pending--;
                if (error.empty()) error = e.what();
            }
            std::lock_guard<std::mutex> lock(m);
            total.call_s += my_call, total.device_ms += my_ms, total.rays += my_rays, total.calls += my_calls, total.bytes_to_host += my_bytes, total.wavefront_calls += my_shared;
            live--;
            ready.notify_one();
            room.notify_all();
        });
    }
    for (;;) { // the 'running loop of main.rs:211-218 without the window
        // `for message in tile_rx.try_iter()` (main.rs:215): everything that is waiting is taken; messages for the same tile are
        // merged in arrival order in one pass over the frame (merge_tiles == consecutive merge_tile calls, bit for bit)
        // main.rs sleeps 1/60 s between two drains of the channel (main.rs:242), so its passes always find many messages.
        // Here the thread does not sleep; it waits until a few messages are there -- as long as calls that will deliver one
        // are still in flight -- because one pass over the frame per message costs twice the memory traffic of one pass per
        // four (the frame's 133 MB are read and written once per pass).
        const size_t want = std::max<size_t>(1, std::min<size_t>(4, workers / 2));
        std::vector<std::unique_ptr<Item>> items;
        {
            std::unique_lock<std::mutex> lock(m);
            ready.wait(lock, [&] { return queue.size() >= want || (!queue.empty() && pending == 0) || live == 0 || !error.empty(); });
            if (queue.empty()) {
                if (live == 0) break;
                continue; // an error is on its way: the workers are leaving
            }
            items.swap(queue);
            room.notify_all();
        }
        const auto tm = std::chrono::steady_clock::now();
        for (size_t i = 0; i < items.size();) {
            std::vector<const AccumulationBuffer *> same{&items[i]->buffer};
            size_t j = i + 1;
            const Tile &t = items[i]->tile;
            for (; j < items.size() && same.size() < 8; j++) {
                const Tile &u = items[j]->tile;
                if (u.start_column != t.start_column || u.end_column != t.end_column || u.start_row != t.start_row || u.end_row != t.end_row) break;
                same.push_back(&items[j]->buffer);
            }
            rendered_image.merge_tiles(t, same);
            total.merge_passes++;
            i = j;
        }
        total.merge_s += seconds(tm);
    }
    for (auto &t : pool) t.join();
    total.wall_s = seconds(t0);
    if (!error.empty()) throw std::runtime_error("render_like_main: " + error);
    return total;
}

// ------------------------------------------------------------------------------ device-resident frame
DeviceAccumulationBuffer::DeviceAccumulationBuffer(size_t width, size_t height, int device) : width_(width), height_(height), device_(device) {
    const size_t n = width * height;
    colour_ = static_cast<double *>(vrj_alloc_device(device, 3 * n * 8)), sum_ = static_cast<double *>(vrj_alloc_device(device, 3 * n * 8));
    bias_ = static_cast<double *>(vrj_alloc_device(device, 3 * n * 8)), weight_ = static_cast<double *>(vrj_alloc_device(device, n * 8));
    weight_bias_ = static_cast<double *>(vrj_alloc_device(device, n * 8)), srgb8_ = static_cast<uint8_t *>(vrj_alloc_device(device, 3 * n));
    if (!colour_ || !sum_ || !bias_ || !weight_ || !weight_bias_ || !srgb8_) {
        const std::string why = vrj_last_error();
        this->~DeviceAccumulationBuffer();
        throw std::runtime_error("DeviceAccumulationBuffer: " + why);
    }
}
DeviceAccumulationBuffer::~DeviceAccumulationBuffer() {
    for (void *p : {(void *)colour_, (void *)sum_, (void *)bias_, (void *)weight_, (void *)weight_bias_, (void *)srgb8_}) vrj_free_device(p);
    colour_ = sum_ = bias_ = weight_ = weight_bias_ = nullptr, srgb8_ = nullptr;
}
// VrjRenderParams of RenderOptions for the device-resident buffers; the lights it points to live in this object
struct DeviceRenderParams {
    VrjRenderParams p{};
    std::vector<VrjLight> lights;
    VrjSpectrumData ambient{};
    explicit DeviceRenderParams(const RenderOptions &o) {
        p.spp = o.spp, p.max_depth = o.max_depth, p.sample_offset = o.sample_offset, p.seed = o.seed;
        p.integrator = o.integrator, p.bvh_filter = o.bvh_filter, p.bias = 0.0000001, p.sample_stride = o.sample_stride;
        auto as_data = [](const Spectrum &s) {
            return VrjSpectrumData{s.shortest_wavelength, s.longest_wavelength, (uint32_t)s.samples.size(), 0u, s.samples.data()};
        };
        ambient = as_data(o.ambient_light);
        if (o.integrator == VRJ_INTEGRATOR_WHITTED) {
            for (const DirectionalLight &l : o.lights) {
                VrjLight d{};
                d.direction[0] = l.direction.x, d.direction[1] = l.direction.y, d.direction[2] = l.direction.z;
                d.spectrum = as_data(l.spectrum);
                lights.push_back(d);
            }
            p.lights = lights.data(), p.n_lights = (uint32_t)lights.size(), p.ambient_light = &ambient;
        }
    }
    DeviceRenderParams(const DeviceRenderParams &) = delete;
};

void DeviceAccumulationBuffer::render(const Scene &scene, RenderOptions o) {
    DeviceRenderParams dp(o);
    VrjRenderParams &p = dp.p;
    p.sample_offset = o.sample_offset + samples_ * o.sample_stride;
    VrjTile t{0, width_, 0, height_};
    VrjAccumOut out{};
    out.memory = VRJ_MEM_DEVICE, out.accumulate = 1; // continue the Kahan state left by the previous pass (zero at first)
    out.colour = colour_, out.colour_sum = sum_, out.colour_bias = bias_, out.weight = weight_, out.weight_bias = weight_bias_;
    out.stats = o.stats;
    if (vrj_render_tile(device_scene(scene, device_), &t, height_, width_, &p, &out) != VRJ_OK)
        throw std::runtime_error(std::string("vrj_render_tile: ") + vrj_last_error());
    samples_ += o.spp;
}
ImageRgbU8 DeviceAccumulationBuffer::to_image_rgb_u8() const {
    ImageRgbU8 image(width_, height_);
    const size_t n = width_ * height_;
    if (vrj_tone_map(device_, VRJ_MEM_DEVICE, VRJ_TONEMAP_XYZ, colour_, n, srgb8_) != VRJ_OK ||
        vrj_copy_to_host(device_, image.pixel_data().data(), srgb8_, 3 * n) != VRJ_OK)
        throw std::runtime_error(std::string("DeviceAccumulationBuffer::to_image_rgb_u8: ") + vrj_last_error());
    return image;
}
AccumulationBuffer DeviceAccumulationBuffer::download() const {
    AccumulationBuffer b(width_, height_, AccumulationBuffer::Uninitialized{});
    const size_t n = width_ * height_;
    const struct {
        double *dst;
        const double *src;
        size_t count;
    } copies[5] = {{b.colour.data(), colour_, 3 * n}, {b.colour_sum.data(), sum_, 3 * n}, {b.colour_bias.data(), bias_, 3 * n},
                   {b.weight.data(), weight_, n}, {b.weight_bias.data(), weight_bias_, n}};
    for (const auto &c : copies)
        if (vrj_copy_to_host(device_, c.dst, c.src, c.count * 8) != VRJ_OK) throw std::runtime_error(std::string("vrj_copy_to_host: ") + vrj_last_error());
    return b;
}

DeviceProgressiveBuffer::DeviceProgressiveBuffer(size_t width, size_t height, int device) : width_(width), height_(height), device_(device) {
    const size_t n = width * height;
    auto f64 = [device](size_t count) { return static_cast<double *>(vrj_alloc_device(device, count * 8)); };
    colour_ = f64(3 * n), sum_ = f64(3 * n), bias_ = f64(3 * n), weight_ = f64(n), weight_bias_ = f64(n), y_sq_sum_ = f64(n);
    normal_ = f64(3 * n), depth_ = f64(n), denoised_ = f64(3 * n);
    material_ = static_cast<int32_t *>(vrj_alloc_device(device, n * 4)), srgb8_ = static_cast<uint8_t *>(vrj_alloc_device(device, 3 * n));
    counts_ = static_cast<uint32_t *>(vrj_alloc_device(device, n * 4));
    if (!colour_ || !sum_ || !bias_ || !weight_ || !weight_bias_ || !y_sq_sum_ || !normal_ || !depth_ || !denoised_ || !material_ || !srgb8_ ||
        !counts_) {
        const std::string why = vrj_last_error();
        this->~DeviceProgressiveBuffer();
        throw std::runtime_error("DeviceProgressiveBuffer: " + why);
    }
}
DeviceProgressiveBuffer::~DeviceProgressiveBuffer() {
    for (void *p : {(void *)colour_, (void *)sum_, (void *)bias_, (void *)weight_, (void *)weight_bias_, (void *)y_sq_sum_, (void *)normal_,
                    (void *)depth_, (void *)denoised_, (void *)material_, (void *)srgb8_, (void *)counts_})
        vrj_free_device(p);
    colour_ = sum_ = bias_ = weight_ = weight_bias_ = y_sq_sum_ = normal_ = depth_ = denoised_ = nullptr;
    material_ = nullptr, srgb8_ = nullptr, counts_ = nullptr;
}
void DeviceProgressiveBuffer::render(const Scene &scene, const RenderOptions &o, const ProgressiveOptions &pp) {
    DeviceRenderParams dp(o);
    dp.p.spp = 0;
    VrjProgressiveParams vp{pp.min_samples, pp.max_samples, pp.pass_samples, pp.max_passes, pp.rel_error, pp.abs_floor};
    VrjTile t{0, width_, 0, height_};
    VrjAccumOut out{};
    out.memory = VRJ_MEM_DEVICE, out.accumulate = started_ ? 1u : 0u;
    out.colour = colour_, out.colour_sum = sum_, out.colour_bias = bias_, out.weight = weight_, out.weight_bias = weight_bias_;
    out.stats = o.stats;
    if (vrj_render_progressive(device_scene(scene, device_), &t, height_, width_, &dp.p, &vp, &out, y_sq_sum_, pp.stats) != VRJ_OK)
        throw std::runtime_error(std::string("vrj_render_progressive: ") + vrj_last_error());
    started_ = true;
}
VrjPlanStats DeviceProgressiveBuffer::plan_counts(const ProgressiveOptions &pp) {
    // a buffer that has not rendered yet holds the zero state (vrj_alloc_device zero-fills): its plan is the uniform pilot
    const VrjAdaptiveParams rule{pp.min_samples, pp.max_samples, pp.pass_samples, 0u, pp.rel_error, pp.abs_floor};
    VrjPlanStats ps{};
    if (vrj_plan_counts(device_, VRJ_MEM_DEVICE, width_ * height_, weight_, sum_, y_sq_sum_, &rule, counts_, &ps) != VRJ_OK)
        throw std::runtime_error(std::string("vrj_plan_counts: ") + vrj_last_error());
    return ps;
}
VrjCountsStats DeviceProgressiveBuffer::render_counts(const Scene &scene, const RenderOptions &o, const uint32_t *counts) {
    DeviceRenderParams dp(o);
    dp.p.spp = 0;
    VrjTile t{0, width_, 0, height_};
    VrjAccumOut out{};
    out.memory = VRJ_MEM_DEVICE, out.accumulate = started_ ? 1u : 0u;
    out.colour = colour_, out.colour_sum = sum_, out.colour_bias = bias_, out.weight = weight_, out.weight_bias = weight_bias_;
    out.stats = o.stats;
    VrjCountsStats cs{};
    if (vrj_render_counts(device_scene(scene, device_), &t, height_, width_, &dp.p, counts ? counts : counts_, &out, y_sq_sum_, &cs) != VRJ_OK)
        throw std::runtime_error(std::string("vrj_render_counts: ") + vrj_last_error());
    started_ = true;
    return cs;
}
ImageRgbU8 DeviceProgressiveBuffer::to_image_rgb_u8() const {
    ImageRgbU8 image(width_, height_);
    const size_t n = width_ * height_;
    if (vrj_tone_map(device_, VRJ_MEM_DEVICE, VRJ_TONEMAP_XYZ, colour_, n, srgb8_) != VRJ_OK ||
        vrj_copy_to_host(device_, image.pixel_data().data(), srgb8_, 3 * n) != VRJ_OK)
        throw std::runtime_error(std::string("DeviceProgressiveBuffer::to_image_rgb_u8: ") + vrj_last_error());
    return image;
}
ImageRgbU8 DeviceProgressiveBuffer::denoised_image_rgb_u8(const Scene &scene, const RenderOptions &options) {
    if (!have_aux_) {
        DeviceRenderParams dp(options);
        VrjTile t{0, width_, 0, height_};
        VrjAuxOut aux{};
        aux.memory = VRJ_MEM_DEVICE, aux.normal = normal_, aux.depth = depth_, aux.material = material_;
        if (vrj_render_aux(device_scene(scene, device_), &t, height_, width_, &dp.p, &aux) != VRJ_OK)
            throw std::runtime_error(std::string("vrj_render_aux: ") + vrj_last_error());
        have_aux_ = true;
    }
    const VrjDenoiseParams params{VRJ_DENOISE_DEFAULT_ITERATIONS, 0u, VRJ_DENOISE_DEFAULT_SIGMA_LUMINANCE, VRJ_DENOISE_DEFAULT_SIGMA_NORMAL,
                                  VRJ_DENOISE_DEFAULT_SIGMA_DEPTH};
    ImageRgbU8 image(width_, height_);
    if (vrj_denoise(device_, VRJ_MEM_DEVICE, width_, height_, sum_, weight_, y_sq_sum_, normal_, depth_, material_, &params, denoised_, srgb8_,
                    nullptr) != VRJ_OK ||
        vrj_copy_to_host(device_, image.pixel_data().data(), srgb8_, 3 * width_ * height_) != VRJ_OK)
        throw std::runtime_error(std::string("DeviceProgressiveBuffer::denoised_image_rgb_u8: ") + vrj_last_error());
    return image;
}
AccumulationBuffer DeviceProgressiveBuffer::download() const {
    AccumulationBuffer b(width_, height_, AccumulationBuffer::Uninitialized{});
    const size_t n = width_ * height_;
    const struct {
        double *dst;
        const double *src;
        size_t count;
    } copies[5] = {{b.colour.data(), colour_, 3 * n}, {b.colour_sum.data(), sum_, 3 * n}, {b.colour_bias.data(), bias_, 3 * n},
                   {b.weight.data(), weight_, n}, {b.weight_bias.data(), weight_bias_, n}};
    for (const auto &c : copies)
        if (vrj_copy_to_host(device_, c.dst, c.src, c.count * 8) != VRJ_OK) throw std::runtime_error(std::string("vrj_copy_to_host: ") + vrj_last_error());
    return b;
}
std::vector<double> DeviceProgressiveBuffer::download_y_sq_sum() const {
    std::vector<double> q(width_ * height_);
    if (vrj_copy_to_host(device_, q.data(), y_sq_sum_, q.size() * 8) != VRJ_OK) throw std::runtime_error(std::string("vrj_copy_to_host: ") + vrj_last_error());
    return q;
}

} // namespace vanrijn
