// vanrijn.hpp -- C++ host-side mirror of the reference's library API for the render loop.
//
// The reference is a Rust crate and the Rust toolchain is not available in the build image, so
// the host side above the C ABI (include/vanrijn_cuda.h) is written in C++ with the reference's
// names, argument meaning and error behaviour; INTEGRATION.md shows the equivalent Rust binding.
// Paths below are relative to /root/reference/src/.
//
//   vanrijn::Scene                       scene.rs:5-8
//   vanrijn::Sphere / Plane / Triangle   raycasting/{sphere,plane,triangle}.rs
//   vanrijn::BoundingVolumeHierarchy     raycasting/bounding_volume_hierarchy.rs:18-75 (median split)
//   vanrijn::PrimitiveList               Vec<Box<dyn Primitive>> (raycasting/vec_aggregate.rs)
//   vanrijn::{Lambertian,Phong,Reflective}Material, SmoothTransparentDialectric   materials/*.rs
//   vanrijn::Spectrum, ColourRgbF, NamedColour                                    colour/*.rs
//   vanrijn::Tile, TileIterator          util/tile_iterator.rs
//   vanrijn::AccumulationBuffer          accumulation_buffer.rs:6-85
//   vanrijn::load_obj                    mesh.rs:74-88
//   vanrijn::partial_render_scene        camera.rs:95-130  <- the drop-in entry point
//
// Types are unchanged in meaning; the only additions are the `flatten` hooks that emit the
// 16-byte-aligned SoA layout uploaded once per scene (the "one additive trait method" of
// SURVEY.md section 7), and RenderOptions for the parameters the reference hard-codes.
#ifndef VANRIJN_HPP
#define VANRIJN_HPP

#include <array>
#include <cstdint>
#include <cstdlib>
#include <memory>
#include <stdexcept>
#include <new>
#include <string>
#include <utility>
#include <vector>

#include "vanrijn_cuda.h"

namespace vanrijn {

struct Vec3 {
    double x = 0, y = 0, z = 0;
    Vec3() = default;
    Vec3(double x_, double y_, double z_) : x(x_), y(y_), z(z_) {}
};

enum class NamedColour { Black, White, Red, Lime, Blue, Yellow, Cyan, Magenta, Gray, Maroon, Olive, Green, Purple, Teal, Navy };

struct ColourRgbF {
    double red = 0, green = 0, blue = 0;
    ColourRgbF() = default;
    ColourRgbF(double r, double g, double b) : red(r), green(g), blue(b) {}
    static ColourRgbF from_named(NamedColour name); // colour/colour_rgb.rs:17-35
};

// colour/spectrum.rs:6-176 -- uniform samples over [shortest, longest]
struct Spectrum {
    double shortest_wavelength = 380.0, longest_wavelength = 740.0;
    std::vector<double> samples;
    static Spectrum black();
    static Spectrum grey(double brightness);
    static Spectrum diamond_index_of_refraction();
    static Spectrum reflection_from_linear_rgb(const ColourRgbF &colour);
};

class FlatSceneBuilder;

// materials/mod.rs:25-34.  The BSDFs themselves run on the device; the host objects carry parameters.
struct Material {
    virtual ~Material() = default;
    virtual uint32_t flatten(FlatSceneBuilder &out) const = 0; // returns the material index
};
struct LambertianMaterial : Material {
    Spectrum colour;
    double diffuse_strength = 1.0;
    LambertianMaterial(Spectrum c, double d) : colour(std::move(c)), diffuse_strength(d) {}
    uint32_t flatten(FlatSceneBuilder &out) const override;
};
struct PhongMaterial : Material {
    Spectrum colour;
    double diffuse_strength, specular_strength, smoothness;
    PhongMaterial(Spectrum c, double d, double s, double sm) : colour(std::move(c)), diffuse_strength(d), specular_strength(s), smoothness(sm) {}
    uint32_t flatten(FlatSceneBuilder &out) const override;
};
struct ReflectiveMaterial : Material {
    Spectrum colour;
    double diffuse_strength, reflection_strength;
    ReflectiveMaterial(Spectrum c, double d, double r) : colour(std::move(c)), diffuse_strength(d), reflection_strength(r) {}
    uint32_t flatten(FlatSceneBuilder &out) const override;
};
struct SmoothTransparentDialectric : Material {
    Spectrum eta;
    explicit SmoothTransparentDialectric(Spectrum e) : eta(std::move(e)) {}
    uint32_t flatten(FlatSceneBuilder &out) const override;
};

// raycasting/mod.rs:135-142
struct Primitive {
    virtual ~Primitive() = default;
    // append this primitive as a top-level traversal item of object `object_id`
    virtual void flatten(FlatSceneBuilder &out, uint32_t object_id, uint32_t prim_id) const = 0;
};
struct Sphere : Primitive {
    Vec3 centre;
    double radius;
    std::shared_ptr<Material> material;
    Sphere(Vec3 c, double r, std::shared_ptr<Material> m) : centre(c), radius(r), material(std::move(m)) {}
    void flatten(FlatSceneBuilder &out, uint32_t object_id, uint32_t prim_id) const override;
};
struct Plane : Primitive {
    Vec3 normal, tangent, cotangent;
    double distance_from_origin;
    std::shared_ptr<Material> material;
    Plane(Vec3 normal, double distance_from_origin, std::shared_ptr<Material> m); // plane.rs:17-32
    void flatten(FlatSceneBuilder &out, uint32_t object_id, uint32_t prim_id) const override;
};
struct Triangle : Primitive {
    std::array<Vec3, 3> vertices, normals;
    std::shared_ptr<Material> material;
    Triangle(std::array<Vec3, 3> v, std::array<Vec3, 3> n, std::shared_ptr<Material> m) : vertices(v), normals(n), material(std::move(m)) {}
    void flatten(FlatSceneBuilder &out, uint32_t object_id, uint32_t prim_id) const override;
};

// raycasting/mod.rs:144-145
struct Aggregate {
    virtual ~Aggregate() = default;
    virtual void flatten(FlatSceneBuilder &out, uint32_t object_id) const = 0;
};
// Vec<Box<dyn Primitive>> as an Aggregate (vec_aggregate.rs:11-24)
struct PrimitiveList : Aggregate {
    std::vector<std::shared_ptr<Primitive>> primitives;
    void flatten(FlatSceneBuilder &out, uint32_t object_id) const override;
};
// The triangles of a mesh as plain arrays: 9 doubles per triangle (v0 xyz, v1 xyz, v2 xyz), normals likewise.
// What mesh.rs:13-72 computes, before it is wrapped into one Arc<dyn Primitive> per triangle.
struct TriangleMesh {
    std::vector<double> vertices, normals;
    size_t triangle_count() const { return vertices.size() / 9; }
};

// bounding_volume_hierarchy.rs:18-75.  Only triangles may be stored (what load_obj produces).
class BoundingVolumeHierarchy : public Aggregate {
  public:
    // Where the recursion of bounding_volume_hierarchy.rs:49-75 runs.  All three produce the same tree (same boxes,
    // node numbering and leaf order).  Device calls vrj_bvh_build and throws if there is no GPU.  AtUpload keeps only
    // the triangles: the tree is built on the GPU when the scene is uploaded (vrj_scene_create, VrjBvh.n_nodes == 0)
    // and never exists on the host, so -- unlike the reference's build(&mut [..]) -- `primitives` is NOT reordered.
    enum class Builder { Host, Device, AtUpload };
    // reorders `primitives` in place, as the reference's build(&mut [Arc<dyn Primitive>]) does
    static std::unique_ptr<BoundingVolumeHierarchy> build(std::vector<std::shared_ptr<Primitive>> &primitives,
                                                          Builder builder = Builder::Host, int device = 0);
    // the same tree straight from arrays (load_obj_mesh), without one heap object per triangle: a 10 M-triangle scene
    // spends seconds in those allocations alone
    static std::unique_ptr<BoundingVolumeHierarchy> build(const TriangleMesh &mesh, std::shared_ptr<Material> material,
                                                          Builder builder = Builder::Host, int device = 0);
    void flatten(FlatSceneBuilder &out, uint32_t object_id) const override;
    uint32_t depth() const { return depth_; }
    size_t triangle_count() const { return tri_v_.size() / 9; }

  private:
    friend class FlatSceneBuilder;
    std::vector<uint32_t> build_arrays(const std::vector<double> &v, const std::vector<double> &n, Builder builder, int device);
    std::vector<double> tri_v_, tri_n_;       // 9 doubles per triangle, leaf (DFS) order
    std::vector<uint32_t> tri_prim_id_;       // original index of each triangle
    std::vector<std::shared_ptr<Material>> tri_material_;
    std::vector<double> node_min_, node_max_; // 3 per node, DFS pre-order
    std::vector<int32_t> node_child_;         // 2 per node, indices local to this BVH
    uint32_t depth_ = 0;
};

// A VrjSceneDesc that owns its arrays: what the scene cache file holds (SURVEY 8f N3, "on-disk cache of the flattened scene").
class FlatScene {
  public:
    explicit FlatScene(const VrjSceneDesc &desc); // deep copy
    FlatScene(FlatScene &&) = default;            // (desc() points into the vectors: movable, not copyable)
    FlatScene(const FlatScene &) = delete;
    static FlatScene load(const std::string &filename); // throws std::runtime_error on a missing, truncated or corrupt file
    void save(const std::string &filename) const;
    const VrjSceneDesc &desc() const { return desc_; }

  private:
    FlatScene() = default;
    void bind();
    std::vector<VrjSpectrum> spectra_;
    std::vector<double> samples_;
    std::vector<VrjMaterial> materials_;
    std::vector<VrjSphere> spheres_;
    std::vector<VrjPlane> planes_;
    std::vector<VrjBvh> bvhs_;
    std::vector<VrjItem> items_;
    std::vector<double> tri_[6], node_min_, node_max_;
    std::vector<uint32_t> tri_material_, tri_prim_id_;
    std::vector<int32_t> node_child_;
    VrjSceneDesc desc_{};
};

// scene.rs:5-8
struct Scene {
    Vec3 camera_location;
    std::vector<std::unique_ptr<Aggregate>> objects;
    // set by load_scene_cache: the flattened form read from disk; `objects` is then empty and the scene can only be rendered
    std::shared_ptr<const FlatScene> flattened;
    Scene() = default;
    Scene(Scene &&) = default;
    Scene &operator=(Scene &&) = default;
    ~Scene();
    // device copy, created on first use and reused (the scene is immutable while it renders)
    struct DeviceCache;
    mutable std::shared_ptr<DeviceCache> device_cache;
};

// util/tile_iterator.rs:2-67
struct Tile {
    size_t start_column, end_column, start_row, end_row;
    size_t width() const { return end_column - start_column; }
    size_t height() const { return end_row - start_row; }
};
class TileIterator {
  public:
    TileIterator(size_t total_width, size_t total_height, size_t tile_size);
    bool next(Tile &tile);

  private:
    size_t tile_size_, total_height_, total_width_, current_column_ = 0, current_row_ = 0;
};

// Allocator of the big host arrays that cross PCIe (the flattened scene, AccumulationBuffer): page-locked memory from
// the library's pool (vrj_alloc_host) when a CUDA device is present, so copies run at PCIe speed and are not staged;
// ordinary memory otherwise.  Elements are default-initialised (no zero fill) unless a value is given.
template <typename T>
struct UploadAllocator {
    using value_type = T;
    UploadAllocator() = default;
    template <typename U>
    UploadAllocator(const UploadAllocator<U> &) {}
    T *allocate(size_t n) {
        const size_t bytes = n * sizeof(T) + 64; // 64-byte prefix records which allocator owns the block
        static const bool pageable_only = std::getenv("VRJ_PAGEABLE_ARRAYS") != nullptr; // experiments only
        char *p = pageable_only ? nullptr : static_cast<char *>(vrj_alloc_host(bytes));
        const bool pinned = p != nullptr;
        if (!p) p = static_cast<char *>(::operator new(bytes));
        p[0] = pinned ? 1 : 0;
        return reinterpret_cast<T *>(p + 64);
    }
    void deallocate(T *q, size_t) {
        char *p = reinterpret_cast<char *>(q) - 64;
        if (p[0]) vrj_free_host(p);
        else ::operator delete(p);
    }
    template <typename U>
    void construct(U *p) noexcept { ::new (static_cast<void *>(p)) U; } // vector(n): no zero fill
    template <typename U, typename... Args>
    void construct(U *p, Args &&...args) { ::new (static_cast<void *>(p)) U(std::forward<Args>(args)...); }
    template <typename U>
    bool operator==(const UploadAllocator<U> &) const { return true; }
    template <typename U>
    bool operator!=(const UploadAllocator<U> &) const { return false; }
};
template <typename T>
using UploadVector = std::vector<T, UploadAllocator<T>>;

// image.rs:7-66 -- 8-bit RGB image, row-major, 3 bytes per pixel
class ImageRgbU8 {
  public:
    ImageRgbU8(size_t width, size_t height) : pixel_data_(3 * width * height, 0), width_(width), height_(height) {}
    size_t get_width() const { return width_; }
    size_t get_height() const { return height_; }
    static size_t num_channels() { return 3; }
    const std::vector<uint8_t> &get_pixel_data() const { return pixel_data_; }
    std::vector<uint8_t> &pixel_data() { return pixel_data_; }
    // image.rs:52-66: 8-bit RGB PNG.  Written with stored (uncompressed) deflate blocks: the pixels decode identically,
    // the file is simply larger than the `png` crate's.  Throws std::runtime_error on I/O failure.
    void write_png(const std::string &filename) const;

  private:
    std::vector<uint8_t> pixel_data_;
    size_t width_, height_;
};

// accumulation_buffer.rs:6-85: five row-major arrays
class AccumulationBuffer {
  public:
    AccumulationBuffer(size_t width, size_t height);
    // accumulation_buffer.rs:38-42 with ClampingToneMapper (image.rs:130-187): XYZ -> sRGB (colour_xyz.rs:48-84) ->
    // clamp -> truncating byte, evaluated on the device (vrj_tone_map)
    ImageRgbU8 to_image_rgb_u8(int device = 0) const;
    size_t width() const { return width_; }
    size_t height() const { return height_; }
    // accumulation_buffer.rs:62-85 -- touches only colour and weight of the destination
    void merge_tile(const Tile &tile, const AccumulationBuffer &src);
    // merge_tile(tile, *srcs[0]); merge_tile(tile, *srcs[1]); ... in ONE pass over the destination: per pixel the same
    // operations in the same order (bit-identical), but the frame's colours and weights cross the memory bus once instead
    // of once per buffer -- what main.rs:215-217 does when several messages are waiting in the channel
    void merge_tiles(const Tile &tile, const std::vector<const AccumulationBuffer *> &srcs);
    UploadVector<double> colour, colour_sum, colour_bias; // 3 per pixel (XYZ)
    UploadVector<double> weight, weight_bias;             // 1 per pixel
    // > 0: a buffer rendered with RenderOptions::kahan_state = false -- every pixel carries this weight (the samples per pixel of
    // the call; hit or miss, each sample enters update_pixel with weight 1.0, camera.rs:121-127) and `weight` is left empty
    double uniform_weight = 0.0;

  private:
    friend AccumulationBuffer partial_render_scene(const Scene &, Tile, size_t, size_t, const struct RenderOptions &);
    friend class DeviceAccumulationBuffer;
    friend class DeviceProgressiveBuffer;
    friend struct MainLoopStats render_like_main(const struct Scene &, size_t, size_t, size_t, uint64_t, unsigned, const struct RenderOptions &, bool,
                                                 AccumulationBuffer &);
    struct Uninitialized {};
    AccumulationBuffer(size_t width, size_t height, Uninitialized, bool kahan_state = true); // arrays about to be overwritten by a render
    size_t width_, height_;
};

// mesh.rs:74-88
std::vector<std::shared_ptr<Primitive>> load_obj(const std::string &filename, std::shared_ptr<Material> material);
// the same parse, as arrays (SURVEY 8f N3: OBJ -> SoA without a Rust dependency); load_obj wraps its result
TriangleMesh load_obj_mesh(const std::string &filename);

// The parameters partial_render_scene hard-codes (camera.rs:69,103), made explicit.
struct DirectionalLight {
    Vec3 direction;
    Spectrum spectrum;
};
struct RenderOptions {
    uint32_t spp = 1;
    uint32_t max_depth = 128;
    uint64_t sample_offset = 0;
    uint64_t seed = 1;
    uint32_t integrator = VRJ_INTEGRATOR_SIMPLE_RANDOM;
    uint32_t bvh_filter = VRJ_FILTER_F32;
    uint32_t sample_stride = 1;
    int device = 0;
    // false: the returned buffer carries only `colour` and one weight for all pixels (`uniform_weight`) -- all that merge_tile
    // (accumulation_buffer.rs:62-85) and to_image_rgb_u8 read; the per-pixel weights and the Kahan arrays (8 of the 11 doubles
    // per pixel) stay empty and are not copied back: 50 MB instead of 182 MB per 1080p call.  Such a buffer cannot be continued
    // with update_pixel.
    bool kahan_state = true;
    std::vector<DirectionalLight> lights; // Whitted
    Spectrum ambient_light = Spectrum::black();
    VrjStats *stats = nullptr;
};

// camera.rs:95-100.  Throws std::runtime_error where the reference would panic or when CUDA fails.
// The reference's signature: every call renders a sample nobody has rendered before (the reference draws from an
// OS-seeded generator; here the sample index comes from next_sample_index()), so the main.rs loop -- call, merge_tile,
// repeat -- converges.  For a reproducible render pass RenderOptions with an explicit sample_offset.
AccumulationBuffer partial_render_scene(const Scene &scene, Tile tile, size_t height, size_t width);
// reserves `count` consecutive sample indices of the process-wide sequence and returns the first
uint64_t next_sample_index(uint64_t count = 1);
AccumulationBuffer partial_render_scene(const Scene &scene, Tile tile, size_t height, size_t width, const RenderOptions &options);

// main.rs:192-217 as a function: `workers` threads (the reference: rayon's pool through par_bridge) take the tiles of
// TileIterator(width, height, tile_size) round and round, call partial_render_scene on each and hand the result to the
// calling thread, which merge_tile()s it into `rendered_image` as it arrives (main.rs:214-216).  `options` defaults to what
// the reference hard-codes (1 spp, RECURSION_LIMIT 128); with `fresh_samples` every call takes its sample indices from
// next_sample_index() like the same-signature call, otherwise pass k over the tiles uses options.sample_offset + k * spp.
// Stops after `calls` calls.  At most `workers` finished tiles wait for the merge.
struct MainLoopStats {
    double wall_s = 0, call_s = 0, merge_s = 0, device_ms = 0; // call_s: summed over the workers
    uint64_t rays = 0, calls = 0, bytes_to_host = 0;
    uint64_t merge_passes = 0; // passes over the frame: messages that were waiting together were merged in one (merge_tiles)
    uint64_t wavefront_calls = 0; // sum over the calls of VrjStats.coalesced_calls (/ calls = mean calls per shared wavefront)
};
MainLoopStats render_like_main(const Scene &scene, size_t width, size_t height, size_t tile_size, uint64_t calls, unsigned workers,
                               const RenderOptions &options, bool fresh_samples, AccumulationBuffer &rendered_image);

// The frame's AccumulationBuffer kept in GPU memory between passes (SURVEY 8f N2, "progressive preview").
// main.rs:199-225 merges a freshly downloaded 1-spp buffer per tile into the frame on the host (merge_tile's weighted
// mean) and tone-maps on the host; here every pass continues the Kahan accumulators where the last one stopped
// (= one long sequence of update_pixel calls, accumulation_buffer.rs:44-60) and a preview is 3 bytes per pixel.
class DeviceAccumulationBuffer {
  public:
    DeviceAccumulationBuffer(size_t width, size_t height, int device = 0);
    ~DeviceAccumulationBuffer();
    DeviceAccumulationBuffer(const DeviceAccumulationBuffer &) = delete;
    DeviceAccumulationBuffer &operator=(const DeviceAccumulationBuffer &) = delete;
    size_t width() const { return width_; }
    size_t height() const { return height_; }
    uint64_t samples_per_pixel() const { return samples_; }
    // options.spp more samples per pixel of the whole frame; sample indices continue from the last call
    void render(const Scene &scene, RenderOptions options);
    ImageRgbU8 to_image_rgb_u8() const; // ClampingToneMapper on the device
    AccumulationBuffer download() const; // the five arrays, as partial_render_scene would have produced them in one call

  private:
    double *colour_ = nullptr, *sum_ = nullptr, *bias_ = nullptr, *weight_ = nullptr, *weight_bias_ = nullptr;
    uint8_t *srgb8_ = nullptr;
    size_t width_, height_;
    int device_;
    uint64_t samples_ = 0;
};

// The schedule of vrj_render_progressive (include/vanrijn_cuda.h): pixels below min_samples, and pixels below max_samples
// whose mean Y is not yet within rel_error, take samples; max_passes passes per render() call (0: until none is active).
struct ProgressiveOptions {
    uint32_t min_samples = 4, max_samples = 64, pass_samples = 4;
    uint32_t max_passes = 1;
    double rel_error = 0.05, abs_floor = 0.0;
    VrjProgressiveStats *stats = nullptr; // optional: what the last call did and the state it left
};

// A progressive frame kept on the GPU, sampled adaptively: the AccumulationBuffer's arrays plus the per-pixel sum of
// squared Y (y_sq_sum) that vrj_denoise needs.  Keep options.seed, sample_offset and sample_stride fixed across calls.
class DeviceProgressiveBuffer {
  public:
    DeviceProgressiveBuffer(size_t width, size_t height, int device = 0);
    ~DeviceProgressiveBuffer();
    DeviceProgressiveBuffer(const DeviceProgressiveBuffer &) = delete;
    DeviceProgressiveBuffer &operator=(const DeviceProgressiveBuffer &) = delete;
    size_t width() const { return width_; }
    size_t height() const { return height_; }
    // continues the frame's state with up to pp.max_passes passes (options.spp is ignored: the counts come from pp)
    void render(const Scene &scene, const RenderOptions &options, const ProgressiveOptions &pp);
    // the planned loop (vrj_plan_counts, vrj_render_counts): plan_counts() writes the frame's count map from its state with
    // pp's rule (pp.max_passes is not used) and returns the plan; render_counts() renders that map -- or `counts`, a
    // device map of width * height counts on this buffer's GPU -- in full wavefronts.  Loop until the plan's samples is 0.
    VrjPlanStats plan_counts(const ProgressiveOptions &pp);
    VrjCountsStats render_counts(const Scene &scene, const RenderOptions &options, const uint32_t *counts = nullptr);
    ImageRgbU8 to_image_rgb_u8() const; // ClampingToneMapper on the device
    // vrj_denoise (the header's defaults) of the frame as it stands, on the device; the first-hit features come from one
    // vrj_render_aux of options.spp camera rays per pixel, traced at the first call and kept for the frame
    ImageRgbU8 denoised_image_rgb_u8(const Scene &scene, const RenderOptions &options);
    AccumulationBuffer download() const; // the five arrays
    std::vector<double> download_y_sq_sum() const;

  private:
    double *colour_ = nullptr, *sum_ = nullptr, *bias_ = nullptr, *weight_ = nullptr, *weight_bias_ = nullptr, *y_sq_sum_ = nullptr;
    double *normal_ = nullptr, *depth_ = nullptr, *denoised_ = nullptr;
    int32_t *material_ = nullptr;
    uint32_t *counts_ = nullptr;
    uint8_t *srgb8_ = nullptr;
    size_t width_, height_;
    int device_;
    bool started_ = false, have_aux_ = false;
};

// Collects the flattened SoA arrays and exposes them as a VrjSceneDesc.
class FlatSceneBuilder {
  public:
    uint32_t add_spectrum(const Spectrum &s);
    uint32_t add_material(uint32_t kind, uint32_t spectrum, double p0, double p1, double p2);
    void add_sphere(const Sphere &s, uint32_t material, uint32_t object_id, uint32_t prim_id);
    void add_plane(const Plane &p, uint32_t material, uint32_t object_id, uint32_t prim_id);
    void add_triangle(const Triangle &t, uint32_t material, uint32_t object_id, uint32_t prim_id);
    void add_bvh(const BoundingVolumeHierarchy &bvh, uint32_t object_id);
    const VrjSceneDesc &desc(const Vec3 &camera);
    uint32_t material_index(const Material *m);

  private:
    std::vector<VrjSpectrum> spectra_;
    std::vector<double> samples_;
    std::vector<VrjMaterial> materials_;
    std::vector<std::pair<const Material *, uint32_t>> material_cache_;
    std::vector<VrjSphere> spheres_;
    std::vector<VrjPlane> planes_;
    std::vector<VrjBvh> bvhs_;
    std::vector<VrjItem> items_;
    UploadVector<double> tri_[6];
    UploadVector<uint32_t> tri_material_, tri_prim_id_;
    UploadVector<double> node_min_, node_max_;
    UploadVector<int32_t> node_child_;
    VrjSceneDesc desc_{};
};

// The flattened form of a scene on disk: save once (OBJ parsed, tree built or left to the device), load in milliseconds.
void save_scene_cache(const Scene &scene, const std::string &filename);
Scene load_scene_cache(const std::string &filename);

// Flatten + upload (cached on the scene).  Exposed for callers that want the raw C ABI.
const VrjScene *device_scene(const Scene &scene, int device = 0);

} // namespace vanrijn
#endif
