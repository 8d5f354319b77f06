/*
 * vanrijn_cuda.h -- C ABI of libvanrijn_cuda.so, the B200 (sm_100a) implementation of
 * vanrijn's per-pixel / per-sample render loop.
 *
 * What it replaces in the reference (paths relative to /root/reference/):
 *   vrj_render_tile   <- partial_render_scene(&Scene, Tile, height, width) -> AccumulationBuffer
 *                        src/camera.rs:95-130 (re-exported src/lib.rs:18), called from
 *                        src/main.rs:204 and benches/simple_scene.rs:45
 *   vrj_trace_rays    <- Sampler::sample(&Ray) -> Option<IntersectionInfo>, src/sampler.rs:9-20
 *   vrj_scene_create  <- the flattened form of Scene { camera_location, objects }
 *                        (src/scene.rs:5-8) that the host-side BVH builder
 *                        (src/raycasting/bounding_volume_hierarchy.rs:49-75) and OBJ loader
 *                        (src/mesh.rs:74-88) emit; uploaded once per scene
 *   vrj_bvh_build     <- BoundingVolumeHierarchy::build (bounding_volume_hierarchy.rs:38-75) on the device,
 *                        the same tree bit for bit (also done inside vrj_scene_create for a VrjBvh without nodes)
 *   vrj_tone_map      <- AccumulationBuffer::to_image_rgb_u8 with ClampingToneMapper
 *                        (src/accumulation_buffer.rs:38-42, src/image.rs:130-187)
 *   vrj_comm_* / vrj_render_sharded  <- the per-worker sample passes + merge of src/main.rs:197-217 over several GPUs
 *
 * The reference has no FFI today; INTEGRATION.md shows the Rust `extern "C"` block and the
 * `partial_render_scene_cuda` wrapper a maintainer would add.  Everything here is plain
 * data: pointers, sizes, fixed-width integers and doubles.  No function unwinds; each returns
 * a VrjStatus and leaves a message for vrj_last_error() (thread-local).
 *
 * Numerics: every hit, shading and accumulation operation is IEEE binary64 in the
 * reference's operation order (compiled with -fmad=false).  `bvh_filter` only selects the
 * precision of the conservative box culling in front of the exact triangle test and cannot
 * change a result.
 *
 * Thread safety: a VrjScene is immutable after creation; vrj_render_tile / vrj_trace_rays
 * may be called concurrently from several host threads on one scene (mirrors the rayon
 * use at src/main.rs:197-209); each call uses its own stream and scratch block.  At most a few
 * calls render on one device at the same moment (a FIFO gate; the others' copies back to the
 * host overlap), and small host-memory calls of the reference's kind (SimpleRandom, <= 4 samples,
 * fresh buffer) that queue up behind it and differ only in sample indices and output buffers are
 * rendered as ONE wavefront, each receiving bit for bit the buffer it would have received alone
 * (VrjStats.coalesced_calls).
 */
#ifndef VANRIJN_CUDA_H
#define VANRIJN_CUDA_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define VRJ_ABI_VERSION 2

#if defined(__GNUC__)
#define VRJ_API __attribute__((visibility("default")))
#else
#define VRJ_API
#endif

typedef struct VrjScene VrjScene; /* opaque: one uploaded scene on one GPU */

typedef int32_t VrjStatus;
enum {
    VRJ_OK = 0,
    VRJ_ERR_INVALID_ARGUMENT = 1,
    VRJ_ERR_CUDA = 2,         /* CUDA runtime error, including "no device" -- there is no CPU fallback */
    VRJ_ERR_UNSUPPORTED = 3,
    VRJ_ERR_OUT_OF_MEMORY = 4
};

/* materials/{lambertian,phong,reflective}_material.rs, smooth_transparent_dialectric.rs */
enum { VRJ_MAT_LAMBERTIAN = 0, VRJ_MAT_PHONG = 1, VRJ_MAT_REFLECTIVE = 2, VRJ_MAT_DIELECTRIC = 3 };
/* integrators/simple_random_integrator.rs, integrators/whitted_integrator.rs */
enum { VRJ_INTEGRATOR_SIMPLE_RANDOM = 0, VRJ_INTEGRATOR_WHITTED = 1 };
/* top-level traversal items, in Scene.objects order (sampler.rs:12-19: first object wins ties) */
enum { VRJ_ITEM_SPHERE = 0, VRJ_ITEM_PLANE = 1, VRJ_ITEM_TRIANGLE = 2, VRJ_ITEM_BVH = 3 };
/* precision / shape of the conservative box culling in front of the exact triangle test; results are identical in all modes.
 * F32: 2-wide nodes, f32 boxes; F64: 2-wide, f64 boxes (cross-check); F32X4: 4-wide nodes (two reference levels per fetch);
 * Q16: 2-wide nodes, boxes rounded outward onto a 16-bit grid over the scene's meshes (32-byte nodes, half the bytes per step) */
enum { VRJ_FILTER_F32 = 0, VRJ_FILTER_F64 = 1, VRJ_FILTER_F32X4 = 2, VRJ_FILTER_Q16 = 3 };
enum { VRJ_MEM_HOST = 0, VRJ_MEM_DEVICE = 1 };
/* VRJ_PRECISION_F64: every hit, shading and accumulation operation in binary64, the reference's type and operation order.
 * VRJ_PRECISION_F32_FAST: the same formulas in binary32 (accumulators stay binary64).  The reference has no binary32 build
 * (realtype.rs is f64 everywhere), so this mode has no parity claim: hit ids can differ next to edges and images agree to
 * about 1e-3; it is reported separately (SURVEY 8d "f32 fast"). */
enum { VRJ_PRECISION_F64 = 0, VRJ_PRECISION_F32_FAST = 1 };

/* colour/spectrum.rs:6-10 -- uniform samples over [shortest, longest] */
typedef struct VrjSpectrum {
    double shortest_wavelength, longest_wavelength;
    uint32_t first_sample; /* index into VrjSceneDesc.spectrum_samples */
    uint32_t n_samples;
} VrjSpectrum;

/* p0..p2: Lambertian {diffuse_strength}; Phong {diffuse, specular, smoothness};
 * Reflective {diffuse, reflection_strength}; Dielectric {} with spectrum = eta(lambda) */
typedef struct VrjMaterial {
    uint32_t kind, spectrum;
    double p0, p1, p2;
} VrjMaterial;

/* raycasting/sphere.rs:9-13 */
typedef struct VrjSphere {
    double centre[3];
    double radius;
    uint32_t material, pad;
} VrjSphere;

/* raycasting/plane.rs:9-15, fields as Plane::new (plane.rs:17-32) leaves them */
typedef struct VrjPlane {
    double normal[3], tangent[3], cotangent[3];
    double distance_from_origin;
    uint32_t material, pad;
} VrjPlane;

/* One BoundingVolumeHierarchy (bounding_volume_hierarchy.rs:18-28), flattened:
 * nodes [first_node, first_node+n_nodes) in DFS pre-order (root first),
 * triangles [first_triangle, first_triangle+n_triangles) in leaf (DFS) order.
 * n_nodes == 0 with n_triangles > 0: the caller has not built the tree; vrj_scene_create builds it on the device
 * (the algorithm of vrj_bvh_build: the reference's tree exactly) from the triangles in the order given, and
 * first_node / depth are ignored. */
typedef struct VrjBvh {
    uint64_t first_node, n_nodes;
    uint64_t first_triangle, n_triangles;
    uint32_t depth, pad;
} VrjBvh;

typedef struct VrjItem {
    uint32_t kind;      /* VRJ_ITEM_* */
    uint32_t index;     /* into spheres / planes / triangles / bvhs */
    uint32_t object_id; /* index of the owning element of Scene.objects */
    uint32_t prim_id;   /* index of the primitive inside that object (0 for a BVH item) */
} VrjItem;

/* The flattened scene: 16-byte aligned structure-of-arrays.  The caller keeps ownership of
 * every array; vrj_scene_create copies what it needs to the device. */
typedef struct VrjSceneDesc {
    uint32_t abi_version; /* VRJ_ABI_VERSION */
    uint32_t pad0;
    double camera_location[3];
    double pad1;

    uint32_t n_spectra, n_spectrum_samples;
    const VrjSpectrum *spectra;
    const double *spectrum_samples;

    uint32_t n_materials, n_spheres;
    const VrjMaterial *materials;
    const VrjSphere *spheres;

    uint32_t n_planes, n_bvhs;
    const VrjPlane *planes;
    const VrjBvh *bvhs;

    /* triangles, SoA; each vertex / normal is 4 doubles {x, y, z, 0} (32-byte records) */
    uint64_t n_triangles;
    const double *tri_v0, *tri_v1, *tri_v2;
    const double *tri_n0, *tri_n1, *tri_n2;
    const uint32_t *tri_material;
    const uint32_t *tri_prim_id; /* index in the order the object was handed its primitives */

    /* BVH nodes, SoA; node_min/node_max are 4 doubles {x, y, z, 0};
     * node_child[2i], node_child[2i+1]: internal node = absolute indices of left/right child (>= 0);
     * leaf = { ~first_triangle (absolute, < 0), triangle count (0 or 1) } */
    uint64_t n_nodes;
    const double *node_min, *node_max;
    const int32_t *node_child;

    uint32_t n_items, pad2;
    const VrjItem *items;
} VrjSceneDesc;

/* util/tile_iterator.rs:2-17 -- half-open column / row ranges of the full image */
typedef struct VrjTile {
    uint64_t start_column, end_column, start_row, end_row;
} VrjTile;

/* A Spectrum passed by value in a call (integrator parameters are not scene content) */
typedef struct VrjSpectrumData {
    double shortest_wavelength, longest_wavelength;
    uint32_t n_samples, pad;
    const double *samples;
} VrjSpectrumData;

/* integrators/whitted_integrator.rs:10-13 */
typedef struct VrjLight {
    double direction[3]; /* used un-normalised in the cosine, as the reference does */
    VrjSpectrumData spectrum;
} VrjLight;

typedef struct VrjRenderParams {
    uint32_t spp;             /* samples per pixel in this call; the reference call is 1 (camera.rs:105-128) */
    uint32_t max_depth;       /* RECURSION_LIMIT, camera.rs:69: 128 */
    uint64_t sample_offset;   /* index of the first sample; samples are pure functions of (seed, pixel, index) */
    uint64_t seed;
    uint32_t integrator;      /* VRJ_INTEGRATOR_*; the reference hard-codes SIMPLE_RANDOM (camera.rs:103) */
    uint32_t bvh_filter;      /* VRJ_FILTER_* */
    double bias;              /* 1e-7: simple_random_integrator.rs:42, whitted_integrator.rs:37,57 */
    const VrjLight *lights;   /* WhittedIntegrator.lights (whitted_integrator.rs:15-18) */
    const VrjSpectrumData *ambient_light; /* WhittedIntegrator.ambient_light; NULL = black */
    uint32_t n_lights;
    uint32_t sample_stride;   /* 0 or 1: consecutive samples; G: this call takes samples offset, offset+G, ... (sharding) */
    uint32_t count_traversal; /* non-zero: also count BVH node visits / triangle tests (slower kernel variant) */
    uint32_t precision;       /* VRJ_PRECISION_*; 0 = the reference's binary64 (the parity path) */
} VrjRenderParams;

typedef struct VrjStats {
    uint64_t primary_rays, bounce_rays, shadow_rays; /* Sampler::sample calls, the unit of Mrays/s */
    uint64_t paths_missed, paths_escaped, paths_depth_limited;
    uint64_t node_visits, triangle_tests; /* only when count_traversal != 0 */
    uint64_t kernel_launches;
    double device_ms; /* CUDA-event time of the kernels of this call (first launch .. last launch) */
    /* CUDA-event time per kernel class, summed over the call's launches (events on the launching stream) */
    double primary_ms, bounce_ms, resolve_ms;   /* k_trace (camera rays), k_trace (bounce rays), k_resolve */
    uint64_t primary_launches, bounce_launches, resolve_launches;
    double shade_ms;                            /* k_raygen + k_shade */
    uint64_t shade_launches;
    uint64_t staged_rays;                       /* rays that passed a BVH root pre-test and went through k_trace */
    double tail_ms;                             /* k_tail (all launches, including the no-op ones) */
    uint64_t tail_launches;
    uint64_t coalesced_calls;                   /* calls that shared this call's wavefront (1 = alone).  When > 1 the ray counters
                                                   and times above are this call's even share of the wavefront's totals (sums over
                                                   the calls stay exact); see vrj_render_tile */
} VrjStats;

/* The five arrays of AccumulationBuffer (accumulation_buffer.rs:6-12), tile-local, row-major like
 * Array2D (util/array2d.rs:54-60): tile.height rows of tile.width pixels; XYZ interleaved.
 * Any pointer may be NULL.  `memory` says whether the pointers are host or device memory
 * (device: same GPU as the scene). */
typedef struct VrjAccumOut {
    uint32_t memory; /* VRJ_MEM_* */
    uint32_t accumulate; /* non-zero: colour_sum/colour_bias/weight/weight_bias hold a previous state to continue from */
    double *colour;      /* 3 per pixel: colour_sum * (1/weight) */
    double *colour_sum;  /* 3 per pixel */
    double *colour_bias; /* 3 per pixel (Kahan compensation) */
    double *weight;      /* 1 per pixel */
    double *weight_bias; /* 1 per pixel */
    double *photons;     /* optional debug output: spp * npix * 2 = (wavelength, intensity*360) per sample */
    VrjStats *stats;     /* host memory */
    uint8_t *srgb8;      /* optional: 3 bytes per pixel, ClampingToneMapper applied to `colour` on the device
                            (AccumulationBuffer::to_image_rgb_u8, accumulation_buffer.rs:38-42) -- a preview needs
                            6 MB back instead of the 66 MB of f64 XYZ at 1080p */
} VrjAccumOut;

VRJ_API const char *vrj_last_error(void);
VRJ_API int32_t vrj_abi_version(void);
/* number of CUDA devices visible; 0 (not an error code) when there is none */
VRJ_API int32_t vrj_device_count(void);

/* Upload the flattened scene to `device` (once per scene). */
VRJ_API VrjStatus vrj_scene_create(const VrjSceneDesc *desc, int32_t device, VrjScene **out);
VRJ_API void vrj_scene_destroy(VrjScene *scene);
/* bytes the scene occupies on the device (the traversal layout), and bytes vrj_scene_create copied host->device
 * (the caller's arrays as they are: the traversal layout is formed on the device) */
VRJ_API uint64_t vrj_scene_device_bytes(const VrjScene *scene);
VRJ_API uint64_t vrj_scene_upload_bytes(const VrjScene *scene);

/* Free what the library keeps between calls: the per-device scratch blocks (path queues etc.) and the pooled device and
 * page-locked host memory (freed scenes, buffers and vrj_alloc_host / vrj_alloc_device blocks are kept for reuse because
 * cudaMalloc / cudaFree / cudaMallocHost cost milliseconds each). */
VRJ_API void vrj_release_scratch(void);
/* Page-locked host memory for output arrays (optional: any host pointer works, pinned ones copy faster). */
VRJ_API void *vrj_alloc_host(uint64_t bytes);
VRJ_API void vrj_free_host(void *p);

/* Device memory for output arrays that stay on the GPU between calls (VrjAccumOut.memory = VRJ_MEM_DEVICE with
 * `accumulate`): a progressive renderer then moves 6 MB (srgb8) per preview instead of 182 MB per pass at 1080p.
 * vrj_alloc_device returns zero-filled memory from the library's pool, or NULL. */
VRJ_API void *vrj_alloc_device(int32_t device, uint64_t bytes);
VRJ_API void vrj_free_device(void *p);
VRJ_API VrjStatus vrj_copy_to_host(int32_t device, void *host_dst, const void *device_src, uint64_t bytes);

/* partial_render_scene (src/camera.rs:95-130): render `tile` of a width x height image, params->spp samples per pixel.
 * Blocks until the output arrays are filled.  Safe to call from many threads on one scene; the library schedules the calls:
 * at most a few render on a device at the same moment, and calls of the reference's kind -- VRJ_INTEGRATOR_SIMPLE_RANDOM,
 * 1..4 samples, a fresh (accumulate == 0) host buffer that asks for `colour`, no photons / srgb8 / count_traversal -- that
 * are waiting at that moment and agree in scene, tile, image size, max_depth, seed, bvh_filter, precision, bias,
 * sample_stride and in WHICH arrays they ask for are rendered as one wavefront.  Every such call receives bit for bit the
 * arrays it would have received alone (a sample is a pure function of seed, pixel and sample index, and each call's samples
 * are applied to its own zeroed buffer in sample order); out->stats->coalesced_calls reports how many calls shared the
 * wavefront.  Environment (experiments): VRJ_COALESCE=0, VRJ_CONCURRENT_RENDERS=<n>.
 * VRJ_FILTER_F32 (the default) lets the library take the 16-bit walk for scenes whose f32 nodes exceed L2; no walk can change
 * a result. */
VRJ_API VrjStatus vrj_render_tile(const VrjScene *scene, const VrjTile *tile, uint64_t height, uint64_t width,
                          const VrjRenderParams *params, VrjAccumOut *out);

/* ---- adaptive sampling: per-pixel sample counts set by an on-device noise estimate ----
 * vrj_render_adaptive renders `tile` in passes and stops sampling a pixel once the estimated error of its mean Y is small.
 * A pixel that ends with n samples holds, bit for bit, what vrj_render_tile with spp = n (same seed, sample_offset,
 * sample_stride) gives it: its k-th sample has index sample_offset + k * stride, and samples are applied in sample order.
 *
 * Passes.  Pass 0 gives every pixel samples 0 .. min_samples-1.  After each pass every active pixel is judged; the active
 * pixels that have not converged and hold fewer than max_samples take min(pass_samples, max_samples - n) more in the next
 * pass.  All active pixels hold the same n, so every count is min_samples + j * pass_samples, capped at max_samples.
 *
 * Stopping rule, in binary64 in exactly this order (n = weight, s = colour_sum.y, q = y_sq_sum):
 *     m = s * (1.0 / n);   v = (q - s * m) / (n - 1.0);   if (v < 0) v = 0;
 *     t = rel_error * (m > abs_floor ? m : abs_floor);   converged  iff  v <= t * t * n
 * i.e. the standard error of the mean, sqrt(v / n), is at most rel_error * max(m, abs_floor).  A NaN anywhere fails the
 * test: such a pixel samples until max_samples.
 *
 * y_sq_sum (optional, NULL: not returned): one double per pixel, memory of the kind out->memory says; q = q + y * y over the
 * pixel's samples in sample order, y being exactly the Y value the sample adds to colour_sum.
 * out: the arrays, layout and memory kinds of vrj_render_tile, srgb8 included; out->stats sums the passes (device_ms spans
 * the first to the last kernel, the per-pass readback of the active count -- 4 bytes -- included).  out->accumulate and
 * out->photons: VRJ_ERR_UNSUPPORTED.  params: every field keeps its meaning (integrators, lights, filters, precisions,
 * sample_stride, count_traversal) except spp, which must be 0 (the counts come from `ap`).  astats may be NULL.
 * Scheduling: the call is never coalesced with others; it takes the device's render turn like any other call and uses a
 * scratch block from the pool (16 bytes per pixel more than vrj_render_tile: y_sq_sum and two pixel lists). */
typedef struct VrjAdaptiveParams {
    uint32_t min_samples;   /* every pixel first takes samples 0..min_samples-1; >= 2 */
    uint32_t max_samples;   /* no pixel takes more; >= min_samples */
    uint32_t pass_samples;  /* samples each still-active pixel takes per further pass; >= 1 */
    uint32_t pad;
    double rel_error;       /* > 0, finite */
    double abs_floor;       /* >= 0, finite */
} VrjAdaptiveParams;

typedef struct VrjAdaptiveStats {
    uint64_t passes;              /* including the first (min_samples) pass */
    uint64_t samples;             /* sum over pixels of the samples each received (= sum of weight) */
    uint64_t pixels_converged;    /* stopped by the error rule */
    uint64_t pixels_unconverged;  /* reached max_samples without meeting it */
} VrjAdaptiveStats;

VRJ_API VrjStatus vrj_render_adaptive(const VrjScene *scene, const VrjTile *tile, uint64_t height, uint64_t width,
                                      const VrjRenderParams *params, const VrjAdaptiveParams *ap, VrjAccumOut *out,
                                      double *y_sq_sum, VrjAdaptiveStats *astats);

/* Sampler::sample on n rays (host arrays, 3 doubles each; directions are normalised like Ray::new).
 * object_id / prim_id are -1 and t is +inf on a miss. */
/* ---- one box, several GPUs (SURVEY 8e): shard by sample index, one NCCL reduce into the first device ----
 * The reference parallelises whole-frame sample passes over workers and merges them (src/main.rs:199-217); here
 * device g of G renders samples g, g+G, ... of the call into its own accumulation buffer, the (sum XYZ, weight)
 * arrays are summed into devices[0] with ncclReduce over NVLink, and colour = sum * (1/weight) is formed there.
 * Single process; NCCL is loaded at run time (libnccl.so.2) -- VRJ_ERR_UNSUPPORTED if it is missing. */
typedef struct VrjComm VrjComm;
typedef struct VrjMultiScene VrjMultiScene;
VRJ_API VrjStatus vrj_comm_create(int32_t n_devices, const int32_t *devices, VrjComm **out);
VRJ_API void vrj_comm_destroy(VrjComm *comm);
/* the scene replicated on every device of the communicator */
VRJ_API VrjStatus vrj_comm_scene_create(VrjComm *comm, const VrjSceneDesc *desc, VrjMultiScene **out);
VRJ_API void vrj_comm_scene_destroy(VrjMultiScene *scene);
/* same arguments and outputs as vrj_render_tile (out->memory = VRJ_MEM_DEVICE means memory of devices[0]);
 * colour_bias / weight_bias are returned as zero (a reduced buffer has no compensation term), `accumulate` and
 * `photons` are not supported; params->sample_stride must be 0 or 1. */
VRJ_API VrjStatus vrj_render_sharded(VrjMultiScene *scene, const VrjTile *tile, uint64_t height, uint64_t width,
                                     const VrjRenderParams *params, VrjAccumOut *out);

/* ClampingToneMapper (src/image.rs:130-187) on `n_pixels` colours (3 doubles each) -> 3 bytes each.
 * source VRJ_TONEMAP_XYZ: ColourXyz::to_srgb (colour_xyz.rs:48-84, constants as written) then clamp + truncating byte
 * conversion (image.rs:120-123, 0.5 -> 127); VRJ_TONEMAP_LINEAR_RGB: clamp + byte only.  `memory` describes both pointers. */
enum { VRJ_TONEMAP_XYZ = 0, VRJ_TONEMAP_LINEAR_RGB = 1 };
VRJ_API VrjStatus vrj_tone_map(int32_t device, uint32_t memory, uint32_t source, const double *colour, uint64_t n_pixels,
                               uint8_t *rgb8);

/* ---- BoundingVolumeHierarchy::build on the device (SURVEY 8f N1) ----
 * Replaces the host-side recursion of src/raycasting/bounding_volume_hierarchy.rs:38-75 (bounds -> largest_dimension
 * -> sort by box centre -> split at len/2) for triangle sets, and returns EXACTLY the tree that recursion builds
 * with a stable sort: same boxes, same DFS pre-order node numbering, same leaf order.  Inputs and outputs are host
 * arrays in the layout VrjSceneDesc uses:
 *   vertices   9 doubles per triangle (v0 xyz, v1 xyz, v2 xyz), in the caller's order
 *   order      n entries: order[i] = input index of the triangle at leaf position i (= VrjSceneDesc.tri_prim_id)
 *   node_min / node_max   4 doubles {x, y, z, 0} per node, 2n-1 nodes (1 node when n == 0)
 *   node_child            2 per node, BVH-local: internal {left, right}; leaf {~leaf position, triangle count}
 *   depth      levels of the tree (VrjBvh.depth); may be NULL.  stats may be NULL. */
typedef struct VrjBvhBuildStats {
    double device_ms;        /* CUDA-event time of the build kernels (copies excluded) */
    uint32_t global_levels;  /* levels sorted with the segmented radix sort */
    uint32_t radix_passes;   /* 8-bit digit passes actually run (constant digits are skipped) */
    uint32_t small_subtrees; /* subtrees finished by one CTA each in shared memory */
    uint32_t pad;
} VrjBvhBuildStats;
VRJ_API VrjStatus vrj_bvh_build(int32_t device, uint64_t n_triangles, const double *vertices, uint32_t *order,
                                double *node_min, double *node_max, int32_t *node_child, uint32_t *depth,
                                VrjBvhBuildStats *stats);

VRJ_API VrjStatus vrj_trace_rays(const VrjScene *scene, uint64_t n, const double *origins, const double *directions,
                         uint32_t bvh_filter, int32_t *object_id, int32_t *prim_id, double *t, VrjStats *stats);

#ifdef __cplusplus
}
#endif
#endif
