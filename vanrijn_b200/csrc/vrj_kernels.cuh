// vrj_kernels.cuh -- the wavefront: persistent-thread kernels for one batch of samples.
//
//   k_trace   : Sampler::sample for every ray of the queue (the first launch generates the camera
//               rays, camera.rs:45-66): a pure map ray -> (item, triangle); carries no shading state,
//               so its register budget is the traversal's alone.
//   k_shade   : consumes those hits: finishes paths (miss: black / sky; depth limit) or runs one level
//               of Integrator::integrate -- rebuild the hit, sample the material (Whitted: trace the
//               shadow rays), update the affine accumulator -- and enqueues the bounce ray,
//               warp-ballot compacted.
//   k_resolve : per pixel, apply the batch's samples IN SAMPLE ORDER to the Kahan accumulator
//               (AccumulationBuffer::update_pixel, accumulation_buffer.rs:44-60).
//
// The recursion of simple_random_integrator.rs:12-55 is unrolled with an affine accumulator:
// every bsdf in the crate maps incoming intensity x to a*x + b, so after bounce k
//   B += A * b_k ;  A *= a_k * (pdf_k * |W_k . n_k|)      and the sample is A * L_leaf + B.
#pragma once
#include "vrj_traverse.cuh"

// minimum resident CTAs (of 128 threads) per SM the register allocator must allow
#ifndef VRJ_SHADE_MINB
#define VRJ_SHADE_MINB 5
#endif
#ifndef VRJ_SHADE_CHUNK
#define VRJ_SHADE_CHUNK 1024
#endif
#ifndef VRJ_TRACE_MINB
#define VRJ_TRACE_MINB 6
#endif
#ifndef VRJ_RAYGEN_CHUNK
#define VRJ_RAYGEN_CHUNK 1024
#endif
// 1: the closest-hit stage 1 of a bounce ray (analytic objects, root pre-test, traversal record) runs in its own streaming
// kernel, k_stage, instead of at the end of k_shade: k_shade loses a quarter of its code (it is bound by instruction fetch and
// binary64 latency at 5 CTAs per SM) and the stage work runs at twice the occupancy; the price is re-reading the ray (48 B)
#ifndef VRJ_SPLIT_STAGE
#define VRJ_SPLIT_STAGE 0
#endif
#ifndef VRJ_STAGE_MINB
#define VRJ_STAGE_MINB 8
#endif
#ifndef VRJ_RAYGEN_MINB
#define VRJ_RAYGEN_MINB VRJ_SHADE_MINB
#endif
#ifndef VRJ_FIRST_UNSORTED
#define VRJ_FIRST_UNSORTED 1
#endif
#ifndef VRJ_SHADOW_QUAD
#define VRJ_SHADOW_QUAD 1
#endif
#ifndef VRJ_TAIL_QUAD
#define VRJ_TAIL_QUAD 1
#endif
#ifndef VRJ_TRACE4_MINB
#define VRJ_TRACE4_MINB 5
#endif
// VRJ_PRECISION_F32_FAST: half the register footprint, so more resident CTAs
#ifndef VRJ_SHADE_MINB_F32
#define VRJ_SHADE_MINB_F32 8
#endif
#ifndef VRJ_TRACE_MINB_F32
#define VRJ_TRACE_MINB_F32 8
#endif
#define VRJ_SHADE_BOUNDS(R) __launch_bounds__(128, sizeof(R) == 4 ? VRJ_SHADE_MINB_F32 : VRJ_SHADE_MINB)
#define VRJ_TRACE_BOUNDS(R) __launch_bounds__(128, sizeof(R) == 4 ? VRJ_TRACE_MINB_F32 : VRJ_TRACE_MINB)

namespace vrj {

constexpr int SHADE_CHUNK = VRJ_SHADE_CHUNK;

struct LightDev {
    double dir[3];
    SpectrumDev spectrum; // samples live in RenderConst::light_samples
};

// Path queue, structure of 16-byte arrays (every access is coalesced).  k_shade writes an entry
// (compacted), k_trace reads its ray and fills hit[]; the next k_shade consumes both.
struct PathQueue {
    double2 *q0; // origin.x, origin.y      of the ray to trace / that produced the hit
    double2 *q1; // origin.z, direction.x
    double2 *q2; // direction.y, direction.z
    double2 *q3; // wavelength, A
    double2 *q4; // B, aux (SimpleRandom: W.y of the un-normalised bounce direction; Whitted: B before the bounce term)
    uint4 *q5;   // result slot, rng draw ordinal, recursion limit of the NEXT integrate level, flags (1 = terminal)
};

// n / d for a divisor fixed per call (Granlund-Montgomery round-up form, exact for every 32-bit n and d >= 1): one IMAD.HI,
// one subtract, two shifts and an add instead of the ~20-instruction 32-bit division sequence; slot_to_pixel runs two of
// them per camera ray and per shaded path
struct FastDiv {
    uint32_t m, s1, s2, d;
    __host__ __device__ static FastDiv make(uint32_t d) {
        FastDiv f;
        uint32_t l = 0;
        while (l < 32 && (1ull << l) < d) l++;
        f.m = (uint32_t)(((1ull << 32) * ((1ull << l) - d)) / d + 1);
        f.s1 = l < 1 ? l : 1, f.s2 = l > 1 ? l - 1 : 0, f.d = d;
        return f;
    }
    __device__ __forceinline__ uint32_t div(uint32_t n) const {
        const uint32_t t = __umulhi(m, n);
        return (t + ((n - t) >> s1)) >> s2;
    }
};

struct RenderConst {
    uint64_t width, height;             // full image
    uint64_t start_column, start_row;   // tile origin
    uint32_t tile_w, tile_h, npix;      // tile
    uint32_t batch_samples;             // samples in this batch
    FastDiv div_batch, div_tile_w;      // division by batch_samples / tile_w
    uint64_t first_sample;              // sample index of batch slot 0
    uint64_t sample_stride;
    const uint64_t *sample_table;       // non-NULL: sample index of batch slot s is sample_table[s] (coalesced calls, MultiCalls)
    uint64_t seed;
    uint32_t max_depth, n_lights;
    uint32_t has_ambient, pad;
    double bias;
    double film_w, film_h;
    const LightDev *lights;      // n_lights entries, then (if has_ambient) the ambient light's spectrum in entry n_lights
    const double *light_samples;
    const uint32_t *pixel_list;  // kernels with LIST = true: batch position p renders tile pixel pixel_list[p] and npix is the
                                 // list's length (the still-active pixels of an adaptive pass, vrj_render_adaptive); slots and
                                 // photons stay indexed by list position
};

template <typename R>
__device__ __forceinline__ R light_intensity(const RenderConst &rc, const SpectrumDev &s, R wavelength) {
    const double *p = rc.light_samples + s.first;
    return spectrum_lookup<R>((R)s.shortest, (R)s.longest, s.n, wavelength, [p](uint32_t i) { return (R)__ldg(p + i); });
}

enum { ST_PRIMARY = 0, ST_BOUNCE, ST_SHADOW, ST_MISSED, ST_ESCAPED, ST_LIMITED, ST_NODES, ST_TRIS, ST_STAGED, ST_COUNT };

struct LocalStats {
    uint32_t v[ST_COUNT];
    __device__ __forceinline__ void clear() {
#pragma unroll
        for (int i = 0; i < ST_COUNT; i++) v[i] = 0;
    }
    __device__ __forceinline__ void flush(unsigned long long *g) {
#pragma unroll
        for (int i = 0; i < ST_COUNT; i++) {
            uint32_t s = __reduce_add_sync(0xffffffffu, v[i]);
            if ((threadIdx.x & 31) == 0 && s) atomicAdd(g + i, (unsigned long long)s);
        }
    }
};

// warp-ballot compaction: one atomic per warp reserves a contiguous run of the output queue
__device__ __forceinline__ uint32_t queue_reserve(bool alive, uint32_t *count) {
    uint32_t mask = __ballot_sync(0xffffffffu, alive);
    uint32_t lane = threadIdx.x & 31;
    uint32_t base = 0;
    if (lane == 0 && mask) base = atomicAdd(count, (uint32_t)__popc(mask));
    base = __shfl_sync(0xffffffffu, base, 0);
    return base + (uint32_t)__popc(mask & ((1u << lane) - 1u));
}

// the queue keeps binary64 slots in both precisions (binary32 values widen exactly)
template <typename R>
__device__ __forceinline__ void queue_store(const PathQueue &q, uint32_t idx, V3<R> o, V3<R> d, R wl, R A, R B, R aux, uint32_t slot,
                                            uint32_t ordinal, uint32_t limit, uint32_t flags) {
    q.q0[idx] = make_double2((double)o.x, (double)o.y);
    q.q1[idx] = make_double2((double)o.z, (double)d.x);
    q.q2[idx] = make_double2((double)d.y, (double)d.z);
    q.q3[idx] = make_double2((double)wl, (double)A);
    q.q4[idx] = make_double2((double)B, (double)aux);
    q.q5[idx] = make_uint4(slot, ordinal, limit, flags);
}
template <typename R>
__device__ __forceinline__ void queue_load_ray(const PathQueue &q, uint32_t j, V3<R> &o, V3<R> &d) {
    const double2 a0 = q.q0[j], a1 = q.q1[j], a2 = q.q2[j];
    o = V3<R>{(R)a0.x, (R)a0.y, (R)a1.x}, d = V3<R>{(R)a1.y, (R)a2.x, (R)a2.y};
}

// Ray::new (raycasting/mod.rs:41-46) then .bias(amount) (raycasting/mod.rs:58-60): normalise, offset, normalise again
template <typename R>
__device__ __forceinline__ void biased_ray(V3<R> origin, V3<R> direction, R amount, V3<R> &o, V3<R> &d) {
    V3<R> d1 = normalize(direction);
    o = origin + d1 * amount;
    d = normalize(d1);
}

// Result slots are PIXEL-major within a batch: slot = pixel * batch_samples + sample.  The samples of one pixel are
// neighbours in queue 0, so the lanes of a warp start from (almost) the same camera ray: the primary traversal fetches the
// same nodes (broadcast loads), hits the same primitive class, and the first bounces leave from neighbouring points
// (k_trace on camera rays 3.5 -> 2.5 ms per 32-spp step, measured).  A sample is still a pure function of
// (seed, pixel, sample index), so the order changes no result.
// LIST: the batch covers the pixels of rc.pixel_list (a compile-time switch, so the tile's kernels carry no trace of it).
template <bool LIST = false>
__device__ __forceinline__ void slot_to_pixel(const RenderConst &rc, uint32_t slot, uint32_t &pixel_global,
                                              uint64_t &sample, uint64_t &grow, uint64_t &gcol) {
    uint32_t p = rc.div_batch.div(slot), s = slot - p * rc.batch_samples;
    if (LIST) p = __ldg(rc.pixel_list + p);
    uint32_t row = rc.div_tile_w.div(p), col = p - row * rc.tile_w;
    grow = rc.start_row + row, gcol = rc.start_column + col;
    pixel_global = (uint32_t)(grow * rc.width + gcol);
    sample = rc.sample_table ? __ldg(rc.sample_table + s) : rc.first_sample + (uint64_t)s * rc.sample_stride;
}

// Stage-1 results of one ray + the list of rays that still need BVH traversal
struct TraceBuffers {
    int2 *hits;            // per queue entry: (item, triangle), -1 = miss
    double *tbest;         // per queue entry: distance of that hit (+inf on a miss)
    uint32_t *list;        // queue entries whose ray passed a BVH root pre-test
    TraceRec *recs;        // non-NULL: those rays as ready-to-walk records instead (default f32 walk in binary64; see TraceRec)
};

// analytic objects + BVH root pre-test for the ray just written to queue entry `idx`; all 32 lanes call
template <bool COUNT, typename R>
__device__ __forceinline__ void stage_ray(const DevScene &sc, bool have_ray, uint32_t idx, V3<R> o, V3<R> d, const TraceBuffers &tb,
                                          uint32_t *list_count, LocalStats &ls) {
    bool need = false;
    HitT<R> best;
    FilterRay<float> fr;
    if (have_ray) {
        TraceCounters tc = {0, 0};
        need = pretrace<COUNT>(sc, o, d, best, tc, fr);
        tb.hits[idx] = make_int2(best.item, best.tri);
        tb.tbest[idx] = (double)best.t;
        if (COUNT) ls.v[ST_TRIS] += tc.tri_tests;
    }
    uint32_t pos = queue_reserve(need, list_count);
    if (need) {
        ls.v[ST_STAGED]++;
        if (sizeof(R) == 8 && tb.recs) store_trace_rec(tb.recs, pos, tri_ray(convert<double>(o), convert<double>(d)), fr, (double)best.t, best.item, idx);
        else tb.list[pos] = idx;
    }
}

// The camera ray of a result slot (camera.rs:45-66): two Philox draws, the film point, Ray::new.  It is a pure function of
// the slot, so the primary level never stores it: k_raygen, k_trace on camera rays and the first k_shade each form it again
// (one Philox block + one normalisation) instead of moving 48 bytes per ray through HBM three times.
template <typename R, bool LIST = false>
__device__ __forceinline__ void camera_ray(const DevScene &sc, const RenderConst &rc, uint32_t slot, V3<R> &o, V3<R> &d) {
    uint32_t pixel;
    uint64_t sample, grow, gcol;
    slot_to_pixel<LIST>(rc, slot, pixel, sample, grow, gcol);
    Rng rng;
    rng.init(rc.seed, pixel, sample, 0);
    R ux = rng.uniform<R>(), uy = rng.uniform<R>();
    const R film_w = (R)rc.film_w, film_h = (R)rc.film_h;
    R px = ((R)gcol + ux) * (film_w * (R(1) / (R)rc.width)) - film_w * R(0.5);
    R py = ((R)(rc.height - (grow + 1)) + uy) * (film_h * (R(1) / (R)rc.height)) - film_h * R(0.5);
    o = V3<R>{(R)sc.cam[0], (R)sc.cam[1], (R)sc.cam[2]};
    d = normalize(V3<R>{px, py, R(1)});
}

// ---- k_raygen: camera rays (camera.rs:45-66), staged for traversal ----
template <typename R, bool COUNT, bool LIST = false>
__global__ void __launch_bounds__(128, sizeof(R) == 4 ? VRJ_SHADE_MINB_F32 : VRJ_RAYGEN_MINB) k_raygen(DevScene sc, RenderConst rc, PathQueue q, TraceBuffers tb, uint32_t *list_count,
                                                uint32_t *work, unsigned long long *stats) {
    const uint32_t n = rc.npix * rc.batch_samples;
    LocalStats ls;
    ls.clear();
    // a CTA takes VRJ_RAYGEN_CHUNK slots per fetch: one atomic on the shared counter per 1024 rays, not one per warp of 32
    __shared__ uint32_t s_base;
    while (true) {
        __syncthreads();
        if (threadIdx.x == 0) s_base = atomicAdd(work, (uint32_t)VRJ_RAYGEN_CHUNK);
        __syncthreads();
        const uint32_t base = s_base;
        if (base >= n) break;
#pragma unroll 1
        for (uint32_t k = threadIdx.x; k < (uint32_t)VRJ_RAYGEN_CHUNK; k += 128) {
            const uint32_t j = base + k;
            if (base + (k & ~31u) >= n) break; // the whole warp is past the end
            V3<R> o = V3<R>{R(0), R(0), R(0)}, d = V3<R>{R(0), R(0), R(1)};
            if (j < n) {
                camera_ray<R, LIST>(sc, rc, j, o, d);
                ls.v[ST_PRIMARY]++;
            }
            stage_ray<COUNT>(sc, j < n, j, o, d, tb, list_count, ls);
        }
    }
    ls.flush(stats);
}

// ---- k_trace: BVH traversal for the staged rays; updates hits / tbest where a triangle is closer ----
struct ListRaySource {
    const PathQueue &q;
    const TraceBuffers &tb;
    template <typename R>
    __device__ __forceinline__ void load(uint32_t r, V3<R> &o, V3<R> &d, HitT<R> &best) {
        uint32_t j = tb.list[r];
        queue_load_ray(q, j, o, d);
        int2 h = tb.hits[j];
        best.item = h.x, best.tri = h.y, best.t = (R)tb.tbest[j];
    }
    template <typename NT, typename R>
    __device__ __forceinline__ uint32_t load_setup(uint32_t r, TriRayT<R> &tr, FilterRay<NT> &fr, HitT<R> &best) {
        V3<R> o, d;
        load(r, o, d, best);
        tr = tri_ray(o, d);
        fr = filter_ray<NT>(o, d);
        return r;
    }
};
// rays staged as records: nothing to compute, three 256-bit loads; the handle is the queue entry itself
struct RecRaySource {
    const TraceBuffers &tb;
    __device__ __forceinline__ uint32_t load_setup(uint32_t r, TriRayT<double> &tr, FilterRay<float> &fr, HitT<double> &best) {
        return load_trace_rec(tb.recs, r, tr, fr, best);
    }
};
struct RecHitSink {
    const TraceBuffers &tb;
    __device__ __forceinline__ void store(uint32_t j, const HitT<double> &best, bool improved) {
        if (!improved) return;
        tb.hits[j] = make_int2(best.item, best.tri);
        tb.tbest[j] = best.t;
    }
};
// the same for the camera rays of a batch: the ray is formed from its slot, nothing is read from the queue
template <bool LIST = false>
struct PrimaryRaySource {
    const DevScene &sc;
    const RenderConst &rc;
    const TraceBuffers &tb;
    template <typename R>
    __device__ __forceinline__ void load(uint32_t r, V3<R> &o, V3<R> &d, HitT<R> &best) {
        uint32_t j = tb.list[r];
        camera_ray<R, LIST>(sc, rc, j, o, d);
        int2 h = tb.hits[j];
        best.item = h.x, best.tri = h.y, best.t = (R)tb.tbest[j];
    }
    template <typename NT, typename R>
    __device__ __forceinline__ uint32_t load_setup(uint32_t r, TriRayT<R> &tr, FilterRay<NT> &fr, HitT<R> &best) {
        V3<R> o, d;
        load(r, o, d, best);
        tr = tri_ray(o, d);
        fr = filter_ray<NT>(o, d);
        return r;
    }
};
struct ListHitSink {
    const TraceBuffers &tb;
    template <typename R>
    __device__ __forceinline__ void store(uint32_t r, const HitT<R> &best, bool improved) {
        if (!improved) return;
        uint32_t j = tb.list[r];
        tb.hits[j] = make_int2(best.item, best.tri);
        tb.tbest[j] = (double)best.t;
    }
};

template <typename NT, typename R, bool COUNT>
__global__ void VRJ_TRACE_BOUNDS(R) k_trace(DevScene sc, PathQueue q, TraceBuffers tb, const uint32_t *list_count,
                                               uint32_t *work, unsigned long long *stats, const uint32_t *tail_done) {
    if (tail_done && *tail_done) return;
    const uint32_t n = *list_count;
    ListRaySource source{q, tb};
    ListHitSink sink{tb};
    TraceCounters tc = {0, 0};
    trace_persistent<NT, R, COUNT>(sc, n, work, source, sink, tc);
    if (COUNT) {
        LocalStats ls;
        ls.clear();
        ls.v[ST_NODES] = tc.node_visits, ls.v[ST_TRIS] = tc.tri_tests;
        ls.flush(stats);
    }
}

// k_trace for the camera rays of a batch
template <typename NT, typename R, bool COUNT, bool LIST = false>
__global__ void VRJ_TRACE_BOUNDS(R) k_trace_primary(DevScene sc, RenderConst rc, TraceBuffers tb, const uint32_t *list_count, uint32_t *work,
                                                    unsigned long long *stats) {
    const uint32_t n = *list_count;
    PrimaryRaySource<LIST> source{sc, rc, tb};
    ListHitSink sink{tb};
    TraceCounters tc = {0, 0};
    trace_persistent<NT, R, COUNT>(sc, n, work, source, sink, tc);
    if (COUNT) {
        LocalStats ls;
        ls.clear();
        ls.v[ST_NODES] = tc.node_visits, ls.v[ST_TRIS] = tc.tri_tests;
        ls.flush(stats);
    }
}

// k_trace over ready-to-walk records (camera rays and bounce rays alike): the default walk of the parity path
template <bool COUNT>
__global__ void VRJ_TRACE_BOUNDS(double) k_trace_rec(DevScene sc, TraceBuffers tb, const uint32_t *list_count, uint32_t *work,
                                                     unsigned long long *stats, const uint32_t *tail_done) {
    if (tail_done && *tail_done) return;
    const uint32_t n = *list_count;
    RecRaySource source{tb};
    RecHitSink sink{tb};
    TraceCounters tc = {0, 0};
    trace_persistent<float, double, COUNT>(sc, n, work, source, sink, tc);
    if (COUNT) {
        LocalStats ls;
        ls.clear();
        ls.v[ST_NODES] = tc.node_visits, ls.v[ST_TRIS] = tc.tri_tests;
        ls.flush(stats);
    }
}

// the same launch over the 4-wide form of the tree (VRJ_FILTER_F32X4)
template <bool COUNT, bool PRIMARY, bool LIST = false>
__global__ void __launch_bounds__(128, VRJ_TRACE4_MINB) k_trace4(DevScene sc, RenderConst rc, PathQueue q, TraceBuffers tb, const uint32_t *list_count,
                                                                 uint32_t *work, unsigned long long *stats, const uint32_t *tail_done) {
    if (tail_done && *tail_done) return;
    const uint32_t n = *list_count;
    ListHitSink sink{tb};
    TraceCounters tc = {0, 0};
    if (PRIMARY) {
        PrimaryRaySource<LIST> source{sc, rc, tb};
        trace_persistent_quad<COUNT>(sc, n, work, source, sink, tc);
    } else {
        ListRaySource source{q, tb};
        trace_persistent_quad<COUNT>(sc, n, work, source, sink, tc);
    }
    if (COUNT) {
        LocalStats ls;
        ls.clear();
        ls.v[ST_NODES] = tc.node_visits, ls.v[ST_TRIS] = tc.tri_tests;
        ls.flush(stats);
    }
}

// the same launch over 16-bit nodes (VRJ_FILTER_Q16)
template <bool COUNT, bool PRIMARY, bool LIST = false>
__global__ void __launch_bounds__(128, VRJ_TRACE_MINB) k_traceq(DevScene sc, RenderConst rc, PathQueue q, TraceBuffers tb, const uint32_t *list_count,
                                                                uint32_t *work, unsigned long long *stats, const uint32_t *tail_done) {
    if (tail_done && *tail_done) return;
    const uint32_t n = *list_count;
    ListHitSink sink{tb};
    TraceCounters tc = {0, 0};
    if (PRIMARY) {
        PrimaryRaySource<LIST> source{sc, rc, tb};
        trace_persistent_q16<COUNT>(sc, n, work, source, sink, tc);
    } else {
        ListRaySource source{q, tb};
        trace_persistent_q16<COUNT>(sc, n, work, source, sink, tc);
    }
    if (COUNT) {
        LocalStats ls;
        ls.clear();
        ls.v[ST_NODES] = tc.node_visits, ls.v[ST_TRIS] = tc.tri_tests;
        ls.flush(stats);
    }
}

// ---- one level of the integrator for one path (shared by k_shade and k_tail) ----
template <typename R>
struct PathRegsT {
    V3<R> o, d;         // in: the ray that produced `hit`; out: the bounce ray
    R wl, A, B, aux;    // wavelength, affine accumulator, aux (SimpleRandom: W.y; Whitted: B before the bounce term)
    uint32_t slot, ordinal, limit, flags;
};
// a finished sample: (wavelength, intensity * 360); binary64 slots in both precisions
template <typename R>
__device__ __forceinline__ double2 photon_out(R wavelength, R intensity) { return make_double2((double)wavelength, (double)intensity); }

// Consumes the closest hit of p's ray: finishes the path (miss: black / sky; depth limit) and returns false, or
// runs one level of Integrator::integrate -- rebuild the IntersectionInfo, sample the material (Whitted: trace the
// shadow rays), update the affine accumulator -- leaves the bounce ray and the new state in p and returns true.
// `first`: p.slot is set, the rest of the state is initialised here (camera.rs:108-119).
// `load_ray(o, d)` fetches the ray only when it is needed.
template <typename NT, bool COUNT, bool WHITTED, int MM, bool LIST, typename R, typename RayLoader>
__device__ __forceinline__ bool shade_entry(const DevScene &sc, const RenderConst &rc, PathRegsT<R> &p, int2 hit, R hit_t, bool first,
                                            RayLoader load_ray, double2 *photons, LocalStats &ls) {
    const R span = R(740.0) - R(380.0); // photon.rs:18-24, colour/mod.rs:13-14
    if (first) {
        if (hit.x < 0) {
            photons[p.slot] = make_double2(0.0, 0.0); // camera.rs:110-113
            ls.v[ST_MISSED]++;
            return false;
        }
        uint32_t pixel;
        uint64_t sample, grow, gcol;
        slot_to_pixel<LIST>(rc, p.slot, pixel, sample, grow, gcol);
        Rng rng;
        rng.init(rc.seed, pixel, sample, 2);
        p.wl = R(380.0) + span * rng.uniform<R>(); // photon.rs:18-24
        p.ordinal = 4, p.A = R(1), p.B = R(0), p.aux = R(0), p.limit = rc.max_depth, p.flags = 0; // ordinal 3 unused: draws pair up per Philox block
        if (!WHITTED && p.limit == 0) {
            photons[p.slot] = make_double2(0.0, 0.0); // simple_random_integrator.rs:20-25
            ls.v[ST_LIMITED]++;
            return false;
        }
    } else if (WHITTED) {
        // whitted_integrator.rs:52-79: the bounce term counts only if the ray hit and the level had limit > 0
        if (hit.x < 0 || (p.flags & 1u)) {
            photons[p.slot] = photon_out(p.wl, p.aux * span);
            if (hit.x < 0) ls.v[ST_ESCAPED]++;
            else ls.v[ST_LIMITED]++;
            return false;
        }
    } else if (hit.x < 0) {
        R L = rgb_reflection_intensity(p.aux, p.aux, R(1), p.wl); // sky(W): simple_random_integrator.rs:43-46,57-65
        photons[p.slot] = photon_out(p.wl, (p.A * L + p.B) * span);
        ls.v[ST_ESCAPED]++;
        return false;
    } else if (p.limit == 0) {
        // the recursion returns Photon{0,0} (:20-25): wavelength 0 makes the sample's XYZ ~0
        photons[p.slot] = make_double2(0.0, 0.0);
        ls.v[ST_LIMITED]++;
        return false;
    }
    load_ray(p.o, p.d);
    HitFrameT<R> h;
    bool ok = rebuild_hit(sc, p.o, p.d, hit.x, hit.y, hit_t, h);
    // algebra_utils.rs:3-5, mat3.rs:111-118
    M3T<R> w2b = from_rows(h.tangent, h.cotangent, h.normal), b2w;
    ok = try_inverse(w2b, b2w) && ok;
    if (!ok) {
        // the reference panics here (simple_random_integrator.rs:28,31); report a NaN sample
        photons[p.slot] = make_double2((double)p.wl, CUDART_NAN);
        return false;
    }
    MaterialDev m = sc.materials[h.material];
    R s = spectrum_intensity(sc.spectra, sc.spectrum_samples, sc.spectrum_grids, m.spectrum, p.wl);
    V3<R> w_retro = mul(w2b, h.retro);
    if (WHITTED) {
        // whitted_integrator.rs:33-50: one shadow ray per light
        TraceCounters tc = {0, 0};
        R direct = R(0); // fold starts from photon.intensity == 0
        for (uint32_t li = 0; li < rc.n_lights; li++) {
            LightDev Lt = rc.lights[li];
            V3<R> ldir = V3<R>{(R)Lt.dir[0], (R)Lt.dir[1], (R)Lt.dir[2]};
            V3<R> so, sd;
            biased_ray(h.location, ldir, (R)rc.bias, so, sd);
            HitT<R> sh = trace_closest<NT, COUNT, true, R, VRJ_SHADOW_QUAD != 0>(sc, so, sd, tc);
            ls.v[ST_SHADOW]++;
            R term;
            if (sh.item >= 0) {
                term = rc.has_ambient ? light_intensity<R>(rc, rc.lights[rc.n_lights].spectrum, p.wl) : R(0);
            } else {
                R emitted = light_intensity<R>(rc, Lt.spectrum, p.wl);
                emitted = emitted * fabs(dot(ldir, h.normal));
                R la, lb;
                material_bsdf_affine<MM>(m, s, w_retro, mul(w2b, ldir), la, lb); // (retro, incoming) order
                term = la * emitted + lb;
            }
            direct += term;
        }
        if (COUNT) ls.v[ST_NODES] += tc.node_visits, ls.v[ST_TRIS] += tc.tri_tests;
        p.B += p.A * direct;
    }
    Rng rng;
    uint32_t pixel;
    uint64_t sample, grow, gcol;
    slot_to_pixel<LIST>(rc, p.slot, pixel, sample, grow, gcol);
    rng.init(rc.seed, pixel, sample, p.ordinal);
    V3<R> w_s;
    R pdf;
    material_sample<MM>(m, s, w_retro, rng, w_s, pdf);
    p.ordinal = rng.ordinal;
    V3<R> W = mul(b2w, w_s);
    biased_ray(h.location, W, (R)rc.bias, p.o, p.d);
    R cosine = fabs(dot(W, h.normal));
    R ba, bb;
    if (WHITTED) {
        // bsdf(retro, sampled, L_in) * |W.n|, pdf unused; B before the bounce term is kept in aux
        material_bsdf_affine<MM>(m, s, w_retro, w_s, ba, bb);
        p.aux = p.B;
        p.B += p.A * (bb * cosine);
        p.A *= ba * cosine;
        p.flags = p.limit == 0 ? 1u : 0u; // the ray is still traced at limit 0, its result unused
        p.limit = p.limit ? p.limit - 1 : 0;
    } else {
        // simple_random_integrator.rs:39-53: bsdf(sampled, retro, L_in * pdf * |W.n|)
        material_bsdf_affine<MM>(m, s, w_s, w_retro, ba, bb);
        p.B += p.A * bb;
        p.A *= ba * (pdf * cosine);
        p.aux = W.y; // the sky uses the un-normalised W
        p.limit -= 1;
    }
    ls.v[ST_BOUNCE]++;
    return true;
}

// ---- k_shade: consume the hits of a queue; survivors are enqueued warp-ballot compacted and staged ----
template <typename NT, typename R, bool COUNT, bool WHITTED, bool FIRST, int MM, bool LIST = false>
__global__ void VRJ_SHADE_BOUNDS(R) k_shade(DevScene sc, RenderConst rc, PathQueue in, const uint32_t *in_count,
                                               TraceBuffers tb_in, PathQueue out, uint32_t *out_count, TraceBuffers tb_out,
                                               uint32_t *list_count, uint32_t *work, double2 *photons,
                                               unsigned long long *stats, const uint32_t *tail_done) {
    if (*tail_done) return; // a k_tail launch has already finished every remaining path of this batch
    const uint32_t n = FIRST ? rc.npix * rc.batch_samples : *in_count;
    // A CTA takes SHADE_CHUNK queue entries at a time and orders them by hit class (miss / sphere / plane /
    // triangle) in shared memory before shading, so the lanes of a warp run the same rebuild_hit branch.
    __shared__ uint32_t s_sorted[SHADE_CHUNK];
    __shared__ uint32_t s_count[4], s_base;
    LocalStats ls;
    ls.clear();
    while (true) {
        if (threadIdx.x == 0) s_base = atomicAdd(work, (uint32_t)SHADE_CHUNK);
        if (threadIdx.x < 4) s_count[threadIdx.x] = 0;
        __syncthreads();
        const uint32_t base = s_base;
        if (base >= n) break;
        const uint32_t total = min((uint32_t)SHADE_CHUNK, n - base);
        if (FIRST && VRJ_FIRST_UNSORTED) {
            // camera rays arrive pixel-major: a warp's 32 entries are samples of one pixel and already share a hit class
#pragma unroll
            for (int e = 0; e < SHADE_CHUNK / 128; e++) s_sorted[threadIdx.x + e * 128] = base + threadIdx.x + e * 128;
        } else {
            uint32_t cls[SHADE_CHUNK / 128], pos[SHADE_CHUNK / 128];
#pragma unroll
            for (int e = 0; e < SHADE_CHUNK / 128; e++) {
                uint32_t k = threadIdx.x + e * 128;
                cls[e] = 4;
                if (k < total) {
                    int item = tb_in.hits[base + k].x;
                    cls[e] = item < 0 ? 0u : 1u + min(sc.items[item].kind, 2u);
                    pos[e] = atomicAdd(&s_count[cls[e]], 1u);
                }
            }
            __syncthreads();
            const uint32_t c0 = s_count[0], c1 = c0 + s_count[1], c2 = c1 + s_count[2];
#pragma unroll
            for (int e = 0; e < SHADE_CHUNK / 128; e++)
                if (cls[e] < 4) s_sorted[(cls[e] == 0 ? 0u : cls[e] == 1 ? c0 : cls[e] == 2 ? c1 : c2) + pos[e]] = base + threadIdx.x + e * 128;
        }
        __syncthreads();
#pragma unroll 1
        for (uint32_t k = threadIdx.x; k < ((total + 31u) & ~31u); k += 128) {
            const uint32_t j = k < total ? s_sorted[k] : n;
            bool alive = false;
            PathRegsT<R> p;
            p.o = V3<R>{R(0), R(0), R(0)}, p.d = V3<R>{R(0), R(0), R(1)};
            p.wl = p.A = p.B = p.aux = R(0);
            p.slot = p.ordinal = p.limit = p.flags = 0;
            if (j < n) {
                int2 hit = tb_in.hits[j];
                if (FIRST) {
                    p.slot = j;
                } else {
                    double2 a3 = in.q3[j], a4 = in.q4[j];
                    uint4 a5 = in.q5[j];
                    p.wl = (R)a3.x, p.A = (R)a3.y, p.B = (R)a4.x, p.aux = (R)a4.y;
                    p.slot = a5.x, p.ordinal = a5.y, p.limit = a5.z, p.flags = a5.w;
                }
                alive = shade_entry<NT, COUNT, WHITTED, MM, LIST>(
                    sc, rc, p, hit, hit.x >= 0 ? (R)tb_in.tbest[j] : R(0), FIRST,
                    [&in, &sc, &rc, j](V3<R> &o, V3<R> &d) {
                        if (FIRST) camera_ray<R, LIST>(sc, rc, j, o, d); // never stored: see camera_ray
                        else queue_load_ray(in, j, o, d);
                    },
                    photons, ls);
            }
            uint32_t idx = queue_reserve(alive, out_count);
            if (alive) queue_store(out, idx, p.o, p.d, p.wl, p.A, p.B, p.aux, p.slot, p.ordinal, p.limit, p.flags);
#if !VRJ_SPLIT_STAGE
            stage_ray<COUNT>(sc, alive, idx, p.o, p.d, tb_out, list_count, ls);
#endif
        }
        __syncthreads(); // s_sorted / s_count are reused by the next chunk
    }
    ls.flush(stats);
}

// ---- k_stage: stage 1 of the closest hit for the bounce rays k_shade just enqueued (VRJ_SPLIT_STAGE) ----
template <typename R, bool COUNT>
__global__ void __launch_bounds__(128, VRJ_STAGE_MINB) k_stage(DevScene sc, PathQueue q, const uint32_t *count, TraceBuffers tb, uint32_t *list_count,
                                                               uint32_t *work, unsigned long long *stats, const uint32_t *tail_done) {
    if (*tail_done) return;
    const uint32_t n = *count;
    LocalStats ls;
    ls.clear();
    __shared__ uint32_t s_base;
    while (true) {
        __syncthreads();
        if (threadIdx.x == 0) s_base = atomicAdd(work, (uint32_t)VRJ_RAYGEN_CHUNK);
        __syncthreads();
        const uint32_t base = s_base;
        if (base >= n) break;
#pragma unroll 1
        for (uint32_t k = threadIdx.x; k < (uint32_t)VRJ_RAYGEN_CHUNK; k += 128) {
            const uint32_t j = base + k;
            if (base + (k & ~31u) >= n) break; // the whole warp is past the end
            V3<R> o = V3<R>{R(0), R(0), R(0)}, d = V3<R>{R(0), R(0), R(1)};
            if (j < n) queue_load_ray(q, j, o, d);
            stage_ray<COUNT>(sc, j < n, j, o, d, tb, list_count, ls);
        }
    }
    ls.flush(stats);
}

// ---- k_tail: when few paths are left, finish ALL their remaining levels in one launch ----
// A wavefront level costs at least the latency of its longest traversal (~100 us) however few rays it carries;
// here every lane follows one path (trace -> shade -> trace ...) to its end, so the remaining levels overlap.
// Runs before T_k on queue k; does nothing unless the queue is at most `tail_max` long; sets *tail_done so the
// remaining T / S launches of the batch return immediately.
// Persistent warps with per-lane refill: path lengths are geometric (most paths end after one or two more bounces, a few
// run for dozens), so a lane whose path has ended takes the next queue entry at once (one warp-aggregated atomic) instead
// of idling until the longest path of its warp is done -- in the one-path-per-thread form a warp ran ~6 bounces for ~1.7
// useful ones per lane.
template <typename NT, typename R, bool COUNT, bool WHITTED, int MM, bool LIST = false>
__global__ void __launch_bounds__(128, 2) k_tail(DevScene sc, RenderConst rc, PathQueue in, const uint32_t *in_count,
                                              uint32_t tail_max, double2 *photons, unsigned long long *stats,
                                              uint32_t *tail_done, uint32_t *work) {
    const uint32_t n = *in_count;
    if (n > tail_max || *tail_done == 1u) return;
    const unsigned FULL = 0xffffffffu;
    const uint32_t lane = threadIdx.x & 31;
    LocalStats ls;
    ls.clear();
    PathRegsT<R> p;
    p.o = V3<R>{R(0), R(0), R(0)}, p.d = V3<R>{R(0), R(0), R(1)};
    p.wl = p.A = p.B = p.aux = R(0);
    p.slot = p.ordinal = p.limit = p.flags = 0;
    bool alive = false, exhausted = false;
    while (true) {
        const unsigned idle_mask = __ballot_sync(FULL, !alive);
        if (idle_mask) {
            if (!exhausted) {
                const uint32_t want = (uint32_t)__popc(idle_mask);
                const int leader = __ffs(idle_mask) - 1;
                uint32_t base = 0;
                if ((int)lane == leader) base = atomicAdd(work, want);
                base = __shfl_sync(FULL, base, leader);
                if (base + want >= n) exhausted = true;
                if (!alive) {
                    const uint32_t j = base + (uint32_t)__popc(idle_mask & ((1u << lane) - 1u));
                    if (j < n) {
                        double2 a3 = in.q3[j], a4 = in.q4[j];
                        uint4 a5 = in.q5[j];
                        queue_load_ray(in, j, p.o, p.d);
                        p.wl = (R)a3.x, p.A = (R)a3.y, p.B = (R)a4.x, p.aux = (R)a4.y;
                        p.slot = a5.x, p.ordinal = a5.y, p.limit = a5.z, p.flags = a5.w;
                        alive = true;
                    }
                }
            }
            if (exhausted && __ballot_sync(FULL, alive) == 0u) break;
        }
        if (alive) {
            TraceCounters tc = {0, 0};
            // one lane, one path: what it waits on is the chain of dependent node fetches, and the 4-wide tree halves it
            HitT<R> h = trace_closest<NT, COUNT, false, R, VRJ_TAIL_QUAD != 0>(sc, p.o, p.d, tc);
            if (COUNT) ls.v[ST_NODES] += tc.node_visits, ls.v[ST_TRIS] += tc.tri_tests;
            alive = shade_entry<NT, COUNT, WHITTED, MM, LIST>(sc, rc, p, make_int2(h.item, h.tri), h.t, false, [](V3<R> &, V3<R> &) {}, photons, ls);
        }
    }
    ls.flush(stats);
    // every CTA read *in_count before any path could change it (k_tail never writes the queues); 2 = "done by this launch"
    if (n && blockIdx.x == 0 && threadIdx.x == 0) *tail_done = 2u;
}

struct AccumDev {
    double *colour, *sum, *bias; // 3 per pixel
    double *weight, *weight_bias;
};

// accumulation_buffer.rs:44-60 applied for the batch's samples in sample order
// R: precision of ColourXyz::from_photon (the colour matching functions); the accumulators are binary64 in both modes
template <typename R>
__global__ void k_resolve(AccumDev acc, const double2 *photons, uint32_t first, uint32_t npix, uint32_t batch_samples) {
    uint32_t p = first + blockIdx.x * blockDim.x + threadIdx.x; // pixels [first, npix): a call's last batch resolves in pieces
    if (p >= npix) return;
    double sx = acc.sum[3 * p], sy = acc.sum[3 * p + 1], sz = acc.sum[3 * p + 2];
    double bx = acc.bias[3 * p], by = acc.bias[3 * p + 1], bz = acc.bias[3 * p + 2];
    double w = acc.weight[p], wb = acc.weight_bias[p];
    for (uint32_t s = 0; s < batch_samples; s++) {
        double2 ph = photons[(size_t)p * batch_samples + s]; // pixel-major: a thread walks its own 16 * batch_samples bytes
        // colour_xyz.rs:31-35.  A sample of intensity +0 (every primary miss and depth-limited path: 45 % of the bench frame)
        // contributes cmf * 0 = 0 whatever its wavelength; the seven exponentials are skipped and the Kahan update below,
        // which still runs, leaves the same sums (adding +0 or -0 to an accumulator that started at +0 is the identity)
        D3 c = d3(0.0, 0.0, 0.0);
        if (__double_as_longlong(ph.y) != 0ll) c = convert<double>(cmf<R>((R)ph.x) * (R)ph.y);
        const double weight = 1.0;
        double wy = weight - wb;
        double wt = w + wy;
        wb = (wt - w) - wy;
        w = wt;
        double yx = c.x * weight - bx, yy = c.y * weight - by, yz = c.z * weight - bz;
        double tx = sx + yx, ty = sy + yy, tz = sz + yz;
        bx = (tx - sx) - yx, by = (ty - sy) - yy, bz = (tz - sz) - yz;
        sx = tx, sy = ty, sz = tz;
    }
    acc.sum[3 * p] = sx, acc.sum[3 * p + 1] = sy, acc.sum[3 * p + 2] = sz;
    acc.bias[3 * p] = bx, acc.bias[3 * p + 1] = by, acc.bias[3 * p + 2] = bz;
    acc.weight[p] = w, acc.weight_bias[p] = wb;
    double inv = 1.0 / w;
    acc.colour[3 * p] = sx * inv, acc.colour[3 * p + 1] = sy * inv, acc.colour[3 * p + 2] = sz * inv;
}

// k_resolve for one pass of an adaptive render (vrj_render_adaptive): list position i holds tile pixel list[i] (pixel i when
// `list` is NULL) and its samples are the batch's slots i * batch_samples + s.  Besides the Kahan update it keeps
// ysq[pixel] = ysq + y * y in sample order, y being the sample's Y exactly as it enters colour_sum (the noise estimate of
// k_adaptive_select).
template <typename R>
__global__ void k_resolve_adaptive(AccumDev acc, double *ysq, const uint32_t *list, const double2 *photons, uint32_t n, uint32_t batch_samples) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint32_t p = list ? list[i] : i;
    double sx = acc.sum[3 * p], sy = acc.sum[3 * p + 1], sz = acc.sum[3 * p + 2];
    double bx = acc.bias[3 * p], by = acc.bias[3 * p + 1], bz = acc.bias[3 * p + 2];
    double w = acc.weight[p], wb = acc.weight_bias[p], q = ysq[p];
    for (uint32_t s = 0; s < batch_samples; s++) { // accumulation_buffer.rs:44-60, as in k_resolve
        double2 ph = photons[(size_t)i * batch_samples + s];
        D3 c = d3(0.0, 0.0, 0.0);
        if (__double_as_longlong(ph.y) != 0ll) c = convert<double>(cmf<R>((R)ph.x) * (R)ph.y);
        const double weight = 1.0;
        double wy = weight - wb;
        double wt = w + wy;
        wb = (wt - w) - wy;
        w = wt;
        double yx = c.x * weight - bx, yy = c.y * weight - by, yz = c.z * weight - bz;
        double tx = sx + yx, ty = sy + yy, tz = sz + yz;
        bx = (tx - sx) - yx, by = (ty - sy) - yy, bz = (tz - sz) - yz;
        sx = tx, sy = ty, sz = tz;
        q = q + c.y * c.y;
    }
    acc.sum[3 * p] = sx, acc.sum[3 * p + 1] = sy, acc.sum[3 * p + 2] = sz;
    acc.bias[3 * p] = bx, acc.bias[3 * p + 1] = by, acc.bias[3 * p + 2] = bz;
    acc.weight[p] = w, acc.weight_bias[p] = wb;
    ysq[p] = q;
    double inv = 1.0 / w;
    acc.colour[3 * p] = sx * inv, acc.colour[3 * p + 1] = sy * inv, acc.colour[3 * p + 2] = sz * inv;
}

// The stopping rule of vrj_render_adaptive on the n pixels of the pass just resolved (list as in k_resolve_adaptive), in the
// order the header states it so a caller can replay it bit for bit: n = weight, s = colour_sum.y, q = y_sq_sum,
// m = s / n (as s * (1/n)), v = max(0, (q - s m) / (n - 1)), t = rel_error * max(m, abs_floor); converged iff v <= t t n.
// A NaN anywhere fails the comparison: such a pixel keeps sampling.  flag[i] = 1 if pixel i takes another pass (`more` is 0
// when the pass reached max_samples); flag[n] = 0, so the exclusive scan of flag[0..n] ends in the next pass's length.
static __global__ void k_adaptive_select(const double *sum, const double *weight, const double *ysq, const uint32_t *list, uint32_t n,
                                         double rel_error, double abs_floor, uint32_t more, uint32_t *flag, unsigned long long *converged) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    bool conv = false;
    if (i < n) {
        const uint32_t p = list ? list[i] : i;
        const double w = weight[p], s = sum[3 * p + 1], q = ysq[p];
        const double m = s * (1.0 / w);
        double v = (q - s * m) / (w - 1.0);
        if (v < 0.0) v = 0.0;
        const double t = rel_error * (m > abs_floor ? m : abs_floor);
        conv = v <= t * t * w;
        flag[i] = !conv && more ? 1u : 0u;
    } else if (i == n) {
        flag[n] = 0u;
    }
    const uint32_t c = __reduce_add_sync(0xffffffffu, conv ? 1u : 0u);
    if ((threadIdx.x & 31) == 0 && c) atomicAdd(converged, (unsigned long long)c);
}

// order-preserving compaction behind the scan of k_adaptive_select's flags: the next pass's list stays row-major, so its
// camera rays stay as coherent as the tile's
static __global__ void k_adaptive_compact(const uint32_t *list, const uint32_t *offset, uint32_t n, uint32_t *next) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n && offset[i + 1] != offset[i]) next[offset[i]] = list ? list[i] : i;
}

// Several calls rendered as ONE wavefront (vanrijn_cuda.cu, "coalesced calls"): the batch's samples [first[c], first[c] +
// count[c]) belong to call c, whose buffer starts from zero like a fresh AccumulationBuffer (camera.rs:101).  Call c's arrays
// are the c-th npix-sized piece of each output array; `full` = 0: only the colours are wanted.
constexpr int MULTI_MAX_CALLS = 16;
struct MultiCalls {
    uint32_t n, full;
    uint32_t first[MULTI_MAX_CALLS], count[MULTI_MAX_CALLS];
    AccumDev out;
};
// one thread per (pixel, call), call fastest: a warp reads consecutive photons and writes runs of whole pixels per call
template <typename R>
__global__ void k_resolve_multi(MultiCalls mc, const double2 *photons, uint32_t npix, uint32_t batch_samples) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= npix * mc.n) return; // npix * n <= 2^32 is checked by the host
    const uint32_t p = i / mc.n, c = i - p * mc.n;
    double sx = 0.0, sy = 0.0, sz = 0.0, bx = 0.0, by = 0.0, bz = 0.0, w = 0.0, wb = 0.0;
    const uint32_t s0 = mc.first[c], s1 = s0 + mc.count[c];
    for (uint32_t s = s0; s < s1; s++) { // accumulation_buffer.rs:44-60, as in k_resolve
        double2 ph = photons[(size_t)p * batch_samples + s];
        D3 col = d3(0.0, 0.0, 0.0);
        if (__double_as_longlong(ph.y) != 0ll) col = convert<double>(cmf<R>((R)ph.x) * (R)ph.y);
        const double weight = 1.0;
        double wy = weight - wb;
        double wt = w + wy;
        wb = (wt - w) - wy;
        w = wt;
        double yx = col.x * weight - bx, yy = col.y * weight - by, yz = col.z * weight - bz;
        double tx = sx + yx, ty = sy + yy, tz = sz + yz;
        bx = (tx - sx) - yx, by = (ty - sy) - yy, bz = (tz - sz) - yz;
        sx = tx, sy = ty, sz = tz;
    }
    const size_t q = (size_t)c * npix + p;
    double inv = 1.0 / w;
    mc.out.colour[3 * q] = sx * inv, mc.out.colour[3 * q + 1] = sy * inv, mc.out.colour[3 * q + 2] = sz * inv;
    if (mc.full) {
        mc.out.sum[3 * q] = sx, mc.out.sum[3 * q + 1] = sy, mc.out.sum[3 * q + 2] = sz;
        mc.out.bias[3 * q] = bx, mc.out.bias[3 * q + 1] = by, mc.out.bias[3 * q + 2] = bz;
        mc.out.weight[q] = w, mc.out.weight_bias[q] = wb;
    }
}

// debug output (VrjAccumOut.photons) is sample-major: [(sample * npix + pixel)]
static __global__ void k_photons_sample_major(const double2 *__restrict__ photons, double2 *__restrict__ out, uint32_t npix, uint32_t batch_samples) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; // output index
    if (i >= (size_t)npix * batch_samples) return;
    const uint32_t s = (uint32_t)(i / npix), p = (uint32_t)(i - (size_t)s * npix);
    out[i] = photons[(size_t)p * batch_samples + s];
}

// ---- k_tone_map: ClampingToneMapper (image.rs:130-187) ----
// colour_xyz.rs:78-84, constants as written there (12.98 / 1.005, not the sRGB standard's 12.92 / 1.055)
__device__ __forceinline__ double srgb_gamma(double u) { return u <= 0.0031308 ? 12.98 * u : 1.005 * pow(u, 1.0 / 2.4) - 0.055; }
// f64::clamp(0,1) then `(v * 255.0) as u8` (image.rs:120-123,136-138): truncation, saturating, NaN -> 0
__device__ __forceinline__ unsigned char clamp_to_byte(double v) {
    v = v < 0.0 ? 0.0 : (v > 1.0 ? 1.0 : v);
    double b = v * 255.0;
    return b != b ? (unsigned char)0 : (unsigned char)(int)b;
}
static __global__ void k_tone_map(const double *colour, unsigned char *rgb8, uint64_t n, int source) {
    uint64_t p = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= n) return;
    D3 c = d3(colour[3 * p], colour[3 * p + 1], colour[3 * p + 2]);
    if (source == 0) {
        // ColourXyz::to_linear_rgb (colour_xyz.rs:48-56) as Mat3 * Vec3, then the gamma per channel (:69-75)
        D3 lin = d3(dot(d3(3.24096994, -1.53738318, -0.49861076), c), dot(d3(-0.96924364, 1.87596750, 0.04155506), c),
                    dot(d3(0.05563008, -0.20397696, 1.05697151), c));
        c = d3(srgb_gamma(lin.x), srgb_gamma(lin.y), srgb_gamma(lin.z));
    }
    rgb8[3 * p] = clamp_to_byte(c.x), rgb8[3 * p + 1] = clamp_to_byte(c.y), rgb8[3 * p + 2] = clamp_to_byte(c.z);
}

// Sampler::sample on a caller-supplied ray list (the bit-exact id gate): same stages as the render path
template <bool COUNT>
__global__ void __launch_bounds__(128) k_stage_ray_list(DevScene sc, uint32_t n, const double *origins, const double *dirs,
                                                        PathQueue q, TraceBuffers tb, uint32_t *list_count,
                                                        unsigned long long *stats) {
    LocalStats ls;
    ls.clear();
    const uint32_t padded = (n + 31u) & ~31u;
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < padded; i += gridDim.x * blockDim.x) {
        D3 o = d3(0, 0, 0), d = d3(0, 0, 1);
        if (i < n) {
            o = d3(origins[3 * (size_t)i], origins[3 * (size_t)i + 1], origins[3 * (size_t)i + 2]);
            d = normalize(d3(dirs[3 * (size_t)i], dirs[3 * (size_t)i + 1], dirs[3 * (size_t)i + 2])); // Ray::new
            q.q0[i] = make_double2(o.x, o.y);
            q.q1[i] = make_double2(o.z, d.x);
            q.q2[i] = make_double2(d.y, d.z);
            ls.v[ST_PRIMARY]++;
        }
        stage_ray<COUNT>(sc, i < n, i, o, d, tb, list_count, ls);
    }
    ls.flush(stats);
}

static __global__ void k_hit_ids(DevScene sc, uint32_t n, TraceBuffers tb, int32_t *object_id, int32_t *prim_id, double *t,
                          unsigned long long *stats) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    int2 h = tb.hits[i];
    if (h.x < 0) {
        object_id[i] = -1, prim_id[i] = -1, t[i] = CUDART_INF;
        atomicAdd(stats + ST_MISSED, 1ull);
        return;
    }
    ItemDev it = sc.items[h.x];
    object_id[i] = (int32_t)it.object_id;
    if (it.kind >= 2) {
        D3 v0, v1, v2;
        uint32_t mat, pid;
        load_tri_pos(sc, h.y, v0, v1, v2, mat, pid);
        prim_id[i] = (int32_t)pid;
    } else {
        prim_id[i] = (int32_t)it.prim_id;
    }
    t[i] = tb.tbest[i];
}

} // namespace vrj
