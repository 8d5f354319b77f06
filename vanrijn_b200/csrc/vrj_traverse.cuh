// vrj_traverse.cuh -- closest-hit query (Sampler::sample, sampler.rs:9-20) over the flattened scene.
//
// The BVH keeps the reference's topology (median split, <= 1 triangle per leaf) but is walked
// front-to-back with t_max pruning through a CONSERVATIVE box filter; every triangle that
// survives the filter is decided by the exact binary64 Triangle::intersect arithmetic, and ties
// follow the reference's rule (bounding_volume_hierarchy.rs:77-92: the later leaf in DFS order
// wins; sampler.rs:14-19 / vec_aggregate.rs:13-21: the earlier object wins).  The filter may
// only ever pass MORE boxes than the reference's slab test (axis_aligned_bounding_box.rs:9-27),
// so it cannot change a result; its precision (f32 or f64 nodes) is a speed knob only.
#pragma once
#include "vrj_device.cuh"

#include <type_traits>

namespace vrj {

struct ItemDev {
    uint32_t kind, index, object_id, prim_id;
    uint32_t root; // VRJ_ITEM_BVH: index of the root wide node
    uint32_t pad;
    float lo[3], hi[3]; // VRJ_ITEM_BVH: the root's box, rounded outward (pre-test before a ray is queued for traversal)
};

struct DevScene {
    const float4 *__restrict__ nodes32;  // 4 x float4 per wide node (64 B)
    const double2 *__restrict__ nodes64; // 7 x double2 per wide node (112 B)
    const float4 *__restrict__ nodes4;   // 8 x float4 per 4-wide node (128 B): 4 boxes, 4 refs (VRJ_FILTER_F32X4)
    const uint4 *__restrict__ nodesq;    // 2 x uint4 per 2-wide node (32 B): boxes on a 16-bit grid, 2 refs (VRJ_FILTER_Q16)
    double qlo[3], qcell[3];             // that grid: plane coordinate = qlo + q * qcell
    const double2 *__restrict__ tri_pos; // 96-byte records (3 x 256-bit loads): 9 coords + {material, prim_id} + pad
    const double2 *__restrict__ tri_nrm; // 96-byte records: 9 coords + pad
    const float4 *__restrict__ tri_pos32; // f32-fast mode: 48-byte records, 9 coords + {material, prim_id} + pad
    const float4 *__restrict__ tri_nrm32; // 48-byte records: 9 coords + pad
    const SphereDev *__restrict__ spheres;
    const PlaneDev *__restrict__ planes;
    const MaterialDev *__restrict__ materials;
    const SpectrumDev *__restrict__ spectra;
    const double *__restrict__ spectrum_samples;
    const double *__restrict__ spectrum_grids; // wavelength of every sample (same indexing): i / (n-1) * range + shortest
    const ItemDev *__restrict__ items;
    uint32_t n_items;
    // the same items split by kind for the persistent traversal: indices into items[]
    const uint32_t *__restrict__ analytic_items; // spheres, planes, flat-list triangles
    const uint32_t *__restrict__ bvh_items;
    uint32_t n_analytic, n_bvh_items;
    uint32_t material_mask; // bit k: a material of kind k exists (selects the kernel variant; the kernels do not read it)
    // persistent-traversal tuning (lanes): refill when this many lanes are idle; run postponed leaf tests when this many are parked
    int refill_threshold, leaf_threshold, node_batch, max_iters, node_batch4;
    double cam[3];
};

template <typename R>
struct HitT {
    R t;
    int item; // -1 = miss
    int tri;  // triangle index (absolute) for triangle hits
};
typedef HitT<double> Hit;
template <typename R>
__device__ __forceinline__ R real_inf();
template <>
__device__ __forceinline__ double real_inf<double>() { return CUDART_INF; }
template <>
__device__ __forceinline__ float real_inf<float>() { return CUDART_INF_F; }

struct TraceCounters {
    uint32_t node_visits, tri_tests;
};

#define VRJ_LEAF_DONE (-2147483647 - 1)

template <typename T>
struct FilterTraits;
template <>
struct FilterTraits<float> {
    static __device__ __forceinline__ float rel() { return 9.5367431640625e-07f; }  // 2^-20
    static __device__ __forceinline__ double abs_factor() { return 9.5367431640625e-07; }
    static __device__ __forceinline__ double big() { return 1e18; }
    static __device__ __forceinline__ float down(double v) { return __double2float_rd(v); }
    static __device__ __forceinline__ float up(double v) { return __double2float_ru(v); }
    static __device__ __forceinline__ float near(double v) { return __double2float_rn(v); }
    // f32-fast mode: the ray constants are already binary32; the relative pads absorb the missing directed rounding
    static __device__ __forceinline__ float down(float v) { return v; }
    static __device__ __forceinline__ float up(float v) { return v; }
    static __device__ __forceinline__ float near(float v) { return v; }
    static __device__ __forceinline__ float fma_(float a, float b, float c) { return fmaf(a, b, c); }
    static __device__ __forceinline__ float max_(float a, float b) { return fmaxf(a, b); }
    static __device__ __forceinline__ float min_(float a, float b) { return fminf(a, b); }
    static __device__ __forceinline__ float abs_(float a) { return fabsf(a); }
};
template <>
struct FilterTraits<double> {
    static __device__ __forceinline__ double rel() { return 9.094947017729282e-13; }  // 2^-40
    static __device__ __forceinline__ double abs_factor() { return 9.094947017729282e-13; }
    static __device__ __forceinline__ double big() { return 1e150; }
    static __device__ __forceinline__ double down(double v) { return v; }
    static __device__ __forceinline__ double up(double v) { return v; }
    static __device__ __forceinline__ double near(double v) { return v; }
    static __device__ __forceinline__ double fma_(double a, double b, double c) { return fma(a, b, c); }
    static __device__ __forceinline__ double max_(double a, double b) { return fmax(a, b); }
    static __device__ __forceinline__ double min_(double a, double b) { return fmin(a, b); }
    static __device__ __forceinline__ double abs_(double a) { return fabs(a); }
};

// Per-ray constants of the conservative slab filter: t = b * id - o * id with the o*id term
// shifted by an absolute pad (rounding of o, 1/d and the box to NodeT) in the widening direction;
// a relative pad is applied to the final enter / exit values.
template <typename T>
struct FilterRay {
    T id[3], cn[3], cf[3];
};
template <typename T, typename R>
__device__ __forceinline__ FilterRay<T> filter_ray(V3<R> o, V3<R> d) {
    typedef FilterTraits<T> F;
    FilterRay<T> f;
    const R oo[3] = {o.x, o.y, o.z}, dd[3] = {d.x, d.y, d.z};
#pragma unroll
    for (int k = 0; k < 3; k++) {
        R id = R(1) / dd[k];
        if (!(fabs(id) <= (R)F::big())) id = copysign((R)F::big(), dd[k]);
        R ood = oo[k] * id;
        R pad = fabs(ood) * (R)F::abs_factor() + (sizeof(R) == 8 ? R(1e-300) : R(1e-30));
        f.id[k] = F::near(id);
        f.cn[k] = F::down(-(ood + pad));
        f.cf[k] = F::up(-(ood - pad));
    }
    return f;
}
// the prune bound of the filter for a best distance t: rounded up in the node type with the filter's relative slack
template <typename T, typename R>
__device__ __forceinline__ T filter_limit(R t) {
    typedef FilterTraits<T> F;
    return F::up(t * (R(1) + R(4) * (R)F::rel()));
}
// the constants of no ray (a lane that holds none)
template <typename T>
__device__ __forceinline__ void clear_filter(FilterRay<T> &f) {
#pragma unroll
    for (int k = 0; k < 3; k++) f.id[k] = f.cn[k] = f.cf[k] = (T)0;
}
template <typename T>
__device__ __forceinline__ bool box_filter(const FilterRay<T> &f, T lox, T hix, T loy, T hiy, T loz, T hiz, T t_limit,
                                           T &enter) {
    typedef FilterTraits<T> F;
    T nx = f.id[0] < (T)0 ? hix : lox, fx = f.id[0] < (T)0 ? lox : hix;
    T ny = f.id[1] < (T)0 ? hiy : loy, fy = f.id[1] < (T)0 ? loy : hiy;
    T nz = f.id[2] < (T)0 ? hiz : loz, fz = f.id[2] < (T)0 ? loz : hiz;
    T tn = F::max_(F::max_(F::fma_(nx, f.id[0], f.cn[0]), F::fma_(ny, f.id[1], f.cn[1])), F::fma_(nz, f.id[2], f.cn[2]));
    T tf = F::min_(F::min_(F::fma_(fx, f.id[0], f.cf[0]), F::fma_(fy, f.id[1], f.cf[1])), F::fma_(fz, f.id[2], f.cf[2]));
    T ep = F::fma_(-F::rel(), F::abs_(tn), tn);
    T xp = F::fma_(F::rel(), F::abs_(tf), tf);
    enter = ep;
    return (ep <= xp) && (xp >= (T)0) && (ep <= t_limit);
}

template <typename T>
struct WideNode {
    T c0[6], c1[6]; // lo.x, hi.x, lo.y, hi.y, lo.z, hi.z
    int left, right;
};
// 256-bit read-only loads (sm_100: LDG.E.256): a 64-byte node is two L1 transactions per lane instead of four --
// k_trace is bound by L1 wavefronts (every lane fetches a different node), not by bytes.
__device__ __forceinline__ void ldg256(const void *p, float4 &a, float4 &b) {
    asm volatile("ld.global.nc.v8.f32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=f"(a.x), "=f"(a.y), "=f"(a.z), "=f"(a.w), "=f"(b.x), "=f"(b.y), "=f"(b.z), "=f"(b.w)
                 : "l"(p));
}
__device__ __forceinline__ void ldg256(const void *p, double2 &a, double2 &b) {
    asm volatile("ld.global.nc.v4.f64 {%0,%1,%2,%3}, [%4];" : "=d"(a.x), "=d"(a.y), "=d"(b.x), "=d"(b.y) : "l"(p));
}
__device__ __forceinline__ void load_node(const DevScene &sc, int i, WideNode<float> &n) {
    const float4 *p = sc.nodes32 + (size_t)i * 4;
    float4 a, b, c, kf;
    ldg256(p, a, b);
    ldg256(p + 2, c, kf);
    n.c0[0] = a.x, n.c0[1] = a.y, n.c0[2] = a.z, n.c0[3] = a.w, n.c0[4] = c.x, n.c0[5] = c.y;
    n.c1[0] = b.x, n.c1[1] = b.y, n.c1[2] = b.z, n.c1[3] = b.w, n.c1[4] = c.z, n.c1[5] = c.w;
    n.left = __float_as_int(kf.x), n.right = __float_as_int(kf.y);
}
__device__ __forceinline__ void load_node(const DevScene &sc, int i, WideNode<double> &n) {
    const double2 *p = sc.nodes64 + (size_t)i * 7;
    double2 a = __ldg(p), b = __ldg(p + 1), c = __ldg(p + 2), d = __ldg(p + 3), e = __ldg(p + 4), g = __ldg(p + 5);
    int4 k = __ldg(reinterpret_cast<const int4 *>(p + 6));
    n.c0[0] = a.x, n.c0[1] = a.y, n.c0[2] = b.x, n.c0[3] = b.y, n.c0[4] = c.x, n.c0[5] = c.y;
    n.c1[0] = d.x, n.c1[1] = d.y, n.c1[2] = e.x, n.c1[3] = e.y, n.c1[4] = g.x, n.c1[5] = g.y;
    n.left = k.x, n.right = k.y;
}

__device__ __forceinline__ void load_tri_pos(const DevScene &sc, int tri, D3 &v0, D3 &v1, D3 &v2, uint32_t &material,
                                             uint32_t &prim_id) {
    const double2 *p = sc.tri_pos + (size_t)tri * 6;
    double2 a, b, c, d, e, f;
    ldg256(p, a, b);
    ldg256(p + 2, c, d);
    ldg256(p + 4, e, f);
    v0 = d3(a.x, a.y, b.x), v1 = d3(b.y, c.x, c.y), v2 = d3(d.x, d.y, e.x);
    long long bits = __double_as_longlong(e.y);
    material = (uint32_t)(bits & 0xffffffffll), prim_id = (uint32_t)((unsigned long long)bits >> 32);
}
__device__ __forceinline__ void load_tri_nrm(const DevScene &sc, int tri, D3 &n0, D3 &n1, D3 &n2) {
    const double2 *p = sc.tri_nrm + (size_t)tri * 6;
    double2 a, b, c, d, e, f;
    ldg256(p, a, b);
    ldg256(p + 2, c, d);
    ldg256(p + 4, e, f);
    n0 = d3(a.x, a.y, b.x), n1 = d3(b.y, c.x, c.y), n2 = d3(d.x, d.y, e.x);
}

__device__ __forceinline__ void load_tri_pos(const DevScene &sc, int tri, F3 &v0, F3 &v1, F3 &v2, uint32_t &material, uint32_t &prim_id) {
    const float4 *p = sc.tri_pos32 + (size_t)tri * 3;
    const float4 a = __ldg(p), b = __ldg(p + 1), c = __ldg(p + 2);
    v0 = F3{a.x, a.y, a.z}, v1 = F3{a.w, b.x, b.y}, v2 = F3{b.z, b.w, c.x};
    material = __float_as_uint(c.y), prim_id = __float_as_uint(c.z);
}
__device__ __forceinline__ void load_tri_nrm(const DevScene &sc, int tri, F3 &n0, F3 &n1, F3 &n2) {
    const float4 *p = sc.tri_nrm32 + (size_t)tri * 3;
    const float4 a = __ldg(p), b = __ldg(p + 1), c = __ldg(p + 2);
    n0 = F3{a.x, a.y, a.z}, n1 = F3{a.w, b.x, b.y}, n2 = F3{b.z, b.w, c.x};
}

// ------------------------------------------------------------------------------------------
// The node formats.  Each gives the walks below its per-ray filter constants (Ray, formed by ray(sc, o, d)), its prune
// bound for a best distance t (limit(t)), its stack depth, the node steps the persistent engine runs between warp votes
// (batch(sc)), and one node step: fetch node `cur`, test its children, push the farther hit children and descend into the
// nearest.  When no child is hit, step() calls `miss` instead, with `cur` still naming the node: the caller's pop or the
// end of the BVH.

// 2-wide nodes over NT boxes (nodes32 / nodes64)
template <typename NT>
struct Nodes2 {
    typedef FilterRay<NT> Ray;
    typedef NT Limit;
    static constexpr int STACK = 32;
    static __device__ __forceinline__ int batch(const DevScene &sc) { return sc.node_batch; }
    template <typename R>
    static __device__ __forceinline__ Ray ray(const DevScene &, V3<R> o, V3<R> d) { return filter_ray<NT>(o, d); }
    template <typename R>
    static __device__ __forceinline__ NT limit(R t) { return filter_limit<NT>(t); }
    template <bool COUNT, typename Miss>
    static __device__ __forceinline__ void step(const DevScene &sc, const Ray &fr, NT limit, int &cur, int *stack, int &sp,
                                                TraceCounters &cnt, Miss miss) {
        WideNode<NT> n;
        load_node(sc, cur, n);
        if (COUNT) cnt.node_visits += 2;
        NT e0, e1;
        bool h0 = box_filter(fr, n.c0[0], n.c0[1], n.c0[2], n.c0[3], n.c0[4], n.c0[5], limit, e0);
        bool h1 = box_filter(fr, n.c1[0], n.c1[1], n.c1[2], n.c1[3], n.c1[4], n.c1[5], limit, e1);
        if (h0 && h1) {
            bool swap = e1 < e0;
            stack[sp++] = swap ? n.left : n.right;
            cur = swap ? n.right : n.left;
        } else if (h0 || h1) {
            cur = h0 ? n.left : n.right;
        } else {
            miss();
        }
    }
};

// 4-wide nodes with f32 boxes (nodes4, vrj_scene_prep.cuh): one 128-byte fetch decides four boxes, the hit children are
// ordered by entry distance with a 5-comparator network, the nearest is followed and the others are pushed farthest first.
// Same filter as Nodes2<float>: results are identical to the 2-wide walk; only the number of dependent fetches per ray (about
// half) differs.
__device__ __forceinline__ void cswap(float &ka, int &ra, float &kb, int &rb) {
    const bool sw = kb < ka;
    const float k = sw ? kb : ka, K = sw ? ka : kb;
    const int r = sw ? rb : ra, R = sw ? ra : rb;
    ka = k, kb = K, ra = r, rb = R;
}
struct Nodes4 {
    typedef FilterRay<float> Ray;
    typedef float Limit;
    static constexpr int STACK = 48; // up to three pushes per 4-wide level, 16 levels
    static __device__ __forceinline__ int batch(const DevScene &sc) { return sc.node_batch4; }
    template <typename R>
    static __device__ __forceinline__ Ray ray(const DevScene &, V3<R> o, V3<R> d) { return filter_ray<float>(o, d); }
    template <typename R>
    static __device__ __forceinline__ float limit(R t) { return filter_limit<float>(t); }
    template <bool COUNT, typename Miss>
    static __device__ __forceinline__ void step(const DevScene &sc, const Ray &fr, float limit, int &cur, int *stack, int &sp,
                                                TraceCounters &cnt, Miss miss) {
        const float4 *p = sc.nodes4 + (size_t)cur * 8;
        float4 a, b, c, d, e, f, g, h;
        ldg256(p, a, b);
        ldg256(p + 2, c, d);
        ldg256(p + 4, e, f);
        ldg256(p + 6, g, h);
        if (COUNT) cnt.node_visits += 4;
        float k0, k1, k2, k3;
        const bool h0 = box_filter(fr, a.x, a.y, a.z, a.w, b.x, b.y, limit, k0);
        const bool h1 = box_filter(fr, b.z, b.w, c.x, c.y, c.z, c.w, limit, k1);
        const bool h2 = box_filter(fr, d.x, d.y, d.z, d.w, e.x, e.y, limit, k2);
        const bool h3 = box_filter(fr, e.z, e.w, f.x, f.y, f.z, f.w, limit, k3);
        int r0 = __float_as_int(g.x), r1 = __float_as_int(g.y), r2 = __float_as_int(g.z), r3 = __float_as_int(g.w);
        const float inf = CUDART_INF_F;
        k0 = h0 ? k0 : inf, k1 = h1 ? k1 : inf, k2 = h2 ? k2 : inf, k3 = h3 ? k3 : inf;
        const int nh = (int)h0 + (int)h1 + (int)h2 + (int)h3;
        // misses carry +inf and sink to the end; a hit's key is finite (its box test passed ep <= limit)
        cswap(k0, r0, k1, r1), cswap(k2, r2, k3, r3), cswap(k0, r0, k2, r2), cswap(k1, r1, k3, r3), cswap(k1, r1, k2, r2);
        if (nh == 0) {
            miss();
        } else {
            if (nh > 3) stack[sp++] = r3;
            if (nh > 2) stack[sp++] = r2;
            if (nh > 1) stack[sp++] = r1;
            cur = r0;
        }
    }
};

// 2-wide nodes on a 16-bit grid (nodesq, VRJ_FILTER_Q16): half the bytes per step.  A box plane is qlo + q * qcell; with
// A = qcell / d (binary32) and B = (qlo - o) / d - 2^23 * A (formed in binary64 from the ROUNDED A, then rounded to binary32
// away from the ray's interval, with a pad for q * (A - qcell / d)), the parameter of the plane is fma(2^23 + q, A, B):
// one PRMT builds the float 2^23 + q from a 16-bit field, the bias cancels inside the fused multiply-add.  The box a ray
// sees is at most two cells larger per side than the real one (one from the outward quantisation, one from rounding B),
// never smaller; every triangle is still decided by the exact binary64 test, so results do not change.  All meshes share
// the scene's grid, so a ray's constants hold for every BVH it visits.
struct FilterRayQ {
    float A[3], Bn[3], Bf[3];
    uint32_t neg; // bit k: the direction is negative on axis k (the near plane is the box's hi plane)
};
__device__ __forceinline__ FilterRayQ filter_ray_q(const DevScene &sc, D3 o, D3 d) {
    FilterRayQ f;
    const double oo[3] = {o.x, o.y, o.z}, dd[3] = {d.x, d.y, d.z};
    f.neg = 0;
#pragma unroll
    for (int k = 0; k < 3; k++) {
        double id = 1.0 / dd[k];
        if (!(fabs(id) <= 1e18)) id = copysign(1e18, dd[k]);
        const float A = __double2float_rn(sc.qcell[k] * id);
        const double shift = (sc.qlo[k] - oo[k]) * id;
        const double B = shift - 8388608.0 * (double)A;
        // q * (A - cell/d) <= 65535 * 2^-24 * |A|;  binary64 rounding of `shift` and B;  a floor so the pad is never zero
        const double pad = fabs((double)A) * 0.0079 + (fabs(shift) + fabs(B)) * 1e-15 + 1e-300;
        f.A[k] = A, f.Bn[k] = __double2float_rd(B - pad), f.Bf[k] = __double2float_ru(B + pad);
        if (id < 0.0) f.neg |= 1u << k;
    }
    return f;
}
__device__ __forceinline__ void clear_filter(FilterRayQ &f) {
    f.neg = 0;
#pragma unroll
    for (int k = 0; k < 3; k++) f.A[k] = f.Bn[k] = f.Bf[k] = 0.f;
}
struct NodesQ16 {
    typedef FilterRayQ Ray;
    typedef float Limit;
    static constexpr int STACK = 32;
    static __device__ __forceinline__ int batch(const DevScene &sc) { return sc.node_batch; }
    static __device__ __forceinline__ Ray ray(const DevScene &sc, D3 o, D3 d) { return filter_ray_q(sc, o, d); }
    template <typename R>
    static __device__ __forceinline__ float limit(R t) { return filter_limit<float>(t); }
    // parameter interval of child `sel` (0x7610: low halves, 0x7632: high halves) of the node words
    static __device__ __forceinline__ bool child_test(const Ray &fr, float limit, uint32_t nx, uint32_t fx, uint32_t ny, uint32_t fy,
                                                      uint32_t nz, uint32_t fz, uint32_t sel, float &enter) {
        typedef FilterTraits<float> F;
        const float qnx = __uint_as_float(__byte_perm(nx, 0x4b000000u, sel)), qfx = __uint_as_float(__byte_perm(fx, 0x4b000000u, sel));
        const float qny = __uint_as_float(__byte_perm(ny, 0x4b000000u, sel)), qfy = __uint_as_float(__byte_perm(fy, 0x4b000000u, sel));
        const float qnz = __uint_as_float(__byte_perm(nz, 0x4b000000u, sel)), qfz = __uint_as_float(__byte_perm(fz, 0x4b000000u, sel));
        const float tn = fmaxf(fmaxf(fmaf(qnx, fr.A[0], fr.Bn[0]), fmaf(qny, fr.A[1], fr.Bn[1])), fmaf(qnz, fr.A[2], fr.Bn[2]));
        const float tf = fminf(fminf(fmaf(qfx, fr.A[0], fr.Bf[0]), fmaf(qfy, fr.A[1], fr.Bf[1])), fmaf(qfz, fr.A[2], fr.Bf[2]));
        const float ep = fmaf(-F::rel(), fabsf(tn), tn), xp = fmaf(F::rel(), fabsf(tf), tf);
        enter = ep;
        return (ep <= xp) && (xp >= 0.f) && (ep <= limit);
    }
    template <bool COUNT, typename Miss>
    static __device__ __forceinline__ void step(const DevScene &sc, const Ray &fr, float limit, int &cur, int *stack, int &sp,
                                                TraceCounters &cnt, Miss miss) {
        const uint4 *p = sc.nodesq + (size_t)cur * 2;
        uint4 a, b;
        asm volatile("ld.global.nc.v8.u32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                     : "=r"(a.x), "=r"(a.y), "=r"(a.z), "=r"(a.w), "=r"(b.x), "=r"(b.y), "=r"(b.z), "=r"(b.w)
                     : "l"(p));
        if (COUNT) cnt.node_visits += 2;
        const bool ngx = fr.neg & 1u, ngy = fr.neg & 2u, ngz = fr.neg & 4u;
        const uint32_t nx = ngx ? a.y : a.x, fx = ngx ? a.x : a.y;
        const uint32_t ny = ngy ? a.w : a.z, fy = ngy ? a.z : a.w;
        const uint32_t nz = ngz ? b.y : b.x, fz = ngz ? b.x : b.y;
        float e0, e1;
        const bool h0 = child_test(fr, limit, nx, fx, ny, fy, nz, fz, 0x7610u, e0);
        const bool h1 = child_test(fr, limit, nx, fx, ny, fy, nz, fz, 0x7632u, e1);
        const int left = (int)b.z, right = (int)b.w;
        if (h0 && h1) {
            bool swap = e1 < e0;
            stack[sp++] = swap ? left : right;
            cur = swap ? right : left;
        } else if (h0 || h1) {
            cur = h0 ? left : right;
        } else {
            miss();
        }
    }
};

// The leaf of triangle `tri`: the exact Triangle::intersect, and the rule "later DFS leaf wins ties" inside one BVH
// (bounding_volume_hierarchy.rs:77-92).  Returns true when the triangle became the best.
template <bool COUNT, typename R>
__device__ __forceinline__ bool leaf_test(const DevScene &sc, const TriRayT<R> &tr, int tri, R &best_t, int &best_tri,
                                          TraceCounters &cnt) {
    V3<R> v0, v1, v2, loc;
    uint32_t mat, pid;
    load_tri_pos(sc, tri, v0, v1, v2, mat, pid);
    if (COUNT) cnt.tri_tests += 1;
    R dist, b0, b1, b2;
    if (triangle_test(tr, v0, v1, v2, dist, b0, b1, b2, loc)) {
        if (dist < best_t || (dist == best_t && tri > best_tri)) {
            best_t = dist, best_tri = tri;
            return true;
        }
    }
    return false;
}

// One BoundingVolumeHierarchy::intersect by one thread: closest triangle with distance rule "later DFS leaf wins ties".
// `t_limit` (distance of the best hit found in EARLIER objects) only prunes; the caller merges.
template <typename Format, bool COUNT, bool ANY, typename R>
__device__ __forceinline__ void bvh_closest(const DevScene &sc, int root, const TriRayT<R> &tr, const typename Format::Ray &fr,
                                            R t_limit, R &best_t, int &best_tri, TraceCounters &cnt) {
    int stack[Format::STACK];
    int sp = 0;
    int cur = root;
    best_t = real_inf<R>(), best_tri = -1;
    // prune bound in the node type, rounded up, with the relative slack of the filter
    typename Format::Limit limit = Format::limit(t_limit);
    while (true) {
        while (cur >= 0) {
            Format::template step<COUNT>(sc, fr, limit, cur, stack, sp, cnt, [&]() { cur = sp ? stack[--sp] : VRJ_LEAF_DONE; });
        }
        if (cur == VRJ_LEAF_DONE) break;
        if (leaf_test<COUNT>(sc, tr, ~cur, best_t, best_tri, cnt)) {
            if (ANY) return;
            limit = Format::limit(fmin(best_t, t_limit));
        }
        cur = sp ? stack[--sp] : VRJ_LEAF_DONE;
        if (cur == VRJ_LEAF_DONE) break;
    }
}

// Sampler::sample.  ANY = true stops at the first hit found (shadow rays: only Some/None is used).  QUAD walks the 4-wide
// form of the tree: half the dependent fetches, which is what a single thread following one path to its end (k_tail) waits on.
template <typename NT, bool COUNT, bool ANY, typename R, bool QUAD = false>
__device__ __forceinline__ HitT<R> trace_closest(const DevScene &sc, V3<R> o, V3<R> d, TraceCounters &cnt) {
    typedef typename std::conditional<QUAD, Nodes4, Nodes2<NT>>::type Format;
    HitT<R> best;
    best.t = real_inf<R>(), best.item = -1, best.tri = -1;
    bool have_tri_ray = false;
    TriRayT<R> tr;
    for (uint32_t i = 0; i < sc.n_items; i++) {
        ItemDev it = sc.items[i];
        R t;
        int tri = -1;
        bool hit = false;
        if (it.kind == 0) {
            hit = sphere_test(sc.spheres[it.index], o, d, t);
        } else if (it.kind == 1) {
            hit = plane_test(sc.planes[it.index], o, d, t);
        } else {
            if (!have_tri_ray) tr = tri_ray(o, d), have_tri_ray = true;
            if (it.kind == 2) {
                V3<R> v0, v1, v2, loc;
                uint32_t mat, pid;
                R b0, b1, b2;
                load_tri_pos(sc, (int)it.index, v0, v1, v2, mat, pid);
                if (COUNT) cnt.tri_tests += 1;
                hit = triangle_test(tr, v0, v1, v2, t, b0, b1, b2, loc);
                tri = (int)it.index;
            } else {
                typename Format::Ray fr = Format::ray(sc, o, d);
                bvh_closest<Format, COUNT, ANY>(sc, (int)it.root, tr, fr, best.item < 0 ? real_inf<R>() : best.t, t, tri, cnt);
                hit = tri >= 0;
            }
        }
        // Iterator::min_by: the kept element is replaced only when kept > candidate (NaN keeps)
        if (hit && (best.item < 0 || best.t > t)) {
            best.t = t, best.item = (int)i, best.tri = tri;
            if (ANY) return best;
        }
    }
    return best;
}

// ------------------------------------------------------------------------------------------
// Closest hit, stage 1 (runs inside the fully-SIMD ray-producing kernels): the analytic objects
// (spheres, planes, flat-list triangles) and a conservative pre-test of every BVH's root box.
// Returns the best analytic hit and whether the ray has to be queued for BVH traversal.
template <bool COUNT, typename R>
__device__ __forceinline__ bool pretrace(const DevScene &sc, V3<R> o, V3<R> d, HitT<R> &best, TraceCounters &cnt, FilterRay<float> &fr) {
    best.t = real_inf<R>(), best.item = -1, best.tri = -1;
    for (uint32_t a = 0; a < sc.n_analytic; a++) {
        uint32_t i = sc.analytic_items[a];
        ItemDev it = sc.items[i];
        R t;
        int tri = -1;
        bool hit;
        if (it.kind == 0) hit = sphere_test(sc.spheres[it.index], o, d, t);
        else if (it.kind == 1) hit = plane_test(sc.planes[it.index], o, d, t);
        else {
            TriRayT<R> tr = tri_ray(o, d);
            V3<R> v0, v1, v2, loc;
            uint32_t mat, pid;
            R b0, b1, b2;
            load_tri_pos(sc, (int)it.index, v0, v1, v2, mat, pid);
            if (COUNT) cnt.tri_tests += 1;
            hit = triangle_test(tr, v0, v1, v2, t, b0, b1, b2, loc);
            tri = (int)it.index;
        }
        // sampler.rs:14-19 (min_by keeps the earlier object on ties); items are visited in object order here
        if (hit && (best.item < 0 || t < best.t)) best.t = t, best.item = (int)i, best.tri = tri;
    }
    bool need = false;
    if (sc.n_bvh_items) {
        fr = filter_ray<float>(o, d);
        float limit = filter_limit<float>(best.t);
        for (uint32_t b = 0; b < sc.n_bvh_items; b++) {
            ItemDev it = sc.items[sc.bvh_items[b]];
            float e;
            need = need || box_filter(fr, it.lo[0], it.hi[0], it.lo[1], it.hi[1], it.lo[2], it.hi[2], limit, e);
        }
    }
    return need;
}

// ------------------------------------------------------------------------------------------
// A ray staged for BVH traversal, with everything the walk needs already formed by the kernel that produced the ray
// (k_raygen / k_shade run with full warps; inside the persistent walk only the few lanes that have run dry would do this
// work -- two binary64 divisions for the triangle test's shear, three for the slab filter -- at 8 to 16 lanes of 32).
// 96 bytes = three 256-bit loads; records are written compacted, so the lanes that refill together read neighbours.
//   v0: origin.x, origin.y, origin.z, shear x          (binary64)
//   v1: shear y, distance of the best hit of the other objects (binary64); filter 1/d x, y, z, near-offset x (binary32)
//   v2: near-offset y, z, far-offset x, y, z (binary32); flags (perm | sign(pd.z) << 2); queue entry; item of that best hit
struct TraceRec {
    double2 a0, a1, b0;
    float4 b1;
    float4 c0;
    uint4 c1;
};
static_assert(sizeof(TraceRec) == 96, "TraceRec is three 32-byte vectors");
__device__ __forceinline__ void store_trace_rec(TraceRec *recs, uint32_t pos, const TriRayT<double> &tr, const FilterRay<float> &fr,
                                                double t_best, int item, uint32_t j) {
    double2 *p = reinterpret_cast<double2 *>(recs + pos);
    p[0] = make_double2(tr.o.x, tr.o.y);
    p[1] = make_double2(tr.o.z, tr.sx);
    p[2] = make_double2(tr.sy, t_best);
    reinterpret_cast<float4 *>(p)[3] = make_float4(fr.id[0], fr.id[1], fr.id[2], fr.cn[0]);
    reinterpret_cast<float4 *>(p)[4] = make_float4(fr.cn[1], fr.cn[2], fr.cf[0], fr.cf[1]);
    reinterpret_cast<uint4 *>(p)[5] = make_uint4(__float_as_uint(fr.cf[2]), (uint32_t)tr.perm | (sign_bit(tr.pdz) ? 4u : 0u), j, (uint32_t)item);
}
__device__ __forceinline__ uint32_t load_trace_rec(const TraceRec *recs, uint32_t r, TriRayT<double> &tr, FilterRay<float> &fr, HitT<double> &best) {
    const double2 *p = reinterpret_cast<const double2 *>(recs + r);
    double2 a0, a1, b0, b1d, c0d, c1d;
    ldg256(p, a0, a1);
    ldg256(p + 2, b0, b1d);
    ldg256(p + 4, c0d, c1d);
    tr.o = d3(a0.x, a0.y, a1.x), tr.sx = a1.y, tr.sy = b0.x;
    best.t = b0.y;
    const float id0 = __int_as_float(__double2loint(b1d.x)), id1 = __int_as_float(__double2hiint(b1d.x));
    const float id2 = __int_as_float(__double2loint(b1d.y)), cn0 = __int_as_float(__double2hiint(b1d.y));
    const float cn1 = __int_as_float(__double2loint(c0d.x)), cn2 = __int_as_float(__double2hiint(c0d.x));
    const float cf0 = __int_as_float(__double2loint(c0d.y)), cf1 = __int_as_float(__double2hiint(c0d.y));
    const float cf2 = __int_as_float(__double2loint(c1d.x));
    const uint32_t flags = (uint32_t)__double2hiint(c1d.x);
    fr.id[0] = id0, fr.id[1] = id1, fr.id[2] = id2, fr.cn[0] = cn0, fr.cn[1] = cn1, fr.cn[2] = cn2, fr.cf[0] = cf0, fr.cf[1] = cf1, fr.cf[2] = cf2;
    tr.perm = (int)(flags & 3u), tr.pdz = (flags & 4u) ? -1.0 : 1.0; // only the sign of pd.z is used (triangle.rs:63)
    best.item = __double2hiint(c1d.y), best.tri = -1; // the triangle of an analytic hit stays in hits[]: it is only rewritten on improvement
    return (uint32_t)__double2loint(c1d.y);
}

// ------------------------------------------------------------------------------------------
// Closest hit, stage 2: the persistent-thread BVH engine, over any node format above.  Every lane owns one ray at a time;
// when enough lanes of the warp have run dry they write their results and fetch new rays with ONE warp-aggregated atomic,
// so short traversals do not hold the warp hostage to the longest one.  Box steps run in small batches between warp votes;
// exact triangle tests are postponed until several lanes are parked at a leaf (or nobody has box work left), so the
// expensive binary64 test runs with many lanes.
//
// Semantics: objects compete with "smaller distance wins, earlier object wins ties" (sampler.rs:14-19),
// triangles inside one BVH with "later DFS leaf wins ties" (bounding_volume_hierarchy.rs:77-92).
//
// Source:  uint32_t load_setup<Format>(const DevScene &sc, uint32_t r, TriRay &tr, Format::Ray &fr, Hit &best) -- staged ray
//          r: the constants of the exact triangle test and of the slab filter, and the best hit of the other objects;
//          returns the sink's handle
// Sink:    void store(uint32_t handle, const Hit &best, bool improved)
template <typename Format, typename R, bool COUNT, typename Source, typename Sink>
__device__ __forceinline__ void trace_persistent(const DevScene &sc, uint32_t n, uint32_t *work, Source &source, Sink &sink,
                                                 TraceCounters &cnt) {
    typedef typename Format::Limit Limit;
    const unsigned FULL = 0xffffffffu;
    const uint32_t NONE = 0xffffffffu;
    const uint32_t lane = threadIdx.x & 31;
    const int refill_threshold = sc.refill_threshold, leaf_threshold = sc.leaf_threshold;
    const int node_batch = Format::batch(sc), max_iters = sc.max_iters;
    int stack[Format::STACK];
    int sp = 0, cur = VRJ_LEAF_DONE;
    uint32_t r = NONE, bcur = 0;
    bool improved = false;
    TriRayT<R> tr;
    typename Format::Ray fr;
    HitT<R> best;
    R loc_t = real_inf<R>();
    int loc_tri = -1;
    Limit limit = (Limit)0;
    bool exhausted = false;
    tr.o = V3<R>{R(0), R(0), R(0)}, tr.sx = tr.sy = tr.pdz = R(0), tr.perm = 0;
    best.t = real_inf<R>(), best.item = -1, best.tri = -1;
    clear_filter(fr);

    // the current BVH's closest triangle competes with the best of the other objects, then the next BVH starts
    auto finish_bvh = [&]() {
        uint32_t item = sc.bvh_items[bcur];
        if (loc_tri >= 0 && (best.item < 0 || loc_t < best.t || (loc_t == best.t && (int)item < best.item)))
            best.t = loc_t, best.item = (int)item, best.tri = loc_tri, improved = true;
        bcur++;
        if (bcur < sc.n_bvh_items) {
            cur = (int)sc.items[sc.bvh_items[bcur]].root;
            sp = 0, loc_t = real_inf<R>(), loc_tri = -1;
            limit = Format::limit(best.t);
        } else {
            cur = VRJ_LEAF_DONE;
        }
    };

    while (true) {
        // ---- results out, new rays in ----
        bool idle = cur == VRJ_LEAF_DONE;
        unsigned idle_mask = __ballot_sync(FULL, idle);
        if (idle_mask) {
            if (idle && r != NONE) {
                sink.store(r, best, improved);
                r = NONE;
            }
            if (exhausted) {
                if (idle_mask == FULL) break;
            } else if (idle_mask == FULL || __popc(idle_mask) >= refill_threshold) {
                uint32_t want = (uint32_t)__popc(idle_mask), base = 0;
                int leader = __ffs(idle_mask) - 1;
                if ((int)lane == leader) base = atomicAdd(work, want);
                base = __shfl_sync(FULL, base, leader);
                if (base + want >= n) exhausted = true;
                if (idle) {
                    uint32_t my = base + (uint32_t)__popc(idle_mask & ((1u << lane) - 1u));
                    if (my < n) {
                        r = source.template load_setup<Format>(sc, my, tr, fr, best); // the handle the sink stores the result under
                        improved = false;
                        bcur = 0;
                        cur = (int)sc.items[sc.bvh_items[0]].root;
                        sp = 0, loc_t = real_inf<R>(), loc_tri = -1;
                        limit = Format::limit(best.t);
                    }
                }
            }
        }
        // ---- traverse until enough lanes have run dry ----
#pragma unroll 1
        for (int it = 0; it < max_iters; it++) {
#pragma unroll 1
            for (int u = 0; u < node_batch; u++)
                if (cur >= 0) Format::template step<COUNT>(sc, fr, limit, cur, stack, sp, cnt, [&]() {
                    if (sp) cur = stack[--sp];
                    else finish_bvh();
                });
            bool at_leaf = cur < 0 && cur != VRJ_LEAF_DONE;
            unsigned leaf_mask = __ballot_sync(FULL, at_leaf);
            unsigned node_mask = __ballot_sync(FULL, cur >= 0);
            if (leaf_mask && (node_mask == 0 || __popc(leaf_mask) >= leaf_threshold)) {
                if (at_leaf) {
                    if (leaf_test<COUNT>(sc, tr, ~cur, loc_t, loc_tri, cnt)) limit = Format::limit(fmin(loc_t, best.t));
                    if (sp) cur = stack[--sp];
                    else finish_bvh();
                }
            }
            unsigned done_mask = __ballot_sync(FULL, cur == VRJ_LEAF_DONE);
            if (done_mask == FULL || (!exhausted && __popc(done_mask) >= refill_threshold)) break;
        }
    }
}

// Rebuild the IntersectionInfo (raycasting/mod.rs:67-97) of a known hit with the exact arithmetic
// of the primitive's intersect(): the wavefront stores only (ray, item, triangle).
// `t` is the distance the closest-hit query found for this hit (the value of the primitive's own intersect(), computed by the
// same code on the same ray), so spheres and planes go straight to their frame; triangles need their barycentrics again.
template <typename R>
__device__ __forceinline__ bool rebuild_hit(const DevScene &sc, V3<R> o, V3<R> d, int item, int tri, R t, HitFrameT<R> &h) {
    ItemDev it = sc.items[item];
    if (it.kind == 0) {
        sphere_frame(sc.spheres[it.index], o, d, t, h);
        return true;
    }
    if (it.kind == 1) {
        plane_frame(sc.planes[it.index], o, d, t, h);
        return true;
    }
    TriRayT<R> tr = tri_ray(o, d);
    V3<R> v0, v1, v2, n0, n1, n2;
    uint32_t mat, pid;
    R b0, b1, b2;
    load_tri_pos(sc, tri, v0, v1, v2, mat, pid);
    if (!triangle_test(tr, v0, v1, v2, h.distance, b0, b1, b2, h.location)) return false;
    load_tri_nrm(sc, tri, n0, n1, n2);
    // triangle.rs:73-83
    h.normal = normalize(((V3<R>{R(0), R(0), R(0)} + n0 * b0) + n1 * b1) + n2 * b2);
    h.cotangent = normalize(cross(v0 - v1, h.normal));
    h.tangent = normalize(cross(h.cotangent, h.normal));
    h.retro = normalize(o - h.location);
    h.material = mat;
    return true;
}

} // namespace vrj
