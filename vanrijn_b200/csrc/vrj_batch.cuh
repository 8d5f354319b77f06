// vrj_batch.cuh -- one wavefront batch (launch sequence of the kernels in vrj_kernels.cuh) and the host-side state it runs on.
// Shared by vanrijn_cuda.cu (the C ABI) and vrj_batch_inst.cu, which is compiled once per (box type, real type, counting)
// combination so the six instantiations of run_batch -- each with its own k_shade / k_tail / k_trace variants -- build in
// parallel instead of in one translation unit.
#pragma once
#include "../../include/vanrijn_cuda.h"
#include "vrj_kernels.cuh"
#include "vrj_internal.h"

#include <algorithm>
#include <mutex>
#include <string>
#include <unordered_map>
#include <vector>

// NVTX ranges around the wavefront stages (SURVEY section 5): header-only NVTX 3 (vanrijn_cuda.cu), no-ops unless a tool is attached.
void vrj_nvtx_push(const char *name);
void vrj_nvtx_pop();
struct VrjNvtxRange {
    explicit VrjNvtxRange(const char *name) { vrj_nvtx_push(name); }
    ~VrjNvtxRange() { vrj_nvtx_pop(); }
};
#define VRJ_NVTX_RANGE(var, name) VrjNvtxRange var(name)

namespace vrjimpl {
using namespace vrj;

inline VrjStatus fail(VrjStatus code, const std::string &msg) {
    vrj_set_error(msg);
    return code;
}
#define VRJ_CUDA(expr)                                                                                      \
    do {                                                                                                    \
        cudaError_t e_ = (expr);                                                                            \
        if (e_ != cudaSuccess)                                                                              \
            return fail(e_ == cudaErrorMemoryAllocation ? VRJ_ERR_OUT_OF_MEMORY : VRJ_ERR_CUDA,             \
                        std::string(#expr) + ": " + cudaGetErrorString(e_));                                \
    } while (0)

struct DeviceBuffer {
    void *p = nullptr;
    size_t bytes = 0;
    bool borrowed = false; // p points into another buffer's block (a Scratch slab); nothing to free
    ~DeviceBuffer() { release(); }
    void release() {
        if (p && !borrowed) vrj_pool_free(p);
        p = nullptr, borrowed = false;
    }
    cudaError_t alloc(size_t n) {
        release();
        bytes = n;
        return vrj_pool_alloc(&p, n);
    }
    void borrow(void *q, size_t n) {
        release();
        p = q, bytes = n, borrowed = true;
    }
    template <typename T>
    T *as() const { return static_cast<T *>(p); }
};

// The block's page-locked slots.  Counters come back and the sample table goes out through them: a copy between the device and
// pageable memory holds the enqueueing thread until everything queued before it has finished (the render gate could not
// open before the result's copies).
struct PinnedBlock {
    uint32_t drain[4];                          // run_levels' drain check: (queue length, tail flag) of two groups of levels
    uint64_t sample_table[4 * MULTI_MAX_CALLS]; // coalesced calls: the wavefront's sample indices
    unsigned long long stats[ST_COUNT];         // the call's ray counters
    ProgressiveCounters pass;                   // render_passes: the last select's counters
    uint32_t listed;                            // render_passes: the length of a sub-pass's pixel list
    CountsCounters counts;                      // vrj_render_counts: what k_counts_check found
};

// per-call scratch: path queues, photon results, accumulators, counters
struct Scratch {
    size_t capacity = 0; // paths
    size_t npix = 0;
    uint32_t steps = 0;
    DeviceBuffer queues[2][6];
    DeviceBuffer photons, hits[2], tbest[2], list, counters, stats;
    DeviceBuffer recs;       // TraceRec per staged ray (rec_capacity of them); shared by the levels like `list`
    size_t rec_capacity = 0;
    DeviceBuffer acc_colour, acc_sum, acc_bias, acc_weight, acc_wbias;
    DeviceBuffer queue_slab, rec_slab, acc_slab; // the groups above live in one allocation each (see ensure_scratch)
    DeviceBuffer multi_out, sample_table; // coalesced calls: their output arrays (call-major pieces) and the batch's sample indices
    DeviceBuffer lights, light_samples, srgb8;
    // render_passes: y_sq_sum, the previous / next pass's pixel list, the next pass's first samples, the selects' counters
    DeviceBuffer ysq, pass_list[2], pass_base, pass_counters, pass_slab;
    // vrj_render_counts, in the same slab: the scan of the count map and its counters (per pixel), and the pixel and first
    // sample of every slot of a batch (per path in flight)
    DeviceBuffer count_offset, count_counters, slot_pixel, slot_base;
    size_t pass_npix = 0, pass_slots = 0;
    cudaStream_t stream = nullptr;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr; // first / last kernel of a call
    cudaEvent_t ev_done = nullptr;             // behind the call's last copy
    cudaStream_t copy_stream = nullptr;        // copies of resolved pieces (vrj_render_tile) run here, next to the resolve kernels
    cudaEvent_t piece_ev[8] = {};              // behind the resolve of piece i
    cudaEvent_t copy_done = nullptr;           // behind the last of those copies
    cudaEvent_t call_ev[16] = {};              // coalesced calls: behind the copies of call c (MULTI_MAX_CALLS)
    cudaEvent_t drain_ev[2] = {nullptr, nullptr}; // behind the pinned copies of the drain check (run_levels)
    std::vector<cudaEvent_t> marks; // per-launch boundaries, reused across calls
    std::vector<int> mark_class;    // class of the launch that ENDS at mark i (-1: start of a batch)
    size_t n_marks = 0;
    PinnedBlock *pinned = nullptr;
    ~Scratch() {
        if (stream) cudaStreamDestroy(stream);
        if (ev0) cudaEventDestroy(ev0);
        if (ev1) cudaEventDestroy(ev1);
        if (ev_done) cudaEventDestroy(ev_done);
        if (copy_stream) cudaStreamDestroy(copy_stream);
        if (copy_done) cudaEventDestroy(copy_done);
        for (cudaEvent_t e : piece_ev)
            if (e) cudaEventDestroy(e);
        for (cudaEvent_t e : call_ev)
            if (e) cudaEventDestroy(e);
        for (cudaEvent_t e : drain_ev)
            if (e) cudaEventDestroy(e);
        for (cudaEvent_t e : marks) cudaEventDestroy(e);
        if (pinned) cudaFreeHost(pinned);
    }
    // record a boundary event on the stream; cls = class of the launch it closes
    cudaError_t mark(int cls) {
        if (n_marks == marks.size()) {
            cudaEvent_t e;
            cudaError_t err = cudaEventCreate(&e);
            if (err != cudaSuccess) return err;
            marks.push_back(e), mark_class.push_back(cls);
        }
        mark_class[n_marks] = cls;
        return cudaEventRecord(marks[n_marks++], stream);
    }
    AccumDev accum() const {
        AccumDev a;
        a.colour = acc_colour.as<double>(), a.sum = acc_sum.as<double>(), a.bias = acc_bias.as<double>();
        a.weight = acc_weight.as<double>(), a.weight_bias = acc_wbias.as<double>();
        return a;
    }
    TraceBuffers trace_buffers(int i, bool records = false) const {
        TraceBuffers t;
        t.hits = hits[i].as<int2>(), t.tbest = tbest[i].as<double>(), t.list = list.as<uint32_t>();
        t.recs = records ? recs.as<TraceRec>() : nullptr;
        return t;
    }
    PathQueue queue(int i) const {
        PathQueue q;
        q.q0 = queues[i][0].as<double2>(), q.q1 = queues[i][1].as<double2>(), q.q2 = queues[i][2].as<double2>();
        q.q3 = queues[i][3].as<double2>(), q.q4 = queues[i][4].as<double2>(), q.q5 = queues[i][5].as<uint4>();
        return q;
    }
};

} // namespace vrjimpl

struct VrjScene {
    int device = 0;
    int sm_count = 0;
    uint64_t device_bytes = 0;
    uint64_t upload_bytes = 0;
    vrj::DevScene dev{};
    std::vector<vrjimpl::DeviceBuffer *> owned;
    uint32_t n_spectra = 0;
    uint32_t tail_max = 1u << 18; // queue length at which k_tail finishes the batch in one launch (0 = never)
    uint32_t tail_max_shallow = 0; // the same for recursion limits <= 12
    uint64_t path_budget = 1ull << 27; // paths in flight per batch
    bool auto_q16 = false; // VRJ_FILTER_F32 calls walk the 16-bit nodes: set for scenes whose f32 nodes exceed L2 (effective_filter)
    bool trace_records = true; // staged rays carry their traversal constants (TraceRec); VRJ_RECORDS=0 turns it off (experiments)
    uint32_t kernel_material_mask = VRJ_MM_ALL; // 1: every material is Lambertian (the Lambertian-only kernel variants run)
    ~VrjScene() {
        for (auto *b : owned) delete b;
    }
};

namespace vrjimpl {

// resident CTAs per SM of a kernel at 128 threads; asked once per kernel (the query costs tens of microseconds and a
// 1-spp call makes five of them)
template <typename K>
int persistent_grid(const VrjScene *sc, K kernel) {
    static std::mutex m;
    static std::unordered_map<const void *, int> cache;
    const void *key = reinterpret_cast<const void *>(kernel);
    {
        std::lock_guard<std::mutex> g(m);
        auto it = cache.find(key);
        if (it != cache.end()) return sc->sm_count * it->second;
    }
    int per_sm = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, 128, 0) != cudaSuccess || per_sm < 1) per_sm = 1;
    std::lock_guard<std::mutex> g(m);
    cache[key] = per_sm;
    return sc->sm_count * per_sm;
}

// which calls walk ready-made records: the 2-wide f32 walk of the binary64 path (the default and the bench's)
template <typename NT, typename R>
inline bool wants_records(const VrjScene *sc, int walk) {
    return sizeof(NT) == 4 && sizeof(R) == 8 && walk == 0 && sc->trace_records && sc->dev.n_bvh_items > 0;
}

// One batch with the integrator (WHITTED) and the scene's material kinds (MM, see vrj_device.cuh) fixed at compile time.  It
// leaves the batch's photons in s->photons, pixel-major; the caller resolves them.
template <typename NT, typename R, bool COUNT, bool WHITTED, int MM, bool LIST>
VrjStatus run_levels(const VrjScene *sc, Scratch *s, const RenderConst &rc, int walk, uint64_t *launches) {
    const bool quad = walk == 1, q16 = walk == 2; // 0: the 2-wide tree in NT boxes; 1: 4-wide f32; 2: 2-wide on the 16-bit grid
    // launch sequence: G T S_0 [X_k T_k S_k]*, k = 1..levels (X = k_tail, a no-op until the queue is short);
    // SimpleRandom needs max_depth levels, Whitted one more (its limit-0 level still shades and traces);
    // the final S only finishes paths.
    const uint32_t levels = WHITTED ? rc.max_depth + 1 : rc.max_depth;
    const uint32_t stride = rc.max_depth + 3;
    uint32_t *qcount = s->counters.as<uint32_t>(); // qcount[k]: length of the queue S_{k-1} wrote (k >= 1)
    uint32_t *lcount = qcount + stride;             // lcount[k]: rays of queue k staged for BVH traversal
    uint32_t *work_t = lcount + stride;             // work-fetch counters of T_k
    uint32_t *work_s = work_t + stride;             // ... of G (k = 0 only) / S_k
    uint32_t *tail_done = work_s + stride;          // set by the k_tail launch that finished the batch
    VRJ_CUDA(cudaMemsetAsync(qcount, 0, ((size_t)stride * 5 + 2) * sizeof(uint32_t), s->stream));
    unsigned long long *stats = s->stats.as<unsigned long long>();
    double2 *photons = s->photons.as<double2>();
    const int g_gen = persistent_grid(sc, k_raygen<R, COUNT, LIST>), g_t = quad ? persistent_grid(sc, k_trace4<COUNT, false>) : q16 ? persistent_grid(sc, k_traceq<COUNT, false>) : persistent_grid(sc, k_trace<NT, R, COUNT>);
    const int g_t0 = quad ? persistent_grid(sc, k_trace4<COUNT, true, LIST>) : q16 ? persistent_grid(sc, k_traceq<COUNT, true, LIST>) : persistent_grid(sc, k_trace_primary<NT, R, COUNT, LIST>);
    const int g_s0 = persistent_grid(sc, k_shade<NT, R, COUNT, WHITTED, true, MM, LIST>);
    const int g_s = persistent_grid(sc, k_shade<NT, R, COUNT, WHITTED, false, MM, LIST>);
    // k_tail pays off for deep recursion limits (the reference's 128: 260 launches -> 28); at depth <= 12 the
    // per-level latency it removes is smaller than what its one-thread-per-path traversal costs (measured)
    const uint32_t tail_max = levels > 12 ? sc->tail_max : sc->tail_max_shallow;
    const int g_x = tail_max ? persistent_grid(sc, k_tail<NT, R, COUNT, WHITTED, MM, LIST>) : 0; // persistent warps, per-lane refill
    uint32_t *tail_work = tail_done + 1 + stride;   // k_tail's work-fetch counter (after the k_stage counters)
    const bool has_bvh = sc->dev.n_bvh_items > 0;
    // the default walk of the parity path takes its rays as ready-to-walk records (TraceRec); the other walks form the
    // traversal constants per lane from the queue entry
    const bool rec = wants_records<NT, R>(sc, walk) && s->rec_capacity >= (size_t)rc.npix * rc.batch_samples;
    const TraceBuffers tb0 = s->trace_buffers(0, rec), tb1 = s->trace_buffers(1, rec);
    const int g_tr = rec ? persistent_grid(sc, k_trace_rec<COUNT>) : 0;
    VRJ_NVTX_RANGE(batch_range, "vrj batch");
    VRJ_CUDA(s->mark(-1));
    // the raygen kernel uses work_s[0]; S_0 uses work_t[stride-1] (never used by a T)
    k_raygen<R, COUNT, LIST><<<g_gen, 128, 0, s->stream>>>(sc->dev, rc, s->queue(0), tb0, lcount + 0, work_s + 0, stats);
    (*launches)++;
    VRJ_CUDA(s->mark(4));
    if (has_bvh) {
        if (rec) k_trace_rec<COUNT><<<g_tr, 128, 0, s->stream>>>(sc->dev, tb0, lcount + 0, work_t + 0, stats, tail_done);
        else if (quad) k_trace4<COUNT, true, LIST><<<g_t0, 128, 0, s->stream>>>(sc->dev, rc, s->queue(0), tb0, lcount + 0, work_t + 0, stats, tail_done);
        else if (q16) k_traceq<COUNT, true, LIST><<<g_t0, 128, 0, s->stream>>>(sc->dev, rc, s->queue(0), tb0, lcount + 0, work_t + 0, stats, tail_done);
        else k_trace_primary<NT, R, COUNT, LIST><<<g_t0, 128, 0, s->stream>>>(sc->dev, rc, tb0, lcount + 0, work_t + 0, stats);
        (*launches)++;
        VRJ_CUDA(s->mark(0));
    }
    uint32_t *work_s0 = work_t + (stride - 1);
    k_shade<NT, R, COUNT, WHITTED, true, MM, LIST><<<g_s0, 128, 0, s->stream>>>(sc->dev, rc, s->queue(0), nullptr, tb0, s->queue(1), qcount + 1, tb1, lcount + 1, work_s0, photons, stats, tail_done);
    (*launches)++;
    VRJ_CUDA(s->mark(3));
    bool drain_pending = false;
#if VRJ_SPLIT_STAGE
    const int g_st = persistent_grid(sc, k_stage<R, COUNT>);
    uint32_t *work_st = tail_done + 1; // work-fetch counters of the k_stage launches (stride entries)
#endif
    for (uint32_t k = 1; k <= levels; k++) {
        const int ci = k & 1, ni = (k + 1) & 1;
        VRJ_NVTX_RANGE(level_range, "vrj level: tail / trace / shade");
#if VRJ_SPLIT_STAGE
        k_stage<R, COUNT><<<g_st, 128, 0, s->stream>>>(sc->dev, s->queue(ci), qcount + k, ci ? tb1 : tb0, lcount + k, work_st + k, stats, tail_done);
        (*launches)++;
        VRJ_CUDA(s->mark(4));
#endif
        if (tail_max) {
            k_tail<NT, R, COUNT, WHITTED, MM, LIST><<<g_x, 128, 0, s->stream>>>(sc->dev, rc, s->queue(ci), qcount + k, tail_max, photons, stats, tail_done, tail_work);
            (*launches)++;
            VRJ_CUDA(s->mark(5));
        }
        if (has_bvh) {
            const TraceBuffers &tbc = ci ? tb1 : tb0;
            if (rec) k_trace_rec<COUNT><<<g_tr, 128, 0, s->stream>>>(sc->dev, tbc, lcount + k, work_t + k, stats, tail_done);
            else if (quad) k_trace4<COUNT, false><<<g_t, 128, 0, s->stream>>>(sc->dev, rc, s->queue(ci), tbc, lcount + k, work_t + k, stats, tail_done);
            else if (q16) k_traceq<COUNT, false><<<g_t, 128, 0, s->stream>>>(sc->dev, rc, s->queue(ci), tbc, lcount + k, work_t + k, stats, tail_done);
            else k_trace<NT, R, COUNT><<<g_t, 128, 0, s->stream>>>(sc->dev, s->queue(ci), tbc, lcount + k, work_t + k, stats, tail_done);
            (*launches)++;
            VRJ_CUDA(s->mark(1));
        }
        k_shade<NT, R, COUNT, WHITTED, false, MM, LIST><<<g_s, 128, 0, s->stream>>>(sc->dev, rc, s->queue(ci), qcount + k, ci ? tb1 : tb0, s->queue(ni), qcount + k + 1, ni ? tb1 : tb0, lcount + k + 1, work_s + k, photons, stats, tail_done);
        (*launches)++;
        VRJ_CUDA(s->mark(3));
        // Deep recursion limits (the reference's 128): stop launching once the batch has drained (queue empty, or finished
        // by k_tail).  The check never stalls the launch pipeline: after a group of four levels the queue length and the tail
        // flag are copied to a pinned slot behind an event, the next group is enqueued, and only then does the host look at
        // the PREVIOUS group's slot -- the GPU always has a group queued while the host waits, at the price of at most one
        // group of launches that return at once.
        if (levels > 12 && k % 4 == 0 && k < levels) {
            const int slot = (int)(k / 4) & 1;
            if (drain_pending) {
                VRJ_CUDA(cudaEventSynchronize(s->drain_ev[slot ^ 1]));
                if (s->pinned->drain[2 * (slot ^ 1)] == 0 || s->pinned->drain[2 * (slot ^ 1) + 1] != 0) break;
            }
            VRJ_CUDA(cudaMemcpyAsync(s->pinned->drain + 2 * slot, qcount + k + 1, sizeof(uint32_t), cudaMemcpyDeviceToHost, s->stream));
            VRJ_CUDA(cudaMemcpyAsync(s->pinned->drain + 2 * slot + 1, tail_done, sizeof(uint32_t), cudaMemcpyDeviceToHost, s->stream));
            VRJ_CUDA(cudaEventRecord(s->drain_ev[slot], s->stream));
            drain_pending = true;
        }
    }
    VRJ_CUDA(cudaGetLastError());
    return VRJ_OK;
}

// kernel variants exist for "Lambertian only" (the reference's own scenes: main.rs, benches/simple_scene.rs) and for
// "any material"; VRJ_MATERIAL_MASK=15 in the environment forces the general variant (experiments)
template <typename NT, typename R, bool COUNT, bool LIST>
VrjStatus run_materials(const VrjScene *sc, Scratch *s, const RenderConst &rc, bool whitted, int walk, uint64_t *launches) {
    const bool lambert_only = sc->kernel_material_mask == 1u;
    if (whitted)
        return lambert_only ? run_levels<NT, R, COUNT, true, 1, LIST>(sc, s, rc, walk, launches)
                            : run_levels<NT, R, COUNT, true, VRJ_MM_ALL, LIST>(sc, s, rc, walk, launches);
    return lambert_only ? run_levels<NT, R, COUNT, false, 1, LIST>(sc, s, rc, walk, launches)
                        : run_levels<NT, R, COUNT, false, VRJ_MM_ALL, LIST>(sc, s, rc, walk, launches);
}
// a batch over rc.pixel_list (and rc.pixel_base) runs the LIST variants of the kernels
template <typename NT, typename R, bool COUNT>
VrjStatus run_batch(const VrjScene *sc, Scratch *s, const RenderConst &rc, bool whitted, int walk, uint64_t *launches) {
    return rc.pixel_list ? run_materials<NT, R, COUNT, true>(sc, s, rc, whitted, walk, launches)
                         : run_materials<NT, R, COUNT, false>(sc, s, rc, whitted, walk, launches);
}

} // namespace vrjimpl
