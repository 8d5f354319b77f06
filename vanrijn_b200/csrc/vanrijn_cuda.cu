// vanrijn_cuda.cu -- C ABI (include/vanrijn_cuda.h) over the sm_100a wavefront kernels.
// There is no CPU fallback anywhere in this library: without a CUDA device every entry
// point that computes returns VRJ_ERR_CUDA.
#include "../../include/vanrijn_cuda.h"
#include "vrj_batch.cuh"
#include "vrj_denoise.cuh"
#include "vrj_scene_prep.cuh"
#include "vrj_internal.h"

#include <algorithm>
#include <atomic>
#include <chrono>
#include <cmath>
#include <condition_variable>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <dlfcn.h>
#include <nvtx3/nvToolsExt.h>
#include <thread>
#include <unordered_map>
#include <limits>
#include <mutex>
#include <string>
#include <vector>

using namespace vrj;
using namespace vrjimpl;

namespace {
thread_local std::string g_error;
} // namespace

// the six instantiations live in vrj_batch_inst.cu (one object file each)
namespace vrjimpl {
extern template VrjStatus run_batch<float, double, false>(const VrjScene *, Scratch *, const RenderConst &, bool, int, uint64_t *);
extern template VrjStatus run_batch<float, double, true>(const VrjScene *, Scratch *, const RenderConst &, bool, int, uint64_t *);
extern template VrjStatus run_batch<double, double, false>(const VrjScene *, Scratch *, const RenderConst &, bool, int, uint64_t *);
extern template VrjStatus run_batch<double, double, true>(const VrjScene *, Scratch *, const RenderConst &, bool, int, uint64_t *);
extern template VrjStatus run_batch<float, float, false>(const VrjScene *, Scratch *, const RenderConst &, bool, int, uint64_t *);
extern template VrjStatus run_batch<float, float, true>(const VrjScene *, Scratch *, const RenderConst &, bool, int, uint64_t *);
} // namespace vrjimpl
// NVTX ranges (SURVEY section 5) through the header-only NVTX 3: no library to link or load -- the calls are no-ops until a
// tool (ncu --nvtx, nsys) injects itself
void vrj_nvtx_push(const char *name) { nvtxRangePushA(name); }
void vrj_nvtx_pop() { nvtxRangePop(); }
// other translation units of the library (vrj_bvh_build.cu) report through the same thread-local message
void vrj_set_error(const std::string &msg) { g_error = msg; }

// ---- device memory pool ----
// cudaMalloc / cudaFree cost 4-60 ms per call on the B200 boxes (measured, and erratic), more than uploading and
// preparing a whole bunny-class scene; freed blocks are therefore kept per device and handed out again to requests
// they fit (at most 2x + 1 MiB larger than asked).  vrj_release_scratch() returns everything to the driver.
namespace {
struct PoolBlock {
    int device;
    void *p;
    size_t bytes;
};
std::mutex g_dev_pool_mutex;
std::vector<PoolBlock> g_dev_pool_free;
std::unordered_map<void *, PoolBlock> g_dev_pool_live;
const size_t kPoolCapBytes = size_t(32) << 30;
const size_t kPoolCapBlocks = 48;
} // namespace
void vrj_pool_trim() {
    std::vector<PoolBlock> victims;
    {
        std::lock_guard<std::mutex> g(g_dev_pool_mutex);
        victims.swap(g_dev_pool_free);
    }
    int cur = 0;
    cudaGetDevice(&cur);
    for (const PoolBlock &b : victims) {
        cudaSetDevice(b.device);
        cudaFree(b.p);
    }
    cudaSetDevice(cur);
}
// allocations that went to the driver (VRJ_TIMING prints them at exit: in a steady state both stay flat)
std::atomic<uint64_t> g_n_device_mallocs{0}, g_n_host_mallocs{0};
struct AllocReport {
    ~AllocReport() {
        if (std::getenv("VRJ_TIMING"))
            std::fprintf(stderr, "vanrijn_cuda: %llu cudaMalloc, %llu cudaMallocHost calls\n", (unsigned long long)g_n_device_mallocs.load(),
                         (unsigned long long)g_n_host_mallocs.load());
    }
} g_alloc_report;
cudaError_t vrj_pool_alloc(void **out, size_t bytes) {
    *out = nullptr;
    bytes = (std::max<size_t>(bytes, 256) + 255) & ~size_t(255);
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    {
        std::lock_guard<std::mutex> g(g_dev_pool_mutex);
        size_t best = g_dev_pool_free.size();
        for (size_t i = 0; i < g_dev_pool_free.size(); i++) {
            const PoolBlock &b = g_dev_pool_free[i];
            if (b.device == dev && b.bytes >= bytes && b.bytes <= 2 * bytes + (size_t(1) << 20) &&
                (best == g_dev_pool_free.size() || b.bytes < g_dev_pool_free[best].bytes))
                best = i;
        }
        if (best != g_dev_pool_free.size()) {
            PoolBlock b = g_dev_pool_free[best];
            g_dev_pool_free.erase(g_dev_pool_free.begin() + best);
            g_dev_pool_live[b.p] = b;
            *out = b.p;
            return cudaSuccess;
        }
    }
    void *p = nullptr;
    g_n_device_mallocs++;
    e = cudaMalloc(&p, bytes);
    if (e == cudaErrorMemoryAllocation) { // give the cached blocks back and try once more
        cudaGetLastError();
        vrj_pool_trim();
        e = cudaMalloc(&p, bytes);
    }
    if (e != cudaSuccess) return e;
    std::lock_guard<std::mutex> g(g_dev_pool_mutex);
    g_dev_pool_live[p] = PoolBlock{dev, p, bytes};
    *out = p;
    return cudaSuccess;
}
void vrj_pool_free(void *p) {
    if (!p) return;
    PoolBlock b{0, p, 0};
    bool keep = false;
    {
        std::lock_guard<std::mutex> g(g_dev_pool_mutex);
        auto it = g_dev_pool_live.find(p);
        if (it != g_dev_pool_live.end()) {
            b = it->second;
            g_dev_pool_live.erase(it);
            size_t cached = 0;
            for (const PoolBlock &f : g_dev_pool_free) cached += f.bytes;
            keep = cached + b.bytes <= kPoolCapBytes && g_dev_pool_free.size() < kPoolCapBlocks;
            if (keep) g_dev_pool_free.push_back(b);
        }
    }
    if (!keep) cudaFree(p);
}
namespace {

// next representable float above / below (bit arithmetic: this runs 12x per BVH node at scene upload)
inline float float_up(float f) {
    if (!(f == f) || f == std::numeric_limits<float>::infinity()) return f;
    if (f == 0.0f) return std::numeric_limits<float>::denorm_min();
    int32_t b;
    std::memcpy(&b, &f, 4);
    b += b >= 0 ? 1 : -1;
    std::memcpy(&f, &b, 4);
    return f;
}
inline float float_down(float f) { return -float_up(-f); }
inline float round_down_f32(double v) {
    float f = (float)v;
    return (double)f > v ? float_down(f) : f;
}
inline float round_up_f32(double v) {
    float f = (float)v;
    return (double)f < v ? float_up(f) : f;
}

VrjStatus validate(const VrjSceneDesc *d) {
    if (!d) return fail(VRJ_ERR_INVALID_ARGUMENT, "scene description is NULL");
    if (d->abi_version != VRJ_ABI_VERSION) return fail(VRJ_ERR_INVALID_ARGUMENT, "VrjSceneDesc.abi_version mismatch");
    if (d->n_triangles > 0x7ffffff0ull || d->n_nodes > 0x7ffffff0ull) return fail(VRJ_ERR_UNSUPPORTED, "scene too large for 31-bit indices");
    for (uint32_t i = 0; i < d->n_materials; i++) {
        if (d->materials[i].kind > VRJ_MAT_DIELECTRIC) return fail(VRJ_ERR_INVALID_ARGUMENT, "unknown material kind");
        if (d->materials[i].spectrum >= d->n_spectra) return fail(VRJ_ERR_INVALID_ARGUMENT, "material spectrum out of range");
    }
    for (uint32_t i = 0; i < d->n_spectra; i++) {
        const VrjSpectrum &s = d->spectra[i];
        if (s.n_samples < 2 || (uint64_t)s.first_sample + s.n_samples > d->n_spectrum_samples)
            return fail(VRJ_ERR_INVALID_ARGUMENT, "spectrum sample range out of bounds (need >= 2 samples)");
    }
    for (uint32_t i = 0; i < d->n_spheres; i++)
        if (d->spheres[i].material >= d->n_materials) return fail(VRJ_ERR_INVALID_ARGUMENT, "sphere material out of range");
    for (uint32_t i = 0; i < d->n_planes; i++)
        if (d->planes[i].material >= d->n_materials) return fail(VRJ_ERR_INVALID_ARGUMENT, "plane material out of range");
    for (uint64_t i = 0; i < d->n_triangles; i++)
        if (d->tri_material[i] >= d->n_materials) return fail(VRJ_ERR_INVALID_ARGUMENT, "triangle material out of range");
    for (uint32_t i = 0; i < d->n_items; i++) {
        const VrjItem &it = d->items[i];
        uint64_t lim = it.kind == VRJ_ITEM_SPHERE ? d->n_spheres : it.kind == VRJ_ITEM_PLANE ? d->n_planes
                     : it.kind == VRJ_ITEM_TRIANGLE ? d->n_triangles : it.kind == VRJ_ITEM_BVH ? d->n_bvhs : 0;
        if (it.index >= lim) return fail(VRJ_ERR_INVALID_ARGUMENT, "item index out of range");
    }
    // The C ABI is a trust boundary (a Rust caller builds these arrays): the device code indexes per-BVH temporaries with
    // `child - first_node`, walks with a 32-entry stack and breaks distance ties by triangle index, so every tree must be a
    // proper binary tree in DFS pre-order inside its own node range, no deeper than the stack, with its triangles in leaf order.
    std::vector<uint8_t> level; // 0 = not reached yet; the root is level 1
    for (uint32_t i = 0; i < d->n_bvhs; i++) {
        const VrjBvh &b = d->bvhs[i];
        if (b.first_node > d->n_nodes || b.n_nodes > d->n_nodes - b.first_node || b.first_triangle > d->n_triangles ||
            b.n_triangles > d->n_triangles - b.first_triangle)
            return fail(VRJ_ERR_INVALID_ARGUMENT, "bvh range out of bounds");
        if (b.n_nodes == 0) {
            // n_nodes == 0 with triangles: the tree is built on the device at upload (median split: depth known from n)
            if (b.n_triangles && vrj_build::tree_depth(b.n_triangles) > 31) return fail(VRJ_ERR_UNSUPPORTED, "bvh deeper than the 32-entry traversal stack");
            continue;
        }
        const uint64_t lo = b.first_node, hi = b.first_node + b.n_nodes;
        const uint64_t tlo = b.first_triangle, thi = b.first_triangle + b.n_triangles;
        level.assign((size_t)b.n_nodes, 0);
        level[0] = 1;
        uint64_t leaves = 0, leaf_triangles = 0;
        int64_t last_triangle = -1;
        for (uint64_t n = lo; n < hi; n++) {
            const uint8_t lv = level[(size_t)(n - lo)];
            if (lv == 0) return fail(VRJ_ERR_INVALID_ARGUMENT, "bvh node is not reachable from the root (nodes must be in DFS pre-order)");
            const int32_t l = d->node_child[2 * n], r = d->node_child[2 * n + 1];
            if (l >= 0) {
                // pre-order: both children come after their parent, inside this tree's range; each node has one parent
                if (r < 0 || (uint64_t)l <= n || (uint64_t)l >= hi || (uint64_t)r <= n || (uint64_t)r >= hi || l == r)
                    return fail(VRJ_ERR_INVALID_ARGUMENT, "bvh child out of range (children must follow their parent inside the bvh's own node range)");
                if (lv >= 31) return fail(VRJ_ERR_UNSUPPORTED, "bvh deeper than the 32-entry traversal stack");
                uint8_t &ll = level[(size_t)((uint64_t)l - lo)], &rl = level[(size_t)((uint64_t)r - lo)];
                if (ll || rl) return fail(VRJ_ERR_INVALID_ARGUMENT, "bvh node has two parents");
                ll = rl = (uint8_t)(lv + 1);
            } else {
                leaves++;
                if (r < 0 || r > 1) return fail(VRJ_ERR_UNSUPPORTED, "bvh leaves hold at most one triangle (as the reference builds them)");
                if (r == 1) {
                    const uint64_t t = (uint64_t)(~l);
                    if (t < tlo || t >= thi) return fail(VRJ_ERR_INVALID_ARGUMENT, "bvh leaf triangle outside the bvh's own triangle range");
                    if ((int64_t)t <= last_triangle) return fail(VRJ_ERR_INVALID_ARGUMENT, "bvh triangles must be stored in leaf (DFS) order");
                    last_triangle = (int64_t)t, leaf_triangles++;
                }
            }
        }
        if (b.n_nodes != 2 * leaves - 1) return fail(VRJ_ERR_INVALID_ARGUMENT, "bvh is not a full binary tree (n_nodes != 2 * leaves - 1)");
        if (leaf_triangles != b.n_triangles) return fail(VRJ_ERR_INVALID_ARGUMENT, "bvh leaves do not cover the bvh's triangle range");
    }
    return VRJ_OK;
}

// Scratch blocks are pooled per device for the life of the process (not per scene): a caller that creates a
// scene per frame does not pay multi-GB cudaMalloc/cudaFree each time.  vrj_release_scratch() empties the pool.
// Host arrays reach the device through one page-locked staging block kept for the life of the process (a pageable
// cudaMemcpy ran at 0.2-2 GB/s on the B200 boxes; memcpy into pinned memory + one async copy runs at PCIe speed).
// Arrays that are already page-locked (vrj_alloc_host) skip the staging copy.
// One staging block, one stream and one lock PER DEVICE: scenes for different GPUs (vrj_comm_scene_create, or one host thread
// per GPU) are prepared side by side, and nothing here touches the legacy default stream.
struct StagingArea {
    std::mutex mutex;
    char *block = nullptr;
    size_t bytes = 0;
    cudaStream_t stream = nullptr; // non-blocking; created with the first scene for the device
};
StagingArea g_staging_area[64];
struct Stager {
    StagingArea &area;
    size_t cursor = 0, copied = 0;
    cudaStream_t stream = nullptr;
    explicit Stager(StagingArea &a) : area(a) {}
    cudaError_t reserve(size_t bytes) {
        if (!area.stream) {
            cudaError_t e = cudaStreamCreateWithFlags(&area.stream, cudaStreamNonBlocking);
            if (e != cudaSuccess) return e;
        }
        stream = area.stream;
        if (area.bytes >= bytes) return cudaSuccess;
        if (area.block) cudaFreeHost(area.block), area.block = nullptr, area.bytes = 0;
        cudaError_t e = cudaMallocHost(reinterpret_cast<void **>(&area.block), bytes);
        if (e == cudaSuccess) area.bytes = bytes;
        return e;
    }
    static void parallel_memcpy(char *dst, const char *src, size_t bytes) {
        const size_t min_per_thread = size_t(4) << 20;
        unsigned hw = std::thread::hardware_concurrency();
        size_t n_threads = std::min<size_t>(std::min<size_t>(hw ? hw : 4, 8), bytes / min_per_thread);
        if (n_threads < 2) {
            std::memcpy(dst, src, bytes);
            return;
        }
        std::vector<std::thread> pool;
        const size_t per = ((bytes + n_threads - 1) / n_threads + 4095) & ~size_t(4095);
        for (size_t t = 0; t < n_threads; t++) {
            const size_t lo = t * per, hi = std::min(bytes, lo + per);
            if (lo >= hi) break;
            pool.emplace_back([=] { std::memcpy(dst + lo, src + lo, hi - lo); });
        }
        for (auto &th : pool) th.join();
    }
    cudaError_t copy(void *dst, const void *src, size_t bytes) {
        if (!bytes) return cudaSuccess;
        copied += bytes;
        cudaPointerAttributes attr;
        if (cudaPointerGetAttributes(&attr, src) == cudaSuccess && attr.type == cudaMemoryTypeHost)
            return cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, stream);
        cudaGetLastError();
        char *st = area.block + cursor;
        cursor += (bytes + 255) & ~size_t(255);
        parallel_memcpy(st, static_cast<const char *>(src), bytes);
        return cudaMemcpyAsync(dst, st, bytes, cudaMemcpyHostToDevice, stream);
    }
};

std::mutex g_pool_mutex;
std::vector<std::pair<int, Scratch *>> g_pool;
struct HostBlock {
    void *p;
    size_t bytes;
};
std::mutex g_host_pool_mutex;
std::vector<HostBlock> g_host_pool_free;
std::unordered_map<void *, size_t> g_host_pool_live;

// Blocks are kept for concurrent callers (main.rs:197-209 drives the entry point from a pool of workers, each call needing
// its own block): up to 16 per device as long as what the pool holds stays under 48 GB -- sixteen 1-spp 1080p blocks are
// 14 GB, one 64-spp block is 45 GB.  A caller is handed the smallest pooled block that is large enough, else the largest.
size_t scratch_bytes(const Scratch *s) { return s->capacity * 240 + s->rec_capacity * sizeof(TraceRec) + s->npix * 88 + s->pass_npix * 20; }
std::atomic<int> g_active_calls[64];

// Render gate: how many calls may have their wavefronts on one device at the same moment.  main.rs:197-209 drives the entry
// point from a pool of workers; every call's kernels are persistent grids sized to fill all 148 SMs, so many of them
// interleaved only evict each other's queues from L2 (1-spp 1080p calls, device time per call: 1.33 ms with two in flight,
// 1.73 with four, 2.07 with eight) -- but a few in flight pay, because a wavefront ends in a latency-bound tail (the last
// levels carry a handful of long paths) that another wavefront's bulk fills.  Callers past the gate's width wait their turn
// (FIFO) before enqueueing, and while they wait, compatible calls pile up behind them and are rendered together (see
// "coalesced calls"); the gate opens again when the call's last kernel has finished, so its copy back to the host overlaps
// the next caller's rendering.  Width 4 measured best at 4 to 16 workers once calls are coalesced (8 workers: 3.3 / 3.5 / 3.5
// Grays/s through the loop of main.rs at widths 2 / 3 / 4).  VRJ_CONCURRENT_RENDERS overrides the width (experiments).
struct RenderGate {
    std::mutex m;
    std::condition_variable cv;
    int running = 0;
    uint64_t next_ticket = 0, serving = 0;
};
RenderGate g_render_gate[64];
int render_gate_width() {
    static const int width = [] {
        const char *e = std::getenv("VRJ_CONCURRENT_RENDERS");
        return e ? std::max(1, std::atoi(e)) : 4;
    }();
    return width;
}
struct RenderTurn {
    RenderGate &g;
    bool held = false;
    explicit RenderTurn(int device) : g(g_render_gate[(unsigned)device % 64]) {}
    void acquire() {
        std::unique_lock<std::mutex> lock(g.m);
        const uint64_t ticket = g.next_ticket++;
        g.cv.wait(lock, [&] { return ticket == g.serving && g.running < render_gate_width(); });
        g.serving++, g.running++, held = true;
        g.cv.notify_all();
    }
    void release() {
        if (!held) return;
        {
            std::lock_guard<std::mutex> lock(g.m);
            g.running--, held = false;
        }
        g.cv.notify_all();
    }
    ~RenderTurn() { release(); }
};

// Waiting for the device: a lone caller spins on the event (lowest latency); when several calls are in flight on the device
// (main.rs's worker pool) a waiting thread sleeps until the GPU's interrupt instead -- eight workers spinning on their copies
// would take the cores the host's merge_tile threads need (measured: the loop of main.rs:192-217 collapsed from 1.6 to 3-17 ms
// per call once workers + merge threads exceeded the host's cores).  Events that may be slept on carry cudaEventBlockingSync.
cudaError_t wait_event(cudaEvent_t e, int device) {
    if (g_active_calls[(unsigned)device % 64].load(std::memory_order_relaxed) > 1) return cudaEventSynchronize(e);
    for (;;) {
        const cudaError_t q = cudaEventQuery(e);
        if (q != cudaErrorNotReady) return q;
    }
}
Scratch *acquire_scratch(VrjScene *sc, size_t want_capacity) {
    std::lock_guard<std::mutex> g(g_pool_mutex);
    size_t best = g_pool.size();
    for (size_t i = 0; i < g_pool.size(); i++) {
        if (g_pool[i].first != sc->device) continue;
        if (best == g_pool.size()) {
            best = i;
            continue;
        }
        const size_t c = g_pool[i].second->capacity, b = g_pool[best].second->capacity;
        const bool c_fits = c >= want_capacity, b_fits = b >= want_capacity;
        if ((c_fits && (!b_fits || c < b)) || (!c_fits && !b_fits && c > b)) best = i;
    }
    if (best != g_pool.size()) {
        Scratch *s = g_pool[best].second;
        g_pool.erase(g_pool.begin() + best);
        return s;
    }
    return new Scratch();
}
void release_scratch(VrjScene *sc, Scratch *s) {
    std::lock_guard<std::mutex> g(g_pool_mutex);
    size_t same = 0, bytes = scratch_bytes(s);
    for (auto &e : g_pool)
        if (e.first == sc->device) same++, bytes += scratch_bytes(e.second);
    if (same < 16 && (same < 2 || bytes <= (size_t(48) << 30))) g_pool.push_back({sc->device, s});
    else delete s;
}
// a call's block: whatever path leaves the call (an error in the middle of a batch loop included), nothing may still be
// running on the block's streams when another caller is handed it
struct BlockLease {
    VrjScene *sc;
    Scratch *s = nullptr;
    ~BlockLease() {
        if (!s) return;
        if (s->stream) cudaStreamSynchronize(s->stream);
        if (s->copy_stream) cudaStreamSynchronize(s->copy_stream);
        release_scratch(sc, s);
    }
};

// A group of a block's buffers is all-or-nothing: a failed allocation leaves the group empty with its size field at 0 (never
// half-sized or stale), so the block can go back to the pool and the caller can retry
// ... and ONE allocation: cudaMalloc waits for a gap in the device's work, so with another caller's persistent kernels
// running the 25 buffers of a block cost 30 ms each (measured: 840 ms for the second block of a worker pool)
VrjStatus alloc_group(DeviceBuffer &slab, std::vector<std::pair<DeviceBuffer *, size_t>> &want, const char *what) {
    for (auto &w : want) w.first->release();
    slab.release();
    size_t total = 0;
    for (auto &w : want) total += (w.second + 255) & ~size_t(255);
    cudaError_t e = slab.alloc(total);
    if (e != cudaSuccess) {
        slab.release();
        cudaGetLastError();
        return fail(e == cudaErrorMemoryAllocation ? VRJ_ERR_OUT_OF_MEMORY : VRJ_ERR_CUDA, std::string(what) + ": " + cudaGetErrorString(e));
    }
    size_t at = 0;
    for (auto &w : want) {
        w.first->borrow(static_cast<char *>(slab.p) + at, w.second);
        at += (w.second + 255) & ~size_t(255);
    }
    return VRJ_OK;
}

// `queue_oom` (optional): set when the allocation that failed was the path queues -- the only part a smaller batch shrinks
VrjStatus ensure_scratch(Scratch *s, size_t capacity, size_t rec_capacity, size_t npix, uint32_t steps, uint32_t n_lights, size_t n_light_samples, bool *queue_oom = nullptr) {
    if (queue_oom) *queue_oom = false;
    if (!s->stream) {
        VRJ_CUDA(cudaStreamCreateWithFlags(&s->stream, cudaStreamNonBlocking));
        VRJ_CUDA(cudaEventCreate(&s->ev0));
        VRJ_CUDA(cudaEventCreateWithFlags(&s->ev1, cudaEventBlockingSync)); // timing stays enabled; see wait_event
        VRJ_CUDA(cudaEventCreateWithFlags(&s->ev_done, cudaEventBlockingSync | cudaEventDisableTiming));
        for (cudaEvent_t &e : s->call_ev) VRJ_CUDA(cudaEventCreateWithFlags(&e, cudaEventBlockingSync | cudaEventDisableTiming));
        VRJ_CUDA(cudaStreamCreateWithFlags(&s->copy_stream, cudaStreamNonBlocking));
        VRJ_CUDA(cudaEventCreateWithFlags(&s->copy_done, cudaEventDisableTiming));
        for (cudaEvent_t &e : s->piece_ev) VRJ_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        for (cudaEvent_t &e : s->drain_ev) VRJ_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        VRJ_CUDA(cudaMallocHost(reinterpret_cast<void **>(&s->pinned), sizeof(PinnedBlock)));
    }
    // every group below is all-or-nothing (alloc_group)
    if (s->capacity < capacity) {
        s->capacity = 0;
        std::vector<std::pair<DeviceBuffer *, size_t>> want;
        for (int i = 0; i < 2; i++)
            for (int k = 0; k < 6; k++) want.push_back({&s->queues[i][k], capacity * 16});
        want.push_back({&s->photons, capacity * sizeof(double2)});
        for (int i = 0; i < 2; i++) want.push_back({&s->hits[i], capacity * sizeof(int2)}), want.push_back({&s->tbest[i], capacity * sizeof(double)});
        want.push_back({&s->list, capacity * sizeof(uint32_t)});
        VrjStatus st = alloc_group(s->queue_slab, want, "path queues");
        if (st != VRJ_OK) {
            if (queue_oom) *queue_oom = st == VRJ_ERR_OUT_OF_MEMORY;
            return st;
        }
        s->capacity = capacity;
    }
    if (s->rec_capacity < rec_capacity) {
        s->rec_capacity = 0;
        std::vector<std::pair<DeviceBuffer *, size_t>> want = {{&s->recs, rec_capacity * sizeof(TraceRec)}};
        VrjStatus st = alloc_group(s->rec_slab, want, "trace records");
        if (st != VRJ_OK) {
            if (queue_oom) *queue_oom = st == VRJ_ERR_OUT_OF_MEMORY;
            return st;
        }
        s->rec_capacity = rec_capacity;
    }
    if (s->npix < npix) {
        s->npix = 0;
        std::vector<std::pair<DeviceBuffer *, size_t>> want = {{&s->acc_colour, npix * 24}, {&s->acc_sum, npix * 24}, {&s->acc_bias, npix * 24},
                                                               {&s->acc_weight, npix * 8}, {&s->acc_wbias, npix * 8}};
        VrjStatus st = alloc_group(s->acc_slab, want, "accumulators");
        if (st != VRJ_OK) return st;
        s->npix = npix;
    }
    if (s->steps < steps) {
        s->steps = 0;
        cudaError_t e = s->counters.alloc(((size_t)steps * 5 + 4) * sizeof(uint32_t));
        if (e != cudaSuccess) {
            s->counters.release();
            cudaGetLastError();
            return fail(e == cudaErrorMemoryAllocation ? VRJ_ERR_OUT_OF_MEMORY : VRJ_ERR_CUDA, std::string("level counters: ") + cudaGetErrorString(e));
        }
        s->steps = steps;
    }
    if (!s->stats.p) VRJ_CUDA(s->stats.alloc(ST_COUNT * sizeof(unsigned long long)));
    if (!s->lights.p || s->lights.bytes < (size_t)(n_lights + 1) * sizeof(LightDev)) {
        s->lights.release();
        VRJ_CUDA(s->lights.alloc((size_t)(n_lights + 1) * sizeof(LightDev)));
    }
    if (!s->light_samples.p || s->light_samples.bytes < n_light_samples * sizeof(double)) {
        s->light_samples.release();
        VRJ_CUDA(s->light_samples.alloc(std::max<size_t>(2, n_light_samples) * sizeof(double)));
    }
    return VRJ_OK;
}

// Which walk a call takes.  VRJ_FILTER_F32 is the default; for scenes whose f32 nodes do not fit L2 (config C4: 634 MB) the
// library walks the 16-bit nodes instead -- half the bytes per step, +2-4 % on C4 (profiles/r02_ab_variants.txt), slower on an
// L2-resident scene.  The filter only decides which boxes are opened, never a result (every walk is bit-identical to every
// other: tests/test_gpu_parity.py, tests/test_gpu_bvh_build.py), so this is a scheduling decision.  VRJ_AUTO_Q16=0 turns it off.
uint32_t effective_filter(const VrjScene *scene, const VrjRenderParams *p) {
    if (p->bvh_filter == VRJ_FILTER_F32 && p->precision == VRJ_PRECISION_F64 && scene->auto_q16) return VRJ_FILTER_Q16;
    return p->bvh_filter;
}

// the per-call constants of the kernels (camera.rs:24-34 for the film size)
RenderConst make_render_const(const VrjTile *tile, uint64_t height, uint64_t width, const VrjRenderParams *p) {
    RenderConst rc{};
    rc.width = width, rc.height = height;
    rc.start_column = tile->start_column, rc.start_row = tile->start_row;
    rc.tile_w = (uint32_t)(tile->end_column - tile->start_column), rc.tile_h = (uint32_t)(tile->end_row - tile->start_row);
    rc.npix = rc.tile_w * rc.tile_h;
    rc.sample_stride = p->sample_stride ? p->sample_stride : 1;
    rc.seed = p->seed;
    rc.max_depth = p->max_depth, rc.n_lights = p->n_lights, rc.has_ambient = p->ambient_light ? 1u : 0u;
    // binary32 cannot represent origin + 1e-7 * direction at scene scale (ulp(5) = 4.8e-7): the fast mode needs a bias of a
    // few hundred ulps or every bounce ray re-hits the surface it leaves
    rc.bias = p->precision == VRJ_PRECISION_F32_FAST ? std::max(p->bias, 1e-4) : p->bias;
    { // camera.rs:24-34
        double w = (double)width, h = (double)height;
        if (w > h) rc.film_w = w / h, rc.film_h = 1.0;
        else rc.film_w = 1.0, rc.film_h = w / h;
    }
    return rc;
}

void fill_stats(VrjStats *st, const unsigned long long *h, uint64_t launches, float ms) {
    st->primary_rays = h[ST_PRIMARY], st->bounce_rays = h[ST_BOUNCE], st->shadow_rays = h[ST_SHADOW];
    st->paths_missed = h[ST_MISSED], st->paths_escaped = h[ST_ESCAPED], st->paths_depth_limited = h[ST_LIMITED];
    st->node_visits = h[ST_NODES], st->triangle_tests = h[ST_TRIS];
    st->staged_rays = h[ST_STAGED];
    st->kernel_launches = launches;
    st->device_ms = ms;
}


// ---------------------------------------------------------------------------------------------- shared by the render calls
// a call in flight on a device: the path budget is shared between such calls, and wait_event sleeps instead of spinning
struct ActiveCall {
    std::atomic<int> &n;
    int others;
    explicit ActiveCall(std::atomic<int> &c) : n(c), others(c.fetch_add(1)) {}
    ~ActiveCall() { n.fetch_sub(1); }
};

// the tile lies inside the image, and the image's pixel indices fit 32 bits
VrjStatus check_tile(const VrjTile *tile, uint64_t height, uint64_t width) {
    if (tile->end_column < tile->start_column || tile->end_row < tile->start_row || tile->end_column > width || tile->end_row > height)
        return fail(VRJ_ERR_INVALID_ARGUMENT, "tile outside the image");
    // width * height can wrap in 64 bits (2^32 x 2^32, 2^63 x 2): compare by division
    if (height != 0 && width > 0xffffffffull / height) return fail(VRJ_ERR_UNSUPPORTED, "image larger than 2^32 - 1 pixels");
    return VRJ_OK;
}

// the argument checks of vrj_render_tile and vrj_render_adaptive; *n_light_samples: samples of the call's light spectra
VrjStatus check_render_args(const VrjScene *scene, const VrjTile *tile, uint64_t height, uint64_t width, const VrjRenderParams *p,
                            const VrjAccumOut *out, size_t *n_light_samples) {
    if (!scene || !tile || !p || !out) return fail(VRJ_ERR_INVALID_ARGUMENT, "NULL argument");
    const VrjStatus st = check_tile(tile, height, width);
    if (st != VRJ_OK) return st;
    if (p->integrator > VRJ_INTEGRATOR_WHITTED) return fail(VRJ_ERR_INVALID_ARGUMENT, "unknown integrator");
    if (p->bvh_filter > VRJ_FILTER_Q16) return fail(VRJ_ERR_INVALID_ARGUMENT, "unknown bvh_filter");
    if (p->precision > VRJ_PRECISION_F32_FAST) return fail(VRJ_ERR_INVALID_ARGUMENT, "unknown precision");
    if (p->max_depth > 65535) return fail(VRJ_ERR_INVALID_ARGUMENT, "max_depth exceeds u16 (RECURSION_LIMIT is a u16)");
    if (p->n_lights && !p->lights) return fail(VRJ_ERR_INVALID_ARGUMENT, "lights is NULL");
    size_t n = 0;
    for (uint32_t i = 0; i < p->n_lights; i++) {
        if (p->lights[i].spectrum.n_samples < 2 || !p->lights[i].spectrum.samples) return fail(VRJ_ERR_INVALID_ARGUMENT, "light spectrum needs >= 2 samples");
        n += p->lights[i].spectrum.n_samples;
    }
    if (p->ambient_light) {
        if (p->ambient_light->n_samples < 2 || !p->ambient_light->samples) return fail(VRJ_ERR_INVALID_ARGUMENT, "ambient spectrum needs >= 2 samples");
        n += p->ambient_light->n_samples;
    }
    *n_light_samples = n;
    return VRJ_OK;
}

// Paths in flight per batch: 128 Mi by default = 45 GB of queue state (sized for 180 GB of HBM), shared between the calls
// running on this device right now, so several callers asking for many samples each do not have to find out through failed
// allocations that they cannot all have a full budget
uint64_t call_path_budget(const VrjScene *scene, const ActiveCall &active) {
    return std::max<uint64_t>(scene->path_budget / (uint64_t)(active.others + 1), std::min<uint64_t>(scene->path_budget, uint64_t(1) << 22));
}

// TraceRec records: only the calls that walk them need the extra 96 bytes per path in flight
bool call_wants_records(const VrjScene *scene, const VrjRenderParams *p, uint32_t filter) {
    return p->precision == VRJ_PRECISION_F64 && filter == VRJ_FILTER_F32 && scene->trace_records && scene->dev.n_bvh_items > 0;
}

// the block for accumulators of npix pixels and batches of *batch units of `unit` paths each (a tile's batch: samples of
// unit = npix pixels; vrj_render_counts: unit = 1 path per slot)
VrjStatus ensure_call_scratch(Scratch *s, const VrjRenderParams *p, bool records, uint64_t npix, uint64_t unit, uint32_t *batch, size_t n_light_samples) {
    bool queue_oom = false;
    auto ensure = [&] {
        return ensure_scratch(s, unit * *batch, records ? unit * *batch : 0, npix, p->max_depth + 3, p->n_lights, n_light_samples, &queue_oom);
    };
    VrjStatus st = ensure();
    while (st == VRJ_ERR_OUT_OF_MEMORY && queue_oom && *batch > 1) { // 240 bytes per path in flight: halve the batch until the queues fit
        vrj_pool_trim();
        *batch = (*batch + 1) / 2;
        st = ensure();
    }
    if (st == VRJ_ERR_OUT_OF_MEMORY && !queue_oom) { // the accumulators do not shrink with the batch: give cached blocks back, once
        vrj_pool_trim();
        st = ensure();
    }
    return st;
}

// the call's lights and ambient spectrum into the block (RenderConst::lights / light_samples)
VrjStatus stage_lights(Scratch *s, const VrjRenderParams *p) {
    if (!p->n_lights && !p->ambient_light) return VRJ_OK;
    std::vector<LightDev> lights(p->n_lights + 1);
    std::vector<double> lsamples;
    auto put = [&lsamples](const VrjSpectrumData &sd) {
        SpectrumDev d{sd.shortest_wavelength, sd.longest_wavelength, (uint32_t)lsamples.size(), sd.n_samples};
        lsamples.insert(lsamples.end(), sd.samples, sd.samples + sd.n_samples);
        return d;
    };
    for (uint32_t i = 0; i < p->n_lights; i++) {
        for (int k = 0; k < 3; k++) lights[i].dir[k] = p->lights[i].direction[k];
        lights[i].spectrum = put(p->lights[i].spectrum);
    }
    lights[p->n_lights] = LightDev{};
    if (p->ambient_light) lights[p->n_lights].spectrum = put(*p->ambient_light);
    VRJ_CUDA(cudaMemcpyAsync(s->lights.p, lights.data(), lights.size() * sizeof(LightDev), cudaMemcpyHostToDevice, s->stream));
    if (!lsamples.empty())
        VRJ_CUDA(cudaMemcpyAsync(s->light_samples.p, lsamples.data(), lsamples.size() * sizeof(double), cudaMemcpyHostToDevice, s->stream));
    VRJ_CUDA(cudaStreamSynchronize(s->stream)); // the staging vectors are locals
    return VRJ_OK;
}

// one batch in the kernel variant the call's precision, walk and counting select
VrjStatus dispatch_batch(const VrjScene *scene, Scratch *s, const RenderConst &rc, const VrjRenderParams *p, uint32_t filter, uint64_t *launches) {
    const bool whitted = p->integrator == VRJ_INTEGRATOR_WHITTED;
    // F32X4: the staged rays walk the 4-wide tree; inline any-hit queries (Whitted shadow rays, k_tail) use the 2-wide f32 tree
    const int quad = filter == VRJ_FILTER_F32X4 ? 1 : filter == VRJ_FILTER_Q16 ? 2 : 0;
    // VRJ_PRECISION_F32_FAST: the whole sample in binary32 over the 2-wide f32 tree (no reference counterpart; not a parity mode)
    const bool fast = p->precision == VRJ_PRECISION_F32_FAST;
    if (p->count_traversal)
        return fast ? run_batch<float, float, true>(scene, s, rc, whitted, 0, launches)
             : filter == VRJ_FILTER_F64 ? run_batch<double, double, true>(scene, s, rc, whitted, 0, launches)
                                        : run_batch<float, double, true>(scene, s, rc, whitted, quad, launches);
    return fast ? run_batch<float, float, false>(scene, s, rc, whitted, 0, launches)
         : filter == VRJ_FILTER_F64 ? run_batch<double, double, false>(scene, s, rc, whitted, 0, launches)
                                    : run_batch<float, double, false>(scene, s, rc, whitted, quad, launches);
}

// The resolve of the batch dispatch_batch left in s->photons: `launch` enqueues its kernels in the real type R of the call's
// colour matching (run_batch's R: float for VRJ_PRECISION_F32_FAST), then the boundary that closes the resolve (resolve_ms).
template <typename F>
VrjStatus resolve_batch(Scratch *s, const VrjRenderParams *p, F &&launch) {
    VRJ_NVTX_RANGE(resolve_range, "vrj resolve");
    const VrjStatus st = p->precision == VRJ_PRECISION_F32_FAST ? launch(float{}) : launch(double{});
    if (st != VRJ_OK) return st;
    VRJ_CUDA(s->mark(2));
    VRJ_CUDA(cudaGetLastError());
    return VRJ_OK;
}

// VrjStats of a call from its counters and the boundary events run_levels recorded
void fill_call_stats(VrjStats *st, const Scratch *s, const unsigned long long *hstats, uint64_t launches, float ms) {
    fill_stats(st, hstats, launches, ms);
    double cls_ms[6] = {0, 0, 0, 0, 0, 0}; // 0 T (camera rays), 1 T (bounce rays), 2 resolve, 3 shade, 4 raygen, 5 tail
    uint64_t cls_n[6] = {0, 0, 0, 0, 0, 0};
    for (size_t i = 1; i < s->n_marks; i++) {
        int c = s->mark_class[i];
        if (c < 0) continue;
        float seg = 0.f;
        if (cudaEventElapsedTime(&seg, s->marks[i - 1], s->marks[i]) == cudaSuccess) cls_ms[c] += seg, cls_n[c]++;
    }
    st->primary_ms = cls_ms[0], st->bounce_ms = cls_ms[1], st->resolve_ms = cls_ms[2];
    st->primary_launches = cls_n[0], st->bounce_launches = cls_n[1], st->resolve_launches = cls_n[2];
    st->shade_ms = cls_ms[3] + cls_ms[4], st->shade_launches = cls_n[3] + cls_n[4];
    st->tail_ms = cls_ms[5], st->tail_launches = cls_n[5];
    st->coalesced_calls = 1;
}

// VrjAccumOut.colour from (colour_sum, weight), as k_resolve computes it (vrj_render_sharded, render_passes)
__global__ void k_finalize(const double *sum, const double *weight, double *colour, uint32_t npix) {
    uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= npix) return;
    store_colour(colour, p, sum[3 * p], sum[3 * p + 1], sum[3 * p + 2], weight[p]);
}

// the tone-mapped colours of the block's accumulators to out->srgb8
VrjStatus copy_srgb8(Scratch *s, uint64_t npix, uint8_t *dst, cudaMemcpyKind kind, uint64_t *launches) {
    if (s->srgb8.bytes < npix * 3) {
        s->srgb8.release();
        VRJ_CUDA(s->srgb8.alloc(npix * 3));
    }
    k_tone_map<<<(unsigned)((npix + 255) / 256), 256, 0, s->stream>>>(s->acc_colour.as<double>(), s->srgb8.as<unsigned char>(), npix, 0);
    (*launches)++;
    VRJ_CUDA(cudaMemcpyAsync(dst, s->srgb8.p, npix * 3, kind, s->stream));
    return VRJ_OK;
}

// one of a call's arrays: the caller's (NULL: not wanted), the block's, doubles per pixel
struct Arr {
    double *user;
    DeviceBuffer *dev;
    size_t per;
};

// What every render call (vrj_render_tile, render_passes, vrj_render_counts) does around its kernels.  prepare(): a block from
// the pool for batches of up to `widest` samples of the tile (prepare_paths: of up to `widest` units of `unit` paths);
// load_state(): the call's arrays and its state in the block; start(): the call's counters, lights and constants, the render
// turn and ev0; finish(): ev1, the counters, the copies of the outputs and the sRGB preview, the waits, VrjStats.  `turn` is
// declared after `block`: an early return gives the turn back before the block.
struct RenderCall {
    VrjScene *scene;
    const VrjRenderParams *p;
    uint64_t npix;
    BlockLease block;
    RenderTurn turn;
    Scratch *s = nullptr;
    uint32_t filter = 0, batch = 0;
    RenderConst rc{};
    uint64_t launches = 0;
    VrjAccumOut *out = nullptr;
    Arr arrs[6] = {}; // out's colour, colour_sum, colour_bias, weight, weight_bias, and y_sq_sum for the calls that keep it
    int n_arrs = 0;
    cudaMemcpyKind in_kind = cudaMemcpyHostToDevice, out_kind = cudaMemcpyDeviceToHost;
    bool pieces_copied = false; // the arrays went out with the last resolve's pieces (vrj_render_tile): wait for those copies
    float ms = 0.f;             // device time, ev0 .. ev1
    std::chrono::steady_clock::time_point t_start, t_enqueued, t_done; // turn taken, last copy enqueued, copies arrived
    RenderCall(VrjScene *sc, const VrjRenderParams *params, uint64_t n) : scene(sc), p(params), npix(n), block{sc}, turn(sc->device) {}

    VrjStatus prepare(uint32_t widest, const ActiveCall &active, size_t n_light_samples) { return prepare_paths(npix, widest, active, n_light_samples); }
    VrjStatus prepare_paths(uint64_t unit, uint32_t widest, const ActiveCall &active, size_t n_light_samples) {
        batch = (uint32_t)std::max<uint64_t>(1, std::min<uint64_t>(widest, call_path_budget(scene, active) / unit));
        if (unit * (uint64_t)batch > 0xfffffff0ull) return fail(VRJ_ERR_UNSUPPORTED, "tile too large");
        s = block.s = acquire_scratch(scene, unit * batch);
        filter = effective_filter(scene, p);
        return ensure_call_scratch(s, p, call_wants_records(scene, p, filter), npix, unit, &batch, n_light_samples);
    }
    // The call's arrays: out's, and with `ysq` (render_passes, vrj_render_counts) y_sq_sum.  The state -- every array but
    // colour -- comes into the block from the caller's arrays when `load` (a NULL array starts at zero), else it is zero.
    VrjStatus load_state(VrjAccumOut *o, bool load, bool ysq = false, double *y_sq_sum = nullptr) {
        out = o;
        in_kind = out->memory == VRJ_MEM_DEVICE ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice;
        out_kind = out->memory == VRJ_MEM_DEVICE ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost;
        const Arr a[6] = {{out->colour, &s->acc_colour, 3}, {out->colour_sum, &s->acc_sum, 3}, {out->colour_bias, &s->acc_bias, 3},
                          {out->weight, &s->acc_weight, 1}, {out->weight_bias, &s->acc_wbias, 1}, {y_sq_sum, &s->ysq, 1}};
        n_arrs = ysq ? 6 : 5;
        std::copy(a, a + n_arrs, arrs);
        for (int i = 1; i < n_arrs; i++) {
            if (load && arrs[i].user) VRJ_CUDA(cudaMemcpyAsync(arrs[i].dev->p, arrs[i].user, npix * arrs[i].per * sizeof(double), in_kind, s->stream));
            else VRJ_CUDA(cudaMemsetAsync(arrs[i].dev->p, 0, npix * arrs[i].per * sizeof(double), s->stream));
        }
        return VRJ_OK;
    }
    VrjStatus start(const VrjTile *tile, uint64_t height, uint64_t width) {
        VRJ_CUDA(cudaMemsetAsync(s->stats.p, 0, ST_COUNT * sizeof(unsigned long long), s->stream));
        const VrjStatus st = stage_lights(s, p);
        if (st != VRJ_OK) return st;
        rc = make_render_const(tile, height, width, p);
        rc.lights = s->lights.as<LightDev>();
        rc.light_samples = s->light_samples.as<double>();
        rc.div_tile_w = FastDiv::make(rc.tile_w);
        s->n_marks = 0;
        turn.acquire();
        t_start = std::chrono::steady_clock::now();
        VRJ_CUDA(cudaEventRecord(s->ev0, s->stream));
        return VRJ_OK;
    }
    VrjStatus finish() {
        VRJ_CUDA(cudaEventRecord(s->ev1, s->stream)); // before the counters' copy: that one queues up behind the pieces' copies on the copy engine
        VRJ_CUDA(cudaMemcpyAsync(s->pinned->stats, s->stats.p, ST_COUNT * sizeof(unsigned long long), cudaMemcpyDeviceToHost, s->stream));
        if (pieces_copied) {
            VRJ_CUDA(cudaStreamWaitEvent(s->stream, s->copy_done, 0)); // ev_done below then stands behind the pieces' copies too
        } else {
            for (int i = 0; i < n_arrs; i++)
                if (arrs[i].user) VRJ_CUDA(cudaMemcpyAsync(arrs[i].user, arrs[i].dev->p, npix * arrs[i].per * sizeof(double), out_kind, s->stream));
        }
        if (out->srgb8) {
            const VrjStatus st = copy_srgb8(s, npix, out->srgb8, out_kind, &launches);
            if (st != VRJ_OK) return st;
        }
        t_enqueued = std::chrono::steady_clock::now();
        VRJ_CUDA(cudaEventRecord(s->ev_done, s->stream));
        VRJ_CUDA(wait_event(s->ev1, scene->device)); // the last kernel is done: the next caller may render while this one's copies run
        turn.release();
        VRJ_CUDA(wait_event(s->ev_done, scene->device));
        t_done = std::chrono::steady_clock::now();
        VRJ_CUDA(cudaEventElapsedTime(&ms, s->ev0, s->ev1));
        if (out->stats) fill_call_stats(out->stats, s, s->pinned->stats, launches, ms);
        return VRJ_OK;
    }
};

// y_sq_sum, two pixel lists, the first samples of one and the selects' counters for npix pixels (render_passes); with
// slots > 0 (vrj_render_counts) also the scan of the count map (npix + 1 values and the scan's scratch), its counters, and
// a pixel and a first sample for each of `slots` paths in flight: 8 bytes per path
VrjStatus ensure_pass_buffers(Scratch *s, uint64_t npix, uint64_t slots = 0) {
    if (s->pass_npix >= npix && s->pass_slots >= slots) return VRJ_OK;
    npix = std::max<uint64_t>(npix, s->pass_npix), slots = std::max<uint64_t>(slots, s->pass_slots);
    s->pass_npix = 0, s->pass_slots = 0;
    std::vector<std::pair<DeviceBuffer *, size_t>> want = {{&s->ysq, npix * 8}, {&s->pass_list[0], npix * 4}, {&s->pass_list[1], npix * 4},
                                                           {&s->pass_base, npix * 4}, {&s->pass_counters, sizeof(ProgressiveCounters)}};
    if (slots)
        want.insert(want.end(), {{&s->count_offset, (npix + npix / 2048 + 4) * 4}, {&s->count_counters, sizeof(CountsCounters)},
                                 {&s->slot_pixel, slots * 4}, {&s->slot_base, slots * 4}});
    const VrjStatus st = alloc_group(s->pass_slab, want, "adaptive sampling buffers");
    if (st != VRJ_OK) return st;
    s->pass_npix = npix, s->pass_slots = slots;
    return VRJ_OK;
}

// the fields VrjAdaptiveParams and VrjProgressiveParams share, and params->spp, which must be 0
template <typename P>
VrjStatus check_rule(const P *ap, PassRule *rule) {
    if (!ap) return fail(VRJ_ERR_INVALID_ARGUMENT, "NULL argument");
    if (ap->min_samples < 2) return fail(VRJ_ERR_INVALID_ARGUMENT, "min_samples must be >= 2 (the variance needs two samples)");
    if (ap->max_samples < ap->min_samples) return fail(VRJ_ERR_INVALID_ARGUMENT, "max_samples must be >= min_samples");
    if (ap->pass_samples < 1) return fail(VRJ_ERR_INVALID_ARGUMENT, "pass_samples must be >= 1");
    if (!(ap->rel_error > 0.0) || !std::isfinite(ap->rel_error)) return fail(VRJ_ERR_INVALID_ARGUMENT, "rel_error must be > 0 and finite");
    if (!(ap->abs_floor >= 0.0) || !std::isfinite(ap->abs_floor)) return fail(VRJ_ERR_INVALID_ARGUMENT, "abs_floor must be >= 0 and finite");
    *rule = PassRule{ap->min_samples, ap->max_samples, ap->pass_samples, 0u, ap->rel_error, ap->abs_floor};
    return VRJ_OK;
}
template <typename P>
VrjStatus check_pass_rule(const VrjRenderParams *p, const P *ap, const char *call, const char *type, PassRule *rule) {
    if (!ap) return fail(VRJ_ERR_INVALID_ARGUMENT, "NULL argument");
    if (p->spp != 0) return fail(VRJ_ERR_INVALID_ARGUMENT, std::string("params->spp must be 0: ") + call + " takes its sample counts from " + type);
    return check_rule(ap, rule);
}

struct PassResult {
    uint64_t passes = 0, samples = 0;
    ProgressiveCounters counts{}; // converged and at_max over the call, active at return
};

// The passes of vrj_render_adaptive and vrj_render_progressive (the header states the schedule) on a tile of npix >= 1
// pixels.  The state starts at zero, or (out->accumulate) comes from out's four state arrays and y_sq_sum; every output array
// may be NULL.  A pass renders its pixels' samples in batches split to the path budget like vrj_render_tile's, and
// k_resolve_adaptive applies them to the tile's accumulators and y_sq_sum.
//  - A fresh state's pass 0 is known on the host (every pixel takes samples 0 .. min_samples-1): it runs over the tile on
//    the tile's kernels, with no select before it.  A continued state is first judged over the whole tile, which is also
//    where weights that are no sample counts are found.
//  - Before every further pass k_progressive_select judges the pixels the previous pass rendered (an inactive pixel stays
//    inactive) and the host reads back its counters.  When every active pixel takes the same count -- always, for a state
//    this schedule produced with unchanged parameters -- an exclusive scan (vrj_build::exclusive_scan_u32) of its flags and
//    k_progressive_compact list the active pixels in tile order with their first new sample, and the LIST kernels render
//    them.  Otherwise k_progressive_group lists the pixels of each count, largest first, in a segment of the list of its own,
//    and each segment is rendered as a sub-pass once all are listed.
//  - colour: a fresh state's pixels were all resolved, which writes it; a continued state's comes from k_finalize.
VrjStatus render_passes(VrjScene *scene, const VrjTile *tile, uint64_t height, uint64_t width, const VrjRenderParams *p, const PassRule &rule,
                        uint32_t max_passes, size_t n_light_samples, VrjAccumOut *out, double *y_sq_sum, PassResult *res) {
    const uint64_t npix = (tile->end_column - tile->start_column) * (tile->end_row - tile->start_row);
    const bool fresh = !out->accumulate;
    ActiveCall active(g_active_calls[(unsigned)scene->device % 64]);
    RenderCall call(scene, p, npix);
    // the widest pass is the whole tile at max(min, pass) samples (a fresh state's first pass, or a state that every pixel
    // has to continue); the block is sized for it
    VrjStatus st = call.prepare(std::min(rule.max_samples, std::max(rule.min_samples, rule.pass_samples)), active, n_light_samples);
    if (st != VRJ_OK) return st;
    Scratch *s = call.s;
    st = ensure_pass_buffers(s, npix);
    if (st != VRJ_OK) return st;
    st = call.load_state(out, !fresh, true, y_sq_sum);
    if (st != VRJ_OK) return st;
    ProgressiveCounters *ctr = s->pass_counters.as<ProgressiveCounters>(), *hctr = &s->pinned->pass;
    VRJ_CUDA(cudaMemsetAsync(ctr, 0, sizeof(ProgressiveCounters), s->stream));
    st = call.start(tile, height, width);
    if (st != VRJ_OK) return st;

    RenderConst &rc = call.rc;
    const size_t capacity = npix * call.batch; // paths per batch
    const AccumDev acc = s->accum();
    const double *sum = acc.sum, *weight = acc.weight;
    double *ysq = s->ysq.as<double>();
    // the flags and the scan's tile totals live in the photon buffer, which is free between a pass's resolve and the next
    // batch: (n + 1) + (n / 2048 + 2) uint32 fit the 16 bytes per path of a block that holds at least one path per pixel
    uint32_t *flags = s->photons.as<uint32_t>(), *base = s->pass_base.as<uint32_t>();
    // samples base[i] .. base[i] + c - 1 of the m pixels of `list` (the tile's samples 0 .. c - 1 when `list` is NULL)
    auto render = [&](const uint32_t *list, const uint32_t *first, uint32_t m, uint32_t c) -> VrjStatus {
        const uint32_t b = (uint32_t)std::max<size_t>(1, std::min<size_t>(c, capacity / m));
        rc.npix = m, rc.pixel_list = list, rc.pixel_base = first;
        for (uint32_t done = 0; done < c; done += b) {
            rc.batch_samples = std::min(b, c - done);
            rc.div_batch = FastDiv::make(rc.batch_samples);
            rc.first_sample = p->sample_offset + (uint64_t)done * rc.sample_stride;
            VrjStatus bst = dispatch_batch(scene, s, rc, p, call.filter, &call.launches);
            if (bst == VRJ_OK)
                bst = resolve_batch(s, p, [&](auto r) {
                    k_resolve_adaptive<decltype(r)><<<(rc.npix + 255) / 256, 256, 0, s->stream>>>(acc, ysq, rc.pixel_list, s->photons.as<double2>(), rc.npix, rc.batch_samples);
                    call.launches++;
                    return VRJ_OK;
                });
            if (bst != VRJ_OK) return bst;
        }
        res->samples += (uint64_t)m * c;
        return VRJ_OK;
    };
    auto compact = [&](const uint32_t *list, uint32_t n, uint32_t *to, uint32_t *first) -> VrjStatus {
        const VrjStatus sst = vrj_build::exclusive_scan_u32(flags, n + 1, flags + n + 1, s->stream);
        if (sst != VRJ_OK) return sst;
        k_progressive_compact<<<(n + 255) / 256, 256, 0, s->stream>>>(list, weight, flags, n, to, first);
        call.launches += 4;
        VRJ_CUDA(cudaGetLastError());
        return VRJ_OK;
    };
    if (fresh) {
        st = render(nullptr, nullptr, (uint32_t)npix, rule.min_samples);
        if (st != VRJ_OK) return st;
        res->passes = 1;
    }
    const uint32_t *list = nullptr; // the pixels the last select judges (NULL: the tile)
    uint32_t n = (uint32_t)npix, next = 0, held = rule.min_samples; // held: what every pixel of a fresh state's list holds
    for (;;) {
        VRJ_CUDA(cudaMemsetAsync(ctr, 0, offsetof(ProgressiveCounters, converged), s->stream)); // active, cmax, cmin_not
        k_progressive_select<<<(n + 1 + 255) / 256, 256, 0, s->stream>>>(sum, weight, ysq, list, n, rule, flags, ctr);
        call.launches++;
        VRJ_CUDA(cudaGetLastError());
        VRJ_CUDA(cudaMemcpyAsync(hctr, ctr, sizeof(ProgressiveCounters), cudaMemcpyDeviceToHost, s->stream));
        // the last select only counts, and nothing waits for it (its counters arrive with the outputs): the pass limit is
        // reached, or a fresh state's pixels all hold max_samples (no weight can be invalid in either case)
        if ((max_passes && res->passes == max_passes) || (fresh && held >= rule.max_samples)) break;
        VRJ_CUDA(cudaStreamSynchronize(s->stream));
        if (hctr->bad) return fail(VRJ_ERR_INVALID_ARGUMENT, "a weight of the state is not a sample count (negative, fractional, not finite or >= 2^32)");
        if (hctr->active == 0) break;
        const uint32_t m = (uint32_t)hctr->active, cmax = hctr->cmax;
        held += cmax;
        uint32_t *to = s->pass_list[next].as<uint32_t>();
        if (cmax == ~hctr->cmin_not) {
            st = compact(list, n, to, base);
            if (st == VRJ_OK) st = render(to, base, m, cmax);
            if (st != VRJ_OK) return st;
        } else {
            // every segment is listed before any is rendered: rendering changes the state the counts are computed from
            std::vector<std::pair<uint32_t, uint32_t>> segments; // (count, length)
            uint32_t listed = 0;
            for (uint32_t c = cmax; c != 0;) {
                VRJ_CUDA(cudaMemsetAsync(&ctr->next, 0, sizeof(uint32_t), s->stream));
                k_progressive_group<<<(n + 1 + 255) / 256, 256, 0, s->stream>>>(sum, weight, ysq, list, n, rule, c, flags, ctr);
                call.launches++;
                st = compact(list, n, to + listed, base + listed);
                if (st != VRJ_OK) return st;
                VRJ_CUDA(cudaMemcpyAsync(&s->pinned->listed, flags + n, sizeof(uint32_t), cudaMemcpyDeviceToHost, s->stream));
                VRJ_CUDA(cudaMemcpyAsync(&hctr->next, &ctr->next, sizeof(uint32_t), cudaMemcpyDeviceToHost, s->stream));
                VRJ_CUDA(cudaStreamSynchronize(s->stream));
                if (s->pinned->listed) segments.push_back({c, s->pinned->listed}), listed += s->pinned->listed;
                c = hctr->next;
            }
            listed = 0;
            for (const auto &seg : segments) {
                st = render(to + listed, base + listed, seg.second, seg.first);
                if (st != VRJ_OK) return st;
                listed += seg.second;
            }
        }
        list = to, n = m, next ^= 1u;
        res->passes++;
    }
    if (!fresh && (out->colour || out->srgb8)) {
        k_finalize<<<(unsigned)((npix + 255) / 256), 256, 0, s->stream>>>(sum, weight, acc.colour, (uint32_t)npix);
        call.launches++;
        VRJ_CUDA(cudaGetLastError());
    }
    st = call.finish();
    if (st != VRJ_OK) return st;
    res->counts = *hctr;
    return VRJ_OK;
}

// a stream and two events of a call's own (vrj_render_aux, vrj_denoise, vrj_plan_counts, the sums of a device count map:
// short calls that take no render turn and no scratch block).  Declared after the call's DeviceBuffers: nothing may still
// use them when they return to the pool.
struct CallStream {
    cudaStream_t s = nullptr;
    cudaEvent_t e0 = nullptr, e1 = nullptr;
    cudaError_t create() {
        cudaError_t e = cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking);
        if (e == cudaSuccess) e = cudaEventCreate(&e0);
        if (e == cudaSuccess) e = cudaEventCreate(&e1);
        return e;
    }
    ~CallStream() {
        if (s) cudaStreamSynchronize(s), cudaStreamDestroy(s);
        if (e0) cudaEventDestroy(e0);
        if (e1) cudaEventDestroy(e1);
    }
};

// vrj_render_counts (the header states it) on a tile of npix >= 1 pixels.  The count map goes into the block, and
// k_counts_check sums it exactly in 64 bits and checks the state before anything is rendered: a refused call has written
// nothing the caller sees.  The exclusive scan of the map (vrj_build::exclusive_scan_u32) gives each pixel its run of slots;
// the call's samples are then rendered as wavefronts of up to the path budget's slots, each one sample (batch_samples = 1)
// of the LIST kernels: k_counts_expand lists the (pixel, sample) of every slot of the batch and k_resolve_counts applies the
// batch to the accumulators and y_sq_sum.  Batches are resolved in order, so a pixel's run that straddles two of them is
// still applied in sample order.  colour comes from k_finalize.
VrjStatus render_counts(VrjScene *scene, const VrjTile *tile, uint64_t height, uint64_t width, const VrjRenderParams *p, const uint32_t *counts,
                        size_t n_light_samples, VrjAccumOut *out, double *y_sq_sum, VrjCountsStats *cstats) {
    const uint64_t npix = (tile->end_column - tile->start_column) * (tile->end_row - tile->start_row);
    const uint32_t n32 = (uint32_t)npix;
    // the map's total sizes the block: a batch is at most the path budget's slots, and no more than the call renders
    uint64_t total = 0;
    if (out->memory == VRJ_MEM_HOST) {
        for (uint64_t i = 0; i < npix; i++) total += counts[i];
    } else {
        DeviceBuffer sums;
        VRJ_CUDA(sums.alloc(sizeof(CountsCounters)));
        CallStream cs;
        VRJ_CUDA(cs.create());
        CountsCounters h{};
        VRJ_CUDA(cudaMemsetAsync(sums.p, 0, sizeof(CountsCounters), cs.s));
        k_counts_check<<<(n32 + 255) / 256, 256, 0, cs.s>>>(nullptr, counts, n32, nullptr, sums.as<CountsCounters>());
        VRJ_CUDA(cudaGetLastError());
        VRJ_CUDA(cudaMemcpyAsync(&h, sums.p, sizeof(CountsCounters), cudaMemcpyDeviceToHost, cs.s));
        VRJ_CUDA(cudaStreamSynchronize(cs.s));
        total = h.samples;
    }
    if (total > 0xffffffffull) return fail(VRJ_ERR_UNSUPPORTED, "more than 2^32 - 1 samples in one call");
    ActiveCall active(g_active_calls[(unsigned)scene->device % 64]);
    RenderCall call(scene, p, npix);
    VrjStatus st = call.prepare_paths(1, (uint32_t)std::min<uint64_t>(std::max<uint64_t>(total, 1), 0xffffffffull), active, n_light_samples);
    if (st != VRJ_OK) return st;
    Scratch *s = call.s;
    st = ensure_pass_buffers(s, npix, call.batch);
    if (st != VRJ_OK) return st;
    st = call.load_state(out, out->accumulate != 0, true, y_sq_sum);
    if (st != VRJ_OK) return st;
    uint32_t *offset = s->count_offset.as<uint32_t>(), *held = s->pass_base.as<uint32_t>();
    CountsCounters *ctr = s->count_counters.as<CountsCounters>(), *hctr = &s->pinned->counts;
    VRJ_CUDA(cudaMemcpyAsync(offset, counts, npix * sizeof(uint32_t), call.in_kind, s->stream));
    VRJ_CUDA(cudaMemsetAsync(offset + npix, 0, sizeof(uint32_t), s->stream));
    VRJ_CUDA(cudaMemsetAsync(ctr, 0, sizeof(CountsCounters), s->stream));
    k_counts_check<<<(n32 + 255) / 256, 256, 0, s->stream>>>(s->acc_weight.as<double>(), offset, n32, held, ctr);
    VRJ_CUDA(cudaGetLastError());
    VRJ_CUDA(cudaMemcpyAsync(hctr, ctr, sizeof(CountsCounters), cudaMemcpyDeviceToHost, s->stream));
    VRJ_CUDA(cudaStreamSynchronize(s->stream));
    if (hctr->bad) return fail(VRJ_ERR_INVALID_ARGUMENT, "a weight of the state is not a sample count (negative, fractional, not finite or >= 2^32)");
    if (hctr->over) return fail(VRJ_ERR_INVALID_ARGUMENT, "a pixel would hold 2^32 samples or more (weight + count)");
    total = hctr->samples;
    if (cstats) cstats->samples = total, cstats->pixels = hctr->pixels;
    call.launches = 1; // k_counts_check
    st = call.start(tile, height, width);
    if (st != VRJ_OK) return st;

    RenderConst &rc = call.rc;
    double *ysq = s->ysq.as<double>();
    if (total) {
        st = vrj_build::exclusive_scan_u32(offset, n32 + 1, offset + npix + 1, s->stream);
        if (st != VRJ_OK) return st;
        call.launches += 3;
        uint32_t *slot_pixel = s->slot_pixel.as<uint32_t>(), *slot_base = s->slot_base.as<uint32_t>();
        rc.batch_samples = 1, rc.div_batch = FastDiv::make(1);
        rc.first_sample = p->sample_offset;
        rc.pixel_list = slot_pixel, rc.pixel_base = slot_base;
        uint64_t batches = 0;
        for (uint64_t b0 = 0; b0 < total; b0 += call.batch, batches++) {
            const uint32_t b1 = (uint32_t)std::min<uint64_t>(total, b0 + call.batch), m = b1 - (uint32_t)b0;
            k_counts_expand<<<(m + 255) / 256, 256, 0, s->stream>>>(offset, held, n32, (uint32_t)b0, b1, slot_pixel, slot_base);
            call.launches++;
            VRJ_CUDA(cudaGetLastError());
            rc.npix = m;
            st = dispatch_batch(scene, s, rc, p, call.filter, &call.launches);
            if (st == VRJ_OK)
                st = resolve_batch(s, p, [&](auto r) {
                    k_resolve_counts<decltype(r)><<<(n32 + 255) / 256, 256, 0, s->stream>>>(s->accum(), ysq, offset, s->photons.as<double2>(), n32, (uint32_t)b0, b1);
                    call.launches++;
                    return VRJ_OK;
                });
            if (st != VRJ_OK) return st;
        }
        if (cstats) cstats->batches = batches;
    }
    if (out->colour || out->srgb8) {
        k_finalize<<<(n32 + 255) / 256, 256, 0, s->stream>>>(s->acc_sum.as<double>(), s->acc_weight.as<double>(), s->acc_colour.as<double>(), n32);
        call.launches++;
        VRJ_CUDA(cudaGetLastError());
    }
    return call.finish();
}

// ---------------------------------------------------------------------------------------------- coalesced calls
// main.rs:197-209 calls partial_render_scene once per one-sample pass from a pool of workers.  Each such call is a small
// wavefront (2 M paths at 1080p) whose ~28 launches do not fill 148 SMs: 1.7 ms of device time against 0.52 ms per sample
// when 64 samples share a wavefront.  Calls that arrive while the device is busy and differ only in their sample indices and
// output buffers are therefore rendered TOGETHER: one of the waiting callers (the leader) takes its turn at the render gate,
// collects every compatible caller that has queued up behind it, runs one wavefront over all their samples (the batch's slots
// carry their sample indices in a table, RenderConst::sample_table), resolves each call's samples into that call's own
// fresh buffer (k_resolve_multi) and copies every buffer back.  A sample is a pure function of (seed, pixel, sample index)
// and each call's samples are applied to its buffer in sample order, so every caller receives bit for bit what it would have
// received alone (tests/test_gpu_parity.py::test_coalesced_calls_bit_identical).  The ray counters of a shared wavefront are
// split evenly over its calls (the remainder goes to the first; sums stay exact) and VrjStats.coalesced_calls says how many
// shared it.  VRJ_COALESCE=0 turns this off (experiments).
struct CoalesceRequest {
    const VrjScene *scene;
    VrjTile tile;
    uint64_t height, width;
    VrjRenderParams params;
    VrjAccumOut *out;
    VrjStatus status = VRJ_OK;
    std::string error;
    bool done = false;     // a leader failed before launching anything: `status` / `error` say why
    bool launched = false; // rendered by a leader: stats are filled, the buffers are on their way, `wait_ev` fires on arrival
    cudaEvent_t wait_ev = nullptr;
    uint32_t wanted() const {
        return (out->colour ? 1u : 0u) | (out->colour_sum ? 2u : 0u) | (out->colour_bias ? 4u : 0u) | (out->weight ? 8u : 0u) | (out->weight_bias ? 16u : 0u);
    }
    bool compatible(const CoalesceRequest &o) const {
        return scene == o.scene && tile.start_column == o.tile.start_column && tile.end_column == o.tile.end_column &&
               tile.start_row == o.tile.start_row && tile.end_row == o.tile.end_row && height == o.height && width == o.width &&
               params.max_depth == o.params.max_depth && params.seed == o.params.seed && params.bvh_filter == o.params.bvh_filter &&
               params.precision == o.params.precision && params.bias == o.params.bias &&
               (params.sample_stride ? params.sample_stride : 1u) == (o.params.sample_stride ? o.params.sample_stride : 1u) && wanted() == o.wanted();
    }
};
struct Coalescer {
    std::mutex m;
    std::condition_variable cv;
    std::vector<CoalesceRequest *> waiting;
    bool collecting = false; // a leader is waiting for its turn at the gate; arrivals pile up behind it
};
Coalescer g_coalescer[64];
constexpr uint64_t kCoalesceMaxPaths = uint64_t(1) << 25; // 32 Mi paths = 11 GB of queue state per shared wavefront

bool coalescing_enabled() {
    static const bool on = [] {
        const char *e = std::getenv("VRJ_COALESCE");
        return !e || std::atoi(e) != 0;
    }();
    return on;
}
static_assert(sizeof(PinnedBlock::sample_table) == 4 * MULTI_MAX_CALLS * sizeof(uint64_t),
              "the sample table of a coalesced wavefront holds MULTI_MAX_CALLS calls of up to 4 samples (coalescable)");
bool coalescable(const VrjRenderParams *p, const VrjAccumOut *out, uint64_t npix) {
    return coalescing_enabled() && out->memory == VRJ_MEM_HOST && !out->accumulate && !out->photons && !out->srgb8 && out->colour &&
           p->integrator == VRJ_INTEGRATOR_SIMPLE_RANDOM && p->n_lights == 0 && !p->ambient_light && !p->count_traversal &&
           p->spp >= 1 && p->spp <= 4 && npix * p->spp * 2 <= kCoalesceMaxPaths;
}

// one wavefront for `n` compatible requests; fills their buffers and stats; the status applies to all of them
VrjStatus render_group(Coalescer &co, CoalesceRequest *const *reqs, uint32_t n, RenderTurn &turn, bool *published) {
    static const bool timing = std::getenv("VRJ_TIMING") != nullptr;
    const auto t1 = std::chrono::steady_clock::now();
    const CoalesceRequest &r0 = *reqs[0];
    VrjScene *scene = const_cast<VrjScene *>(r0.scene);
    const VrjRenderParams *p = &r0.params;
    RenderConst rc = make_render_const(&r0.tile, r0.height, r0.width, p);
    const uint64_t npix = rc.npix;
    uint32_t total = 0;
    MultiCalls mc{};
    mc.n = n, mc.full = (r0.wanted() & ~1u) ? 1u : 0u;
    std::vector<uint64_t> table;
    for (uint32_t c = 0; c < n; c++) {
        mc.first[c] = total, mc.count[c] = reqs[c]->params.spp;
        for (uint32_t i = 0; i < reqs[c]->params.spp; i++) table.push_back(reqs[c]->params.sample_offset + (uint64_t)i * rc.sample_stride);
        total += reqs[c]->params.spp;
    }
    VRJ_NVTX_RANGE(call_range, "vrj_render_tile (coalesced)");
    // group sizes vary from wavefront to wavefront: blocks are sized in steps of eight 1-sample calls so that a block taken
    // from the pool almost never has to grow (growing re-allocates every queue: tens of milliseconds)
    const size_t capacity = npix * (size_t)((total + 7u) / 8u * 8u);
    const BlockLease lease{scene, acquire_scratch(scene, capacity)};
    Scratch *s = lease.s;
    const uint32_t filter = effective_filter(scene, p);
    const bool records = call_wants_records(scene, p, filter);
    VrjStatus st = ensure_scratch(s, capacity, records ? capacity : 0, 0, p->max_depth + 3, 0, 0);
    if (st == VRJ_ERR_OUT_OF_MEMORY) { // fall back to exactly what this wavefront needs
        vrj_pool_trim();
        st = ensure_scratch(s, npix * total, records ? npix * total : 0, 0, p->max_depth + 3, 0, 0);
    }
    if (st != VRJ_OK) return st;
    const auto t1b = std::chrono::steady_clock::now();
    const size_t per_call = npix * (mc.full ? 11 : 3) * sizeof(double);
    if (s->multi_out.bytes < per_call * n || !s->multi_out.p) {
        // sized once for the largest group this tile size can form (1-sample calls up to the path limit)
        const size_t max_calls = std::max<size_t>(n, std::min<size_t>(MULTI_MAX_CALLS, kCoalesceMaxPaths / std::max<uint64_t>(npix, 1)));
        s->multi_out.release();
        VRJ_CUDA(s->multi_out.alloc(per_call * max_calls));
    }
    if (!s->sample_table.p) VRJ_CUDA(s->sample_table.alloc(sizeof(PinnedBlock::sample_table)));
    double *base = s->multi_out.as<double>();
    mc.out.colour = base;
    if (mc.full) {
        mc.out.sum = base + 3 * npix * n, mc.out.bias = base + 6 * npix * n;
        mc.out.weight = base + 9 * npix * n, mc.out.weight_bias = base + 10 * npix * n;
    }
    std::memcpy(s->pinned->sample_table, table.data(), table.size() * sizeof(uint64_t));
    VRJ_CUDA(cudaMemcpyAsync(s->sample_table.p, s->pinned->sample_table, table.size() * sizeof(uint64_t), cudaMemcpyHostToDevice, s->stream));
    VRJ_CUDA(cudaMemsetAsync(s->stats.p, 0, ST_COUNT * sizeof(unsigned long long), s->stream));
    rc.sample_table = s->sample_table.as<uint64_t>();
    rc.lights = s->lights.as<LightDev>(), rc.light_samples = s->light_samples.as<double>();
    rc.batch_samples = total;
    rc.div_batch = FastDiv::make(total), rc.div_tile_w = FastDiv::make(rc.tile_w);
    rc.first_sample = 0;
    uint64_t launches = 0;
    s->n_marks = 0;
    VRJ_CUDA(cudaEventRecord(s->ev0, s->stream));
    st = dispatch_batch(scene, s, rc, p, filter, &launches);
    if (st == VRJ_OK)
        st = resolve_batch(s, p, [&](auto r) {
            k_resolve_multi<decltype(r)><<<(rc.npix * mc.n + 255) / 256, 256, 0, s->stream>>>(mc, s->photons.as<double2>(), rc.npix, rc.batch_samples);
            launches++;
            return VRJ_OK;
        });
    if (st != VRJ_OK) return st;
    unsigned long long *hstats = s->pinned->stats;
    VRJ_CUDA(cudaMemcpyAsync(hstats, s->stats.p, ST_COUNT * sizeof(unsigned long long), cudaMemcpyDeviceToHost, s->stream));
    VRJ_CUDA(cudaEventRecord(s->ev1, s->stream));
    // every call's arrays cross PCIe behind an event of their own, the leader's (call 0) last: a caller returns as soon as ITS
    // buffer has arrived, so the host's merge of the first buffer overlaps the copies of the others
    const double *dev_arr[5] = {mc.out.colour, mc.out.sum, mc.out.bias, mc.out.weight, mc.out.weight_bias};
    const size_t per[5] = {3, 3, 3, 1, 1};
    for (uint32_t k = 0; k < n; k++) {
        const uint32_t c = (k + 1) % n;
        double *user[5] = {reqs[c]->out->colour, reqs[c]->out->colour_sum, reqs[c]->out->colour_bias, reqs[c]->out->weight, reqs[c]->out->weight_bias};
        for (int i = 0; i < 5; i++)
            if (user[i]) VRJ_CUDA(cudaMemcpyAsync(user[i], dev_arr[i] + (size_t)c * npix * per[i], npix * per[i] * sizeof(double), cudaMemcpyDeviceToHost, s->stream));
        VRJ_CUDA(cudaEventRecord(s->call_ev[c], s->stream));
    }
    const auto t2 = std::chrono::steady_clock::now();
    VRJ_CUDA(wait_event(s->ev1, scene->device));
    turn.release(); // the next wavefront may start while this one's buffers cross PCIe
    float ms = 0.f;
    VRJ_CUDA(cudaEventElapsedTime(&ms, s->ev0, s->ev1));
    for (uint32_t c = 0; c < n; c++) {
        VrjStats *o = reqs[c]->out->stats;
        if (!o) continue;
        unsigned long long share[ST_COUNT];
        for (int k = 0; k < ST_COUNT; k++) share[k] = hstats[k] / n + (c == 0 ? hstats[k] % n : 0);
        std::memset(o, 0, sizeof *o);
        fill_call_stats(o, s, share, launches, ms / (float)n); // device time: the call's share of the wavefront
        o->primary_ms /= n, o->bounce_ms /= n, o->resolve_ms /= n, o->shade_ms /= n, o->tail_ms /= n;
        o->coalesced_calls = n;
    }
    // the other callers wait for their own buffers from here on
    {
        std::lock_guard<std::mutex> lock(co.m);
        for (uint32_t c = 1; c < n; c++) reqs[c]->wait_ev = s->call_ev[c], reqs[c]->launched = true;
        *published = true; // from here on those requests belong to their callers again
    }
    co.cv.notify_all();
    VRJ_CUDA(wait_event(s->call_ev[0], scene->device)); // recorded last: everything queued on the stream has finished
    if (timing) {
        auto msd = [](std::chrono::steady_clock::time_point a, std::chrono::steady_clock::time_point b) {
            return std::chrono::duration<double, std::milli>(b - a).count();
        };
        std::fprintf(stderr, "vrj_render_tile (coalesced): %u calls, %u samples: scratch %.3f ms, enqueue %.3f ms, wait %.3f ms (device %.3f ms, %llu launches), mallocs %llu / %llu\n", n, total,
                     msd(t1, t1b), msd(t1b, t2), msd(t2, std::chrono::steady_clock::now()), ms, (unsigned long long)launches,
                     (unsigned long long)g_n_device_mallocs.load(), (unsigned long long)g_n_host_mallocs.load());
    }
    return VRJ_OK;
}

// entry of a coalescable call: queue up, then either be served by a leader or become one
VrjStatus render_coalesced(const VrjScene *scene, const VrjTile *tile, uint64_t height, uint64_t width, const VrjRenderParams *p, VrjAccumOut *out) {
    CoalesceRequest req;
    req.scene = scene, req.tile = *tile, req.height = height, req.width = width, req.params = *p, req.out = out;
    Coalescer &co = g_coalescer[(unsigned)scene->device % 64];
    const uint64_t npix = (tile->end_column - tile->start_column) * (tile->end_row - tile->start_row);
    std::unique_lock<std::mutex> lock(co.m);
    co.waiting.push_back(&req);
    co.cv.wait(lock, [&] { return req.done || req.launched || (!co.collecting && !co.waiting.empty() && co.waiting.front() == &req); });
    if (req.launched) { // a leader rendered this call with its own and will not touch `req` again: wait for the buffers
        const cudaEvent_t ev = req.wait_ev;
        lock.unlock();
        const cudaError_t e = wait_event(ev, scene->device);
        if (e != cudaSuccess) return fail(VRJ_ERR_CUDA, std::string("coalesced call: ") + cudaGetErrorString(e));
        return VRJ_OK;
    }
    if (req.done) { // the leader failed before anything was launched
        vrj_set_error(req.error);
        return req.status;
    }
    co.collecting = true;
    lock.unlock();
    RenderTurn turn(scene->device);
    turn.acquire(); // callers that arrive while this one waits for the device join its wavefront
    lock.lock();
    std::vector<CoalesceRequest *> group{&req};
    uint64_t paths = npix * p->spp;
    for (size_t i = 0; i < co.waiting.size();) {
        CoalesceRequest *w = co.waiting[i];
        if (w == &req) {
            co.waiting.erase(co.waiting.begin() + i);
            continue;
        }
        if (group.size() < (size_t)MULTI_MAX_CALLS && w->compatible(req) && paths + npix * w->params.spp <= kCoalesceMaxPaths) {
            paths += npix * w->params.spp;
            group.push_back(w);
            co.waiting.erase(co.waiting.begin() + i);
            continue;
        }
        i++;
    }
    co.collecting = false;
    lock.unlock();
    co.cv.notify_all(); // the next caller in line may start collecting
    bool published = false; // true once the other callers have been told to wait for their buffers (they may return at any moment)
    const VrjStatus st = render_group(co, group.data(), (uint32_t)group.size(), turn, &published);
    turn.release();
    if (!published) {
        const std::string err = st != VRJ_OK ? std::string(vrj_last_error()) : std::string("coalesced call: not rendered");
        lock.lock();
        for (CoalesceRequest *g : group)
            if (g != &req) g->status = st != VRJ_OK ? st : VRJ_ERR_CUDA, g->error = err, g->done = true;
        lock.unlock();
        co.cv.notify_all();
    }
    return st;
}

} // namespace

extern "C" {

const char *vrj_last_error(void) { return g_error.c_str(); }
int32_t vrj_abi_version(void) { return VRJ_ABI_VERSION; }
int32_t vrj_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    return n;
}

VrjStatus vrj_scene_create(const VrjSceneDesc *d, int32_t device, VrjScene **out) {
    DeviceGuard device_guard;
    if (!out) return fail(VRJ_ERR_INVALID_ARGUMENT, "out is NULL");
    *out = nullptr;
    VRJ_NVTX_RANGE(create_range, "vrj_scene_create");
    auto t_start = std::chrono::steady_clock::now();
    VrjStatus st = validate(d);
    if (st != VRJ_OK) return st;
    auto t_valid = std::chrono::steady_clock::now();
    VRJ_CUDA(cudaSetDevice(device));
    VrjScene *sc = new VrjScene();
    sc->device = device;
    // one attribute, not cudaGetDeviceProperties: that call took 4-115 ms per scene on the B200 boxes (measured)
    int sm_count = 0;
    cudaError_t pe = cudaDeviceGetAttribute(&sm_count, cudaDevAttrMultiProcessorCount, device);
    if (pe != cudaSuccess) {
        delete sc;
        return fail(VRJ_ERR_CUDA, std::string("cudaDeviceGetAttribute: ") + cudaGetErrorString(pe));
    }
    sc->sm_count = sm_count;
    sc->n_spectra = d->n_spectra;

#define VRJ_TRY(expr)             \
    do {                          \
        VrjStatus s_ = (expr);    \
        if (s_ != VRJ_OK) {       \
            delete sc;            \
            return s_;            \
        }                         \
    } while (0)

    // ---- layout of the device arena: the small tables first (staged on the host, one copy), then the big sections,
    // which kernels write on the device from the caller's arrays (vrj_scene_prep.cuh) ----
    // A VrjBvh with n_nodes == 0 and n_triangles > 0 is built here, on the device (vrj_bvh_build.cu).
    struct BvhPlan {
        bool empty = false, build = false;
        uint64_t first_node = 0, n_nodes = 0, n_wide = 0, wide_base = 0;
    };
    std::vector<BvhPlan> plan(d->n_bvhs);
    uint64_t n_wide = 0, n_dev_nodes = d->n_nodes;
    for (uint32_t b = 0; b < d->n_bvhs; b++) {
        const VrjBvh &bv = d->bvhs[b];
        BvhPlan &pl = plan[b];
        if (bv.n_triangles == 0) {
            pl.empty = true; // an empty BVH never reports a hit
            continue;
        }
        if (bv.n_nodes == 0) {
            pl.build = true;
            pl.first_node = n_dev_nodes, pl.n_nodes = 2 * bv.n_triangles - 1;
            n_dev_nodes += pl.n_nodes;
            pl.n_wide = std::max<uint64_t>(1, bv.n_triangles - 1);
        } else {
            pl.first_node = bv.first_node, pl.n_nodes = bv.n_nodes;
            uint64_t internal = 0;
            for (uint64_t n = bv.first_node; n < bv.first_node + bv.n_nodes; n++) internal += d->node_child[2 * n] >= 0;
            pl.n_wide = std::max<uint64_t>(1, internal);
        }
        pl.wide_base = n_wide;
        n_wide += pl.n_wide;
    }
    if (n_dev_nodes > 0x7ffffff0ull) {
        delete sc;
        return fail(VRJ_ERR_UNSUPPORTED, "scene too large for 31-bit indices");
    }
    struct Section {
        size_t offset, bytes;
    };
    size_t cursor = 0;
    auto reserve_section = [&cursor](size_t bytes) {
        Section sct{cursor, bytes};
        cursor += (bytes + 255) & ~size_t(255);
        return sct;
    };
    const Section s_sph = reserve_section(d->n_spheres * sizeof(SphereDev)), s_pl = reserve_section(d->n_planes * sizeof(PlaneDev));
    const Section s_mat = reserve_section(d->n_materials * sizeof(MaterialDev)), s_spc = reserve_section(d->n_spectra * sizeof(SpectrumDev));
    const Section s_smp = reserve_section(d->n_spectrum_samples * sizeof(double));
    const Section s_grd = reserve_section(d->n_spectrum_samples * sizeof(double));
    const Section s_it = reserve_section(d->n_items * sizeof(ItemDev)), s_an = reserve_section(d->n_items * 4), s_bv = reserve_section(d->n_items * 4);
    const size_t small_bytes = std::max<size_t>(cursor, 256);
    const Section s_n32 = reserve_section(n_wide * 64), s_n64 = reserve_section(n_wide * 112);
    const Section s_n4 = reserve_section(n_wide * 128); // upper bound: at most every internal node becomes a 4-wide node
    const Section s_nq = reserve_section(n_wide * 32);
    const Section s_tp = reserve_section((size_t)d->n_triangles * 96), s_tn = reserve_section((size_t)d->n_triangles * 96);
    const Section s_tp32 = reserve_section((size_t)d->n_triangles * 48), s_tn32 = reserve_section((size_t)d->n_triangles * 48);
    const size_t arena_bytes = std::max<size_t>(cursor, 256);

    DeviceBuffer *arena = new DeviceBuffer();
    sc->owned.push_back(arena);
    {
        cudaError_t ae = arena->alloc(arena_bytes);
        if (ae != cudaSuccess) {
            delete sc;
            return fail(ae == cudaErrorMemoryAllocation ? VRJ_ERR_OUT_OF_MEMORY : VRJ_ERR_CUDA, std::string("scene arena: ") + cudaGetErrorString(ae));
        }
    }
    char *base = arena->as<char>();
#define VRJ_TRY_CUDA(expr)                                                                                                 \
    do {                                                                                                                   \
        cudaError_t e_ = (expr);                                                                                           \
        if (e_ != cudaSuccess) {                                                                                           \
            delete sc;                                                                                                     \
            return fail(e_ == cudaErrorMemoryAllocation ? VRJ_ERR_OUT_OF_MEMORY : VRJ_ERR_CUDA,                            \
                        std::string(#expr) + ": " + cudaGetErrorString(e_));                                               \
        }                                                                                                                  \
    } while (0)

    // ---- the caller's big arrays go to the device as they are (one temporary block, freed when this function returns) ----
    const size_t nt = (size_t)d->n_triangles, nn = (size_t)n_dev_nodes;
    size_t rcur = 0;
    auto reserve_raw = [&rcur](size_t bytes) {
        size_t o = rcur;
        rcur += (bytes + 255) & ~size_t(255);
        return o;
    };
    const size_t r_v[6] = {reserve_raw(nt * 32), reserve_raw(nt * 32), reserve_raw(nt * 32), reserve_raw(nt * 32), reserve_raw(nt * 32), reserve_raw(nt * 32)};
    const size_t r_mat = reserve_raw(nt * 4), r_pid = reserve_raw(nt * 4), r_perm = reserve_raw(nt * 4);
    const size_t r_min = reserve_raw(nn * 32), r_max = reserve_raw(nn * 32), r_child = reserve_raw(nn * 8);
    uint64_t largest_bvh_nodes = 0, largest_build = 0;
    bool any_build = false;
    for (uint32_t b = 0; b < d->n_bvhs; b++) {
        largest_bvh_nodes = std::max(largest_bvh_nodes, plan[b].n_nodes);
        if (plan[b].build) any_build = true, largest_build = std::max<uint64_t>(largest_build, d->bvhs[b].n_triangles);
    }
    const size_t r_flags = reserve_raw(largest_bvh_nodes * 4), r_scan = reserve_raw((largest_bvh_nodes / 2048 + 2) * 4);
    const size_t r_parent = reserve_raw(largest_bvh_nodes * 4), r_isquad = reserve_raw(largest_bvh_nodes * 4);
    const size_t r_bv = reserve_raw(largest_build * 72), r_bo = reserve_raw(largest_build * 4);
    DeviceBuffer raw;
    VRJ_TRY_CUDA(raw.alloc(std::max<size_t>(rcur, 256)));
    char *rb = raw.as<char>();
    auto t_alloc = std::chrono::steady_clock::now();
    StagingArea &area = g_staging_area[(unsigned)device % 64];
    std::lock_guard<std::mutex> staging_guard(area.mutex); // scene creation is synchronous; one at a time per device
    Stager stager(area);
    VRJ_TRY_CUDA(stager.reserve(nt * (6 * 32 + 8) + (size_t)d->n_nodes * 72 + small_bytes + 16 * 256));
    cudaStream_t stream = stager.stream; // the device's preparation stream
    if (nt) {
        const double *src[6] = {d->tri_v0, d->tri_v1, d->tri_v2, d->tri_n0, d->tri_n1, d->tri_n2};
        for (int k = 0; k < 6; k++) VRJ_TRY_CUDA(stager.copy(rb + r_v[k], src[k], nt * 32));
        VRJ_TRY_CUDA(stager.copy(rb + r_mat, d->tri_material, nt * 4));
        VRJ_TRY_CUDA(stager.copy(rb + r_pid, d->tri_prim_id, nt * 4));
    }
    if (d->n_nodes) {
        VRJ_TRY_CUDA(stager.copy(rb + r_min, d->node_min, (size_t)d->n_nodes * 32));
        VRJ_TRY_CUDA(stager.copy(rb + r_max, d->node_max, (size_t)d->n_nodes * 32));
        VRJ_TRY_CUDA(stager.copy(rb + r_child, d->node_child, (size_t)d->n_nodes * 8));
    }
    auto t_raw = std::chrono::steady_clock::now();
    RawTriangles rt;
    rt.v0 = reinterpret_cast<const double *>(rb + r_v[0]), rt.v1 = reinterpret_cast<const double *>(rb + r_v[1]);
    rt.v2 = reinterpret_cast<const double *>(rb + r_v[2]), rt.n0 = reinterpret_cast<const double *>(rb + r_v[3]);
    rt.n1 = reinterpret_cast<const double *>(rb + r_v[4]), rt.n2 = reinterpret_cast<const double *>(rb + r_v[5]);
    rt.material = reinterpret_cast<const uint32_t *>(rb + r_mat), rt.prim_id = reinterpret_cast<const uint32_t *>(rb + r_pid);
    double *dn_min = reinterpret_cast<double *>(rb + r_min), *dn_max = reinterpret_cast<double *>(rb + r_max);
    int32_t *dn_child = reinterpret_cast<int32_t *>(rb + r_child);
    uint32_t *perm = nullptr;
    std::vector<double> built_root(d->n_bvhs * 8, 0.0); // root boxes of the BVHs built here (for the items' pre-test)
    if (any_build) {
        perm = reinterpret_cast<uint32_t *>(rb + r_perm);
        k_identity_perm<<<(unsigned)((nt + 255) / 256), 256, 0, stream>>>((uint32_t)nt, perm);
        for (uint32_t b = 0; b < d->n_bvhs; b++) {
            if (!plan[b].build) continue;
            const VrjBvh &bv = d->bvhs[b];
            const uint32_t n = (uint32_t)bv.n_triangles, first = (uint32_t)bv.first_triangle;
            double *bvv = reinterpret_cast<double *>(rb + r_bv);
            uint32_t *border = reinterpret_cast<uint32_t *>(rb + r_bo);
            k_gather_vertices<<<(n + 255) / 256, 256, 0, stream>>>(n, rt.v0 + 4 * (size_t)first, rt.v1 + 4 * (size_t)first, rt.v2 + 4 * (size_t)first, bvv);
            VrjStatus bs = vrj_build::build_device(n, bvv, border, dn_min + 4 * plan[b].first_node, dn_max + 4 * plan[b].first_node,
                                                   dn_child + 2 * plan[b].first_node, stream, nullptr);
            if (bs != VRJ_OK) {
                delete sc;
                return bs;
            }
            k_offset_perm<<<(n + 255) / 256, 256, 0, stream>>>(n, border, first, perm);
            VRJ_TRY_CUDA(cudaMemcpyAsync(&built_root[b * 8], dn_min + 4 * plan[b].first_node, 32, cudaMemcpyDeviceToHost, stream));
            VRJ_TRY_CUDA(cudaMemcpyAsync(&built_root[b * 8 + 4], dn_max + 4 * plan[b].first_node, 32, cudaMemcpyDeviceToHost, stream));
        }
    }
    // the 16-bit grid of VRJ_FILTER_Q16 spans the root boxes of all meshes (those built above are read back first)
    QGrid grid_q;
    {
        QGrid &grid = grid_q;
        if (any_build) VRJ_TRY_CUDA(cudaStreamSynchronize(stream));
        double glo[3] = {std::numeric_limits<double>::infinity(), std::numeric_limits<double>::infinity(), std::numeric_limits<double>::infinity()};
        double ghi[3] = {-glo[0], -glo[1], -glo[2]};
        for (uint32_t b = 0; b < d->n_bvhs; b++) {
            if (plan[b].empty) continue;
            const double *rmin = plan[b].build ? &built_root[b * 8] : d->node_min + d->bvhs[b].first_node * 4;
            const double *rmax = plan[b].build ? &built_root[b * 8 + 4] : d->node_max + d->bvhs[b].first_node * 4;
            for (int k = 0; k < 3; k++) glo[k] = std::fmin(glo[k], rmin[k]), ghi[k] = std::fmax(ghi[k], rmax[k]);
        }
        for (int k = 0; k < 3; k++) {
            const bool ok = std::isfinite(glo[k]) && std::isfinite(ghi[k]) && ghi[k] > glo[k];
            grid.lo[k] = std::isfinite(glo[k]) ? glo[k] : 0.0;
            grid.cell[k] = ok ? (ghi[k] - glo[k]) / 65534.0 : 1e-30;
            sc->dev.qlo[k] = grid.lo[k], sc->dev.qcell[k] = grid.cell[k];
        }
    }
    if (nt)
        k_pack_triangles<<<(unsigned)((nt + 127) / 128), 128, 0, stream>>>((uint32_t)nt, rt, perm, reinterpret_cast<double *>(base + s_tp.offset),
                                                                           reinterpret_cast<double *>(base + s_tn.offset),
                                                                           reinterpret_cast<float *>(base + s_tp32.offset),
                                                                           reinterpret_cast<float *>(base + s_tn32.offset));
    for (uint32_t b = 0; b < d->n_bvhs; b++) {
        if (plan[b].empty) continue;
        BvhNodes bn;
        bn.node_min = dn_min, bn.node_max = dn_max, bn.node_child = dn_child;
        bn.first_node = (uint32_t)plan[b].first_node, bn.n_nodes = (uint32_t)plan[b].n_nodes;
        bn.child_offset = plan[b].build ? (int32_t)plan[b].first_node : 0;
        bn.triangle_offset = plan[b].build ? (int32_t)d->bvhs[b].first_triangle : 0;
        bn.wide_base = (uint32_t)plan[b].wide_base;
        uint32_t *flags = reinterpret_cast<uint32_t *>(rb + r_flags);
        const unsigned grid = (bn.n_nodes + 255) / 256;
        k_mark_internal<<<grid, 256, 0, stream>>>(bn, flags);
        VrjStatus ss = vrj_build::exclusive_scan_u32(flags, bn.n_nodes, reinterpret_cast<uint32_t *>(rb + r_scan), stream);
        if (ss != VRJ_OK) {
            delete sc;
            return ss;
        }
        k_wide_nodes<<<grid, 256, 0, stream>>>(bn, flags, reinterpret_cast<float *>(base + s_n32.offset), reinterpret_cast<double *>(base + s_n64.offset));
        k_q16_nodes<<<grid, 256, 0, stream>>>(bn, flags, grid_q, reinterpret_cast<uint4 *>(base + s_nq.offset));
        // the 4-wide form of the same tree (VRJ_FILTER_F32X4); its nodes are numbered from the same base (there are fewer of them)
        uint32_t *parent = reinterpret_cast<uint32_t *>(rb + r_parent), *is_quad = reinterpret_cast<uint32_t *>(rb + r_isquad);
        k_parents<<<grid, 256, 0, stream>>>(bn, parent);
        k_quad_flags<<<grid, 256, 0, stream>>>(bn, parent, is_quad);
        VRJ_TRY_CUDA(cudaMemcpyAsync(flags, is_quad, (size_t)bn.n_nodes * 4, cudaMemcpyDeviceToDevice, stream));
        ss = vrj_build::exclusive_scan_u32(flags, bn.n_nodes, reinterpret_cast<uint32_t *>(rb + r_scan), stream);
        if (ss != VRJ_OK) {
            delete sc;
            return ss;
        }
        k_quad_nodes<<<grid, 256, 0, stream>>>(bn, flags, is_quad, reinterpret_cast<float *>(base + s_n4.offset));
    }
    VRJ_TRY_CUDA(cudaGetLastError());
    VRJ_TRY_CUDA(cudaStreamSynchronize(stream)); // built_root is read below

    // ---- the small tables ----
    char *stage = area.block + stager.cursor; // the staged arrays before it were copied before the synchronize above
    std::memset(stage, 0, small_bytes);
    SpectrumDev *spectra = reinterpret_cast<SpectrumDev *>(stage + s_spc.offset);
    for (uint32_t i = 0; i < d->n_spectra; i++)
        spectra[i] = SpectrumDev{d->spectra[i].shortest_wavelength, d->spectra[i].longest_wavelength, d->spectra[i].first_sample, d->spectra[i].n_samples};
    if (d->n_spectrum_samples) std::memcpy(stage + s_smp.offset, d->spectrum_samples, d->n_spectrum_samples * sizeof(double));
    // wavelength of every sample, with the operations of spectrum.rs:62,67 (`i as f64 / (n-1) as f64 * range + shortest`): the
    // lookup on the device reads these instead of dividing twice per call (vrj_device.cuh, spectrum_lookup_grid)
    {
        volatile double *grid = reinterpret_cast<double *>(stage + s_grd.offset); // volatile: no contraction / reassociation by the host compiler
        for (uint32_t i = 0; i < d->n_spectra; i++) {
            const VrjSpectrum &sp = d->spectra[i];
            const double range = sp.longest_wavelength - sp.shortest_wavelength, nm1 = (double)(sp.n_samples - 1);
            for (uint32_t k = 0; k < sp.n_samples; k++) {
                const double q = (double)k / nm1;
                const double scaled = q * range;
                grid[sp.first_sample + k] = scaled + sp.shortest_wavelength;
            }
        }
    }
    MaterialDev *materials = reinterpret_cast<MaterialDev *>(stage + s_mat.offset);
    for (uint32_t i = 0; i < d->n_materials; i++)
        materials[i] = MaterialDev{d->materials[i].kind, d->materials[i].spectrum, d->materials[i].p0, d->materials[i].p1, d->materials[i].p2};
    SphereDev *spheres = reinterpret_cast<SphereDev *>(stage + s_sph.offset);
    for (uint32_t i = 0; i < d->n_spheres; i++)
        spheres[i] = SphereDev{d->spheres[i].centre[0], d->spheres[i].centre[1], d->spheres[i].centre[2], d->spheres[i].radius, d->spheres[i].material, 0};
    PlaneDev *planes = reinterpret_cast<PlaneDev *>(stage + s_pl.offset);
    for (uint32_t i = 0; i < d->n_planes; i++) {
        PlaneDev &p = planes[i];
        for (int k = 0; k < 3; k++) p.n[k] = d->planes[i].normal[k], p.t[k] = d->planes[i].tangent[k], p.c[k] = d->planes[i].cotangent[k];
        p.distance = d->planes[i].distance_from_origin, p.material = d->planes[i].material, p.pad = 0;
    }
    ItemDev *items = reinterpret_cast<ItemDev *>(stage + s_it.offset);
    uint32_t *analytic_items = reinterpret_cast<uint32_t *>(stage + s_an.offset), *bvh_items = reinterpret_cast<uint32_t *>(stage + s_bv.offset);
    uint32_t n_items = 0, n_analytic = 0, n_bvh_items = 0;
    for (uint32_t i = 0; i < d->n_items; i++) {
        const VrjItem &it = d->items[i];
        if (it.kind == VRJ_ITEM_BVH && plan[it.index].empty) continue; // an empty BVH never reports a hit
        ItemDev id{};
        id.kind = it.kind, id.index = it.index, id.object_id = it.object_id, id.prim_id = it.prim_id;
        id.root = it.kind == VRJ_ITEM_BVH ? (uint32_t)plan[it.index].wide_base : 0u;
        if (it.kind == VRJ_ITEM_BVH) {
            const double *rmin = plan[it.index].build ? &built_root[it.index * 8] : d->node_min + d->bvhs[it.index].first_node * 4;
            const double *rmax = plan[it.index].build ? &built_root[it.index * 8 + 4] : d->node_max + d->bvhs[it.index].first_node * 4;
            for (int k = 0; k < 3; k++) id.lo[k] = round_down_f32(rmin[k]), id.hi[k] = round_up_f32(rmax[k]);
            bvh_items[n_bvh_items++] = n_items;
        } else {
            analytic_items[n_analytic++] = n_items;
        }
        items[n_items++] = id;
    }
    auto t_prep = std::chrono::steady_clock::now();
    VRJ_TRY_CUDA(cudaMemcpyAsync(base, stage, small_bytes, cudaMemcpyHostToDevice, stream));
    VRJ_TRY_CUDA(cudaStreamSynchronize(stream));
#undef VRJ_TRY_CUDA
    sc->device_bytes = arena_bytes;
    sc->upload_bytes = stager.copied + small_bytes; // what crossed PCIe: the caller's arrays + the small tables
    sc->dev.nodes32 = reinterpret_cast<const float4 *>(base + s_n32.offset);
    sc->dev.nodes64 = reinterpret_cast<const double2 *>(base + s_n64.offset);
    sc->dev.nodes4 = reinterpret_cast<const float4 *>(base + s_n4.offset);
    sc->dev.nodesq = reinterpret_cast<const uint4 *>(base + s_nq.offset);
    sc->dev.tri_pos = reinterpret_cast<const double2 *>(base + s_tp.offset);
    sc->dev.tri_nrm = reinterpret_cast<const double2 *>(base + s_tn.offset);
    sc->dev.tri_pos32 = reinterpret_cast<const float4 *>(base + s_tp32.offset);
    sc->dev.tri_nrm32 = reinterpret_cast<const float4 *>(base + s_tn32.offset);
    sc->dev.spheres = reinterpret_cast<const SphereDev *>(base + s_sph.offset);
    sc->dev.planes = reinterpret_cast<const PlaneDev *>(base + s_pl.offset);
    sc->dev.materials = reinterpret_cast<const MaterialDev *>(base + s_mat.offset);
    sc->dev.spectra = reinterpret_cast<const SpectrumDev *>(base + s_spc.offset);
    sc->dev.spectrum_samples = reinterpret_cast<const double *>(base + s_smp.offset);
    sc->dev.spectrum_grids = reinterpret_cast<const double *>(base + s_grd.offset);
    sc->dev.material_mask = 0;
    for (uint32_t i = 0; i < d->n_materials; i++) sc->dev.material_mask |= 1u << d->materials[i].kind;
    sc->kernel_material_mask = sc->dev.material_mask == 1u ? 1u : (uint32_t)VRJ_MM_ALL;
    if (const char *mm = std::getenv("VRJ_MATERIAL_MASK")) // experiments only: 15 = always the general kernels
        if (std::atoi(mm) == VRJ_MM_ALL) sc->kernel_material_mask = VRJ_MM_ALL;
    sc->dev.items = reinterpret_cast<const ItemDev *>(base + s_it.offset);
    sc->dev.analytic_items = reinterpret_cast<const uint32_t *>(base + s_an.offset);
    sc->dev.bvh_items = reinterpret_cast<const uint32_t *>(base + s_bv.offset);
    sc->dev.n_items = n_items, sc->dev.n_analytic = n_analytic, sc->dev.n_bvh_items = n_bvh_items;
    for (int k = 0; k < 3; k++) sc->dev.cam[k] = d->camera_location[k];
    sc->dev.refill_threshold = 16, sc->dev.leaf_threshold = 2, sc->dev.node_batch = 4, sc->dev.max_iters = 64, sc->dev.node_batch4 = 2;
    if (const char *tune = std::getenv("VRJ_TUNE")) // experiments only: "refill,leaf,node_batch,max_iters,tail_max,node_batch4"
        std::sscanf(tune, "%d,%d,%d,%d,%u,%d", &sc->dev.refill_threshold, &sc->dev.leaf_threshold, &sc->dev.node_batch, &sc->dev.max_iters, &sc->tail_max,
                    &sc->dev.node_batch4);
    if (const char *pb = std::getenv("VRJ_PATH_BUDGET_LOG2")) sc->path_budget = 1ull << std::min(std::max(std::atoi(pb), 16), 31); // experiments only
    if (const char *r = std::getenv("VRJ_RECORDS")) sc->trace_records = std::atoi(r) != 0; // experiments only
    sc->auto_q16 = (size_t)d->n_triangles * 64 > (size_t(96) << 20); // the f32 nodes (64 bytes per triangle) against the 126 MB L2
    if (const char *aq = std::getenv("VRJ_AUTO_Q16")) sc->auto_q16 = std::atoi(aq) != 0; // experiments only
    if (const char *ts = std::getenv("VRJ_TAIL_SHALLOW")) sc->tail_max_shallow = (uint32_t)std::strtoul(ts, nullptr, 10); // experiments only
    if (std::getenv("VRJ_TIMING")) {
        auto t_end = std::chrono::steady_clock::now();
        auto ms = [](std::chrono::steady_clock::time_point a, std::chrono::steady_clock::time_point b) {
            return std::chrono::duration<double, std::milli>(b - a).count();
        };
        std::fprintf(stderr, "vrj_scene_create: validate %.2f ms, device alloc %.2f ms, copies queued %.2f ms, device build + pack %.2f ms, tables %.2f ms\n",
                     ms(t_start, t_valid), ms(t_valid, t_alloc), ms(t_alloc, t_raw), ms(t_raw, t_prep), ms(t_prep, t_end));
    }
    *out = sc;
    return VRJ_OK;
#undef VRJ_TRY
}

void vrj_scene_destroy(VrjScene *scene) {
    if (!scene) return;
    DeviceGuard device_guard;
    cudaSetDevice(scene->device);
    delete scene;
}

uint64_t vrj_scene_device_bytes(const VrjScene *scene) { return scene ? scene->device_bytes : 0; }
uint64_t vrj_scene_upload_bytes(const VrjScene *scene) { return scene ? scene->upload_bytes : 0; }

void vrj_release_scratch(void) {
    DeviceGuard device_guard;
    {
        std::lock_guard<std::mutex> g(g_pool_mutex);
        for (auto &e : g_pool) {
            cudaSetDevice(e.first);
            delete e.second;
        }
        g_pool.clear();
    }
    vrj_pool_trim();
    std::vector<HostBlock> victims;
    {
        std::lock_guard<std::mutex> g(g_host_pool_mutex);
        victims.swap(g_host_pool_free);
    }
    for (const HostBlock &b : victims) cudaFreeHost(b.p);
}

// Page-locked host memory is pooled like device memory: cudaMallocHost / cudaFreeHost of an AccumulationBuffer's
// 182 MB cost tens of milliseconds, more than rendering into it.  vrj_release_scratch() empties the pool.
void *vrj_alloc_host(uint64_t bytes) {
    const size_t want = (std::max<size_t>(bytes, 1) + 4095) & ~size_t(4095);
    {
        std::lock_guard<std::mutex> g(g_host_pool_mutex);
        size_t best = g_host_pool_free.size();
        for (size_t i = 0; i < g_host_pool_free.size(); i++) {
            const HostBlock &b = g_host_pool_free[i];
            if (b.bytes >= want && b.bytes <= 2 * want + (size_t(1) << 20) && (best == g_host_pool_free.size() || b.bytes < g_host_pool_free[best].bytes))
                best = i;
        }
        if (best != g_host_pool_free.size()) {
            HostBlock b = g_host_pool_free[best];
            g_host_pool_free.erase(g_host_pool_free.begin() + best);
            g_host_pool_live[b.p] = b.bytes;
            return b.p;
        }
    }
    void *p = nullptr;
    g_n_host_mallocs++;
    if (cudaMallocHost(&p, want) != cudaSuccess) {
        g_error = "cudaMallocHost failed";
        cudaGetLastError();
        return nullptr;
    }
    std::lock_guard<std::mutex> g(g_host_pool_mutex);
    g_host_pool_live[p] = want;
    return p;
}
void vrj_free_host(void *p) {
    if (!p) return;
    bool keep = false;
    {
        std::lock_guard<std::mutex> g(g_host_pool_mutex);
        auto it = g_host_pool_live.find(p);
        if (it != g_host_pool_live.end()) {
            size_t cached = 0;
            for (const HostBlock &b : g_host_pool_free) cached += b.bytes;
            // room for the buffers of a pool of concurrent callers (main.rs:197-209): 16 in flight x 5 arrays
            keep = cached + it->second <= (size_t(16) << 30) && g_host_pool_free.size() < 256;
            if (keep) g_host_pool_free.push_back(HostBlock{p, it->second});
            g_host_pool_live.erase(it);
        }
    }
    if (!keep) cudaFreeHost(p);
}

void *vrj_alloc_device(int32_t device, uint64_t bytes) {
    DeviceGuard device_guard;
    void *p = nullptr;
    if (cudaSetDevice(device) != cudaSuccess || vrj_pool_alloc(&p, bytes) != cudaSuccess || cudaMemset(p, 0, bytes) != cudaSuccess) {
        g_error = std::string("vrj_alloc_device: ") + cudaGetErrorString(cudaGetLastError());
        if (p) vrj_pool_free(p);
        return nullptr;
    }
    return p;
}
void vrj_free_device(void *p) { vrj_pool_free(p); }
VrjStatus vrj_copy_to_host(int32_t device, void *host_dst, const void *device_src, uint64_t bytes) {
    DeviceGuard device_guard;
    if (bytes && (!host_dst || !device_src)) return fail(VRJ_ERR_INVALID_ARGUMENT, "NULL argument");
    VRJ_CUDA(cudaSetDevice(device));
    VRJ_CUDA(cudaMemcpy(host_dst, device_src, bytes, cudaMemcpyDeviceToHost));
    return VRJ_OK;
}

VrjStatus vrj_render_tile(const VrjScene *scene_c, const VrjTile *tile, uint64_t height, uint64_t width,
                          const VrjRenderParams *p, VrjAccumOut *out) {
    VrjScene *scene = const_cast<VrjScene *>(scene_c);
    size_t n_light_samples = 0;
    VrjStatus st = check_render_args(scene, tile, height, width, p, out, &n_light_samples);
    if (st != VRJ_OK) return st;
    const uint64_t tw = tile->end_column - tile->start_column, th = tile->end_row - tile->start_row;
    const uint64_t npix = tw * th;
    DeviceGuard device_guard;
    static const bool timing = std::getenv("VRJ_TIMING") != nullptr;
    VRJ_NVTX_RANGE(call_range, "vrj_render_tile");
    const auto t_call0 = std::chrono::steady_clock::now();
    if (out->stats) std::memset(out->stats, 0, sizeof(VrjStats));
    if (npix == 0 || p->spp == 0) return VRJ_OK;
    VRJ_CUDA(cudaSetDevice(scene->device));

    // batch: as many samples of the whole tile in flight as fit the path budget
    ActiveCall active(g_active_calls[(unsigned)scene->device % 64]);
    if (coalescable(p, out, npix)) return render_coalesced(scene, tile, height, width, p, out);
    RenderCall call(scene, p, npix);
    st = call.prepare(p->spp, active, n_light_samples);
    if (st != VRJ_OK) return st;
    Scratch *s = call.s;
    const uint32_t batch = call.batch;

    st = call.load_state(out, out->accumulate);
    if (st != VRJ_OK) return st;
    st = call.start(tile, height, width);
    if (st != VRJ_OK) return st;
    RenderConst &rc = call.rc;
    const AccumDev acc = s->accum();
    const double2 *photons = s->photons.as<double2>();
    // The last batch's resolve runs in `pieces` row-aligned pieces, and each piece's part of the arrays is copied to the caller
    // on a second stream as soon as it is resolved: at 1080p the copy back (66 MB, 1.25 ms over PCIe) hides behind the 1.6 ms
    // the seven exponentials per sample take, instead of following them.  Small tiles and device-memory outputs (copies at HBM
    // speed) keep the single resolve (worth it when the resolve is long enough to hide a copy behind: with a sample or two per
    // pixel it is 0.06 ms against 1.25 ms).
    const uint32_t pieces = 4;
    bool piecewise = out->memory == VRJ_MEM_HOST && npix >= (uint64_t(1) << 18) && std::min(batch, p->spp) >= 8 && !std::getenv("VRJ_NO_PIECEWISE_COPY");
    for (int i = 0; i < 5 && piecewise; i++) { // page-locked destinations only: a copy into pageable memory holds the enqueueing thread
        cudaPointerAttributes attr{};
        if (call.arrs[i].user && (cudaPointerGetAttributes(&attr, call.arrs[i].user) != cudaSuccess || attr.type != cudaMemoryTypeHost)) piecewise = false;
    }
    cudaGetLastError();
    for (uint32_t done = 0; done < p->spp; done += batch) {
        rc.batch_samples = std::min(batch, p->spp - done);
        const bool copy = piecewise && done + batch >= p->spp;
        call.pieces_copied = call.pieces_copied || copy;
        rc.div_batch = FastDiv::make(rc.batch_samples);
        rc.first_sample = p->sample_offset + (uint64_t)done * rc.sample_stride;
        st = dispatch_batch(scene, s, rc, p, call.filter, &call.launches);
        if (st != VRJ_OK) return st;
        st = resolve_batch(s, p, [&](auto r) -> VrjStatus {
            using R = decltype(r);
            if (!copy) {
                k_resolve<R><<<(rc.npix + 255) / 256, 256, 0, s->stream>>>(acc, photons, 0u, rc.npix, rc.batch_samples);
                call.launches++;
                return VRJ_OK;
            }
            const uint32_t step = ((rc.npix + pieces - 1) / pieces + 255u) & ~255u; // whole CTAs per piece
            uint32_t piece = 0;
            for (uint32_t first = 0; first < rc.npix; first += step, piece++) {
                const uint32_t end = std::min(rc.npix, first + step);
                k_resolve<R><<<(end - first + 255) / 256, 256, 0, s->stream>>>(acc, photons, first, end, rc.batch_samples);
                call.launches++;
                VRJ_CUDA(cudaEventRecord(s->piece_ev[piece], s->stream));
                VRJ_CUDA(cudaStreamWaitEvent(s->copy_stream, s->piece_ev[piece], 0));
                for (int i = 0; i < 5; i++) {
                    const Arr &a = call.arrs[i];
                    if (a.user)
                        VRJ_CUDA(cudaMemcpyAsync(a.user + (size_t)first * a.per, a.dev->as<double>() + (size_t)first * a.per, (size_t)(end - first) * a.per * sizeof(double),
                                                 call.out_kind, s->copy_stream));
                }
            }
            VRJ_CUDA(cudaEventRecord(s->copy_done, s->copy_stream));
            return VRJ_OK;
        });
        if (st != VRJ_OK) return st;
        if (out->photons) {
            // debug output, batch-major: [(sample * npix + pixel) * 2]; the device keeps the batch pixel-major, so transpose
            // into queue 0's storage (free at this point: 6 x 16 bytes per path >= 16 bytes per sample)
            double2 *tmp = s->queues[0][0].as<double2>();
            const size_t count = (size_t)rc.batch_samples * npix;
            k_photons_sample_major<<<(unsigned)((count + 255) / 256), 256, 0, s->stream>>>(photons, tmp, (uint32_t)npix, rc.batch_samples);
            call.launches++;
            VRJ_CUDA(cudaMemcpyAsync(out->photons + (size_t)done * npix * 2, tmp, count * sizeof(double2), call.out_kind, s->stream));
        }
    }
    st = call.finish();
    if (st != VRJ_OK) return st;
    if (timing) {
        auto msd = [](std::chrono::steady_clock::time_point a, std::chrono::steady_clock::time_point b) {
            return std::chrono::duration<double, std::milli>(b - a).count();
        };
        std::fprintf(stderr, "vrj_render_tile: setup %.3f ms, enqueue %.3f ms, wait %.3f ms (device %.3f ms, %llu launches)\n",
                     msd(t_call0, call.t_start), msd(call.t_start, call.t_enqueued), msd(call.t_enqueued, call.t_done), call.ms,
                     (unsigned long long)call.launches);
    }
    return VRJ_OK;
}

// Adaptive sampling (the header states the passes and the stopping rule): render_passes from a zero state, until no pixel is
// active.
VrjStatus vrj_render_adaptive(const VrjScene *scene_c, const VrjTile *tile, uint64_t height, uint64_t width, const VrjRenderParams *p,
                              const VrjAdaptiveParams *ap, VrjAccumOut *out, double *y_sq_sum, VrjAdaptiveStats *astats) {
    VrjScene *scene = const_cast<VrjScene *>(scene_c);
    size_t n_light_samples = 0;
    VrjStatus st = check_render_args(scene, tile, height, width, p, out, &n_light_samples);
    if (st != VRJ_OK) return st;
    PassRule rule;
    st = check_pass_rule(p, ap, "vrj_render_adaptive", "VrjAdaptiveParams", &rule);
    if (st != VRJ_OK) return st;
    if (out->accumulate) return fail(VRJ_ERR_UNSUPPORTED, "vrj_render_adaptive does not continue from a previous state (accumulate)");
    if (out->photons) return fail(VRJ_ERR_UNSUPPORTED, "vrj_render_adaptive has no photons output");
    const uint64_t npix = (tile->end_column - tile->start_column) * (tile->end_row - tile->start_row);
    DeviceGuard device_guard;
    VRJ_NVTX_RANGE(call_range, "vrj_render_adaptive");
    if (out->stats) std::memset(out->stats, 0, sizeof(VrjStats));
    if (astats) std::memset(astats, 0, sizeof(VrjAdaptiveStats));
    if (npix == 0) return VRJ_OK;
    VRJ_CUDA(cudaSetDevice(scene->device));
    PassResult res;
    st = render_passes(scene, tile, height, width, p, rule, 0, n_light_samples, out, y_sq_sum, &res);
    if (st != VRJ_OK) return st;
    if (astats) {
        astats->passes = res.passes, astats->samples = res.samples;
        astats->pixels_converged = res.counts.converged, astats->pixels_unconverged = res.counts.at_max;
    }
    return VRJ_OK;
}

// Progressive rendering (the header states the schedule): render_passes on the caller's state.
VrjStatus vrj_render_progressive(const VrjScene *scene_c, const VrjTile *tile, uint64_t height, uint64_t width, const VrjRenderParams *p,
                                 const VrjProgressiveParams *pp, VrjAccumOut *out, double *y_sq_sum, VrjProgressiveStats *pstats) {
    VrjScene *scene = const_cast<VrjScene *>(scene_c);
    size_t n_light_samples = 0;
    VrjStatus st = check_render_args(scene, tile, height, width, p, out, &n_light_samples);
    if (st != VRJ_OK) return st;
    PassRule rule;
    st = check_pass_rule(p, pp, "vrj_render_progressive", "VrjProgressiveParams", &rule);
    if (st != VRJ_OK) return st;
    if (out->memory > VRJ_MEM_DEVICE) return fail(VRJ_ERR_INVALID_ARGUMENT, "unknown memory kind");
    if (!out->colour_sum || !out->colour_bias || !out->weight || !out->weight_bias || !y_sq_sum)
        return fail(VRJ_ERR_INVALID_ARGUMENT, "the state (colour_sum, colour_bias, weight, weight_bias, y_sq_sum) is required");
    if (out->photons) return fail(VRJ_ERR_UNSUPPORTED, "vrj_render_progressive has no photons output");
    const uint64_t npix = (tile->end_column - tile->start_column) * (tile->end_row - tile->start_row);
    DeviceGuard device_guard;
    VRJ_NVTX_RANGE(call_range, "vrj_render_progressive");
    if (out->stats) std::memset(out->stats, 0, sizeof(VrjStats));
    if (pstats) std::memset(pstats, 0, sizeof(VrjProgressiveStats));
    if (npix == 0) return VRJ_OK;
    VRJ_CUDA(cudaSetDevice(scene->device));
    PassResult res;
    st = render_passes(scene, tile, height, width, p, rule, pp->max_passes, n_light_samples, out, y_sq_sum, &res);
    if (st != VRJ_OK) return st;
    if (pstats) {
        pstats->passes = res.passes, pstats->samples = res.samples;
        pstats->pixels_converged = res.counts.converged, pstats->pixels_at_max = res.counts.at_max, pstats->pixels_active = res.counts.active;
    }
    return VRJ_OK;
}

// Per-pixel sample counts in full wavefronts (the header states the call): render_counts on the caller's state.
VrjStatus vrj_render_counts(const VrjScene *scene_c, const VrjTile *tile, uint64_t height, uint64_t width, const VrjRenderParams *p,
                            const uint32_t *counts, VrjAccumOut *out, double *y_sq_sum, VrjCountsStats *cstats) {
    VrjScene *scene = const_cast<VrjScene *>(scene_c);
    size_t n_light_samples = 0;
    VrjStatus st = check_render_args(scene, tile, height, width, p, out, &n_light_samples);
    if (st != VRJ_OK) return st;
    if (p->spp != 0) return fail(VRJ_ERR_INVALID_ARGUMENT, "params->spp must be 0: vrj_render_counts takes its sample counts from `counts`");
    if (out->memory > VRJ_MEM_DEVICE) return fail(VRJ_ERR_INVALID_ARGUMENT, "unknown memory kind");
    if (out->accumulate && (!out->colour_sum || !out->colour_bias || !out->weight || !out->weight_bias))
        return fail(VRJ_ERR_INVALID_ARGUMENT, "a continued state (accumulate) needs colour_sum, colour_bias, weight and weight_bias");
    if (out->photons) return fail(VRJ_ERR_UNSUPPORTED, "vrj_render_counts has no photons output");
    const uint64_t npix = (tile->end_column - tile->start_column) * (tile->end_row - tile->start_row);
    if (npix && !counts) return fail(VRJ_ERR_INVALID_ARGUMENT, "counts is NULL");
    DeviceGuard device_guard;
    VRJ_NVTX_RANGE(call_range, "vrj_render_counts");
    if (out->stats) std::memset(out->stats, 0, sizeof(VrjStats));
    if (cstats) std::memset(cstats, 0, sizeof(VrjCountsStats));
    if (npix == 0) return VRJ_OK;
    VRJ_CUDA(cudaSetDevice(scene->device));
    return render_counts(scene, tile, height, width, p, counts, n_light_samples, out, y_sq_sum, cstats);
}

// The planner (the header states the rule): k_plan_counts, one thread per pixel, on a stream of its own.  The counts go to a
// pooled buffer first and reach the caller only when every weight was a sample count.
VrjStatus vrj_plan_counts(int32_t device, uint32_t memory, uint64_t npix, const double *weight, const double *colour_sum, const double *y_sq_sum,
                          const VrjAdaptiveParams *rule, uint32_t *counts, VrjPlanStats *pstats) {
    PassRule r;
    VrjStatus st = check_rule(rule, &r);
    if (st != VRJ_OK) return st;
    if (memory > VRJ_MEM_DEVICE) return fail(VRJ_ERR_INVALID_ARGUMENT, "unknown memory kind");
    if (pstats) std::memset(pstats, 0, sizeof(VrjPlanStats));
    if (npix == 0) return VRJ_OK;
    if (!weight || !colour_sum || !y_sq_sum || !counts) return fail(VRJ_ERR_INVALID_ARGUMENT, "NULL argument");
    if (npix > 0xffffffffull) return fail(VRJ_ERR_UNSUPPORTED, "more than 2^32 - 1 pixels");
    const uint32_t n32 = (uint32_t)npix;
    DeviceGuard device_guard;
    VRJ_NVTX_RANGE(call_range, "vrj_plan_counts");
    VRJ_CUDA(cudaSetDevice(device));
    DeviceBuffer d_in[3], d_counts, d_ctr;
    const void *src[3] = {weight, colour_sum, y_sq_sum};
    const size_t per[3] = {8, 24, 8};
    const bool host = memory == VRJ_MEM_HOST;
    if (host)
        for (int i = 0; i < 3; i++) VRJ_CUDA(d_in[i].alloc(npix * per[i]));
    VRJ_CUDA(d_counts.alloc(npix * 4));
    VRJ_CUDA(d_ctr.alloc(5 * sizeof(unsigned long long)));
    CallStream cs;
    VRJ_CUDA(cs.create());
    if (host) {
        for (int i = 0; i < 3; i++) VRJ_CUDA(cudaMemcpyAsync(d_in[i].p, src[i], npix * per[i], cudaMemcpyHostToDevice, cs.s));
        for (int i = 0; i < 3; i++) src[i] = d_in[i].p;
    }
    unsigned long long h[5] = {0, 0, 0, 0, 0};
    VRJ_CUDA(cudaMemsetAsync(d_ctr.p, 0, 5 * sizeof(unsigned long long), cs.s));
    k_plan_counts<<<(n32 + 255) / 256, 256, 0, cs.s>>>(static_cast<const double *>(src[0]), static_cast<const double *>(src[1]),
                                                       static_cast<const double *>(src[2]), n32, r, d_counts.as<uint32_t>(), d_ctr.as<unsigned long long>());
    VRJ_CUDA(cudaGetLastError());
    VRJ_CUDA(cudaMemcpyAsync(h, d_ctr.p, sizeof(h), cudaMemcpyDeviceToHost, cs.s));
    VRJ_CUDA(cudaStreamSynchronize(cs.s));
    if (h[4]) return fail(VRJ_ERR_INVALID_ARGUMENT, "a weight of the state is not a sample count (negative, fractional, not finite or >= 2^32)");
    VRJ_CUDA(cudaMemcpyAsync(counts, d_counts.p, npix * 4, host ? cudaMemcpyDeviceToHost : cudaMemcpyDeviceToDevice, cs.s));
    VRJ_CUDA(cudaStreamSynchronize(cs.s));
    if (pstats) pstats->samples = h[0], pstats->pixels_planned = h[1], pstats->pixels_converged = h[2], pstats->pixels_at_max = h[3];
    return VRJ_OK;
}


// First-hit features (the header states them): k_aux, one thread per pixel, forms each pixel's camera rays from the render's
// RenderConst.  Like vrj_trace_rays it runs on a stream of its own and takes no render turn.
VrjStatus vrj_render_aux(const VrjScene *scene_c, const VrjTile *tile, uint64_t height, uint64_t width, const VrjRenderParams *p,
                         VrjAuxOut *out) {
    VrjScene *scene = const_cast<VrjScene *>(scene_c);
    if (!scene || !tile || !p || !out) return fail(VRJ_ERR_INVALID_ARGUMENT, "NULL argument");
    VrjStatus st = check_tile(tile, height, width);
    if (st != VRJ_OK) return st;
    if (p->spp == 0) return fail(VRJ_ERR_INVALID_ARGUMENT, "params->spp must be >= 1");
    if (out->memory > VRJ_MEM_DEVICE) return fail(VRJ_ERR_INVALID_ARGUMENT, "unknown memory kind");
    if (out->stats) std::memset(out->stats, 0, sizeof(VrjStats));
    const uint64_t npix = (tile->end_column - tile->start_column) * (tile->end_row - tile->start_row);
    if (npix == 0) return VRJ_OK;
    if (npix * (uint64_t)p->spp > 0xffffffffull) return fail(VRJ_ERR_UNSUPPORTED, "more than 2^32 camera rays in one call");
    DeviceGuard device_guard;
    VRJ_NVTX_RANGE(call_range, "vrj_render_aux");
    VRJ_CUDA(cudaSetDevice(scene->device));
    RenderConst rc = make_render_const(tile, height, width, p);
    rc.batch_samples = p->spp, rc.first_sample = p->sample_offset;
    rc.div_batch = FastDiv::make(p->spp), rc.div_tile_w = FastDiv::make(rc.tile_w);
    AuxDev a{out->normal, out->depth, out->object_id, out->material};
    DeviceBuffer d_normal, d_depth, d_obj, d_mat;
    const bool host = out->memory == VRJ_MEM_HOST;
    if (host) { // the kernel writes device buffers, copied back below
        if (a.normal) {
            VRJ_CUDA(d_normal.alloc(npix * 24));
            a.normal = d_normal.as<double>();
        }
        if (a.depth) {
            VRJ_CUDA(d_depth.alloc(npix * 8));
            a.depth = d_depth.as<double>();
        }
        if (a.object_id) {
            VRJ_CUDA(d_obj.alloc(npix * 4));
            a.object_id = d_obj.as<int32_t>();
        }
        if (a.material) {
            VRJ_CUDA(d_mat.alloc(npix * 4));
            a.material = d_mat.as<int32_t>();
        }
    }
    CallStream cs;
    VRJ_CUDA(cs.create());
    VRJ_CUDA(cudaEventRecord(cs.e0, cs.s));
    k_aux<float><<<(unsigned)((npix + 127) / 128), 128, 0, cs.s>>>(scene->dev, rc, a);
    VRJ_CUDA(cudaGetLastError());
    VRJ_CUDA(cudaEventRecord(cs.e1, cs.s));
    if (host) {
        if (out->normal) VRJ_CUDA(cudaMemcpyAsync(out->normal, a.normal, npix * 24, cudaMemcpyDeviceToHost, cs.s));
        if (out->depth) VRJ_CUDA(cudaMemcpyAsync(out->depth, a.depth, npix * 8, cudaMemcpyDeviceToHost, cs.s));
        if (out->object_id) VRJ_CUDA(cudaMemcpyAsync(out->object_id, a.object_id, npix * 4, cudaMemcpyDeviceToHost, cs.s));
        if (out->material) VRJ_CUDA(cudaMemcpyAsync(out->material, a.material, npix * 4, cudaMemcpyDeviceToHost, cs.s));
    }
    VRJ_CUDA(cudaStreamSynchronize(cs.s));
    float ms = 0.f;
    VRJ_CUDA(cudaEventElapsedTime(&ms, cs.e0, cs.e1));
    if (out->stats) out->stats->primary_rays = npix * p->spp, out->stats->kernel_launches = 1, out->stats->device_ms = ms;
    return VRJ_OK;
}

// The variance-guided a-trous filter (the header states it; vrj_denoise.cuh): k_denoise_init forms (c, var) per pixel,
// `iterations` launches of k_denoise_step ping-pong two pooled buffers of 32 bytes per pixel, k_denoise_colour writes the last
// one out and k_tone_map makes the optional preview.  Host-memory inputs go through pooled device copies.
VrjStatus vrj_denoise(int32_t device, uint32_t memory, uint64_t tile_width, uint64_t tile_height, const double *colour_sum,
                      const double *weight, const double *y_sq_sum, const double *normal, const double *depth, const int32_t *material,
                      const VrjDenoiseParams *dp, double *colour, uint8_t *srgb8, double *device_ms) {
    if (!dp) return fail(VRJ_ERR_INVALID_ARGUMENT, "NULL argument");
    if (memory > VRJ_MEM_DEVICE) return fail(VRJ_ERR_INVALID_ARGUMENT, "unknown memory kind");
    if (dp->iterations > 10) return fail(VRJ_ERR_INVALID_ARGUMENT, "iterations must be <= 10");
    if (!(dp->sigma_luminance > 0.0) || !std::isfinite(dp->sigma_luminance)) return fail(VRJ_ERR_INVALID_ARGUMENT, "sigma_luminance must be > 0 and finite");
    if (!(dp->sigma_normal >= 0.0) || !std::isfinite(dp->sigma_normal)) return fail(VRJ_ERR_INVALID_ARGUMENT, "sigma_normal must be >= 0 and finite");
    if (!(dp->sigma_depth > 0.0) || !std::isfinite(dp->sigma_depth)) return fail(VRJ_ERR_INVALID_ARGUMENT, "sigma_depth must be > 0 and finite");
    if (device_ms) *device_ms = 0.0;
    if (tile_width == 0 || tile_height == 0) return VRJ_OK;
    if (!colour_sum || !weight || !y_sq_sum || !normal || !depth || !material || !colour) return fail(VRJ_ERR_INVALID_ARGUMENT, "NULL argument");
    if (tile_width > 0xffffffffull || tile_height > 0xffffffffull || tile_width * tile_height > 0xffffffffull)
        return fail(VRJ_ERR_UNSUPPORTED, "tile larger than 2^32 pixels");
    const uint64_t npix = tile_width * tile_height;
    const uint32_t n32 = (uint32_t)npix;
    DeviceGuard device_guard;
    VRJ_NVTX_RANGE(call_range, "vrj_denoise");
    VRJ_CUDA(cudaSetDevice(device));
    DeviceBuffer ping, d_in[6], d_colour, d_srgb8;
    VRJ_CUDA(ping.alloc(npix * 64));
    double4 *buf[2] = {ping.as<double4>(), ping.as<double4>() + npix};
    const void *src[6] = {colour_sum, weight, y_sq_sum, normal, depth, material};
    const size_t per[6] = {24, 8, 8, 24, 8, 4};
    double *out_colour = colour;
    uint8_t *out_srgb8 = srgb8;
    const bool host = memory == VRJ_MEM_HOST;
    if (host) {
        for (int i = 0; i < 6; i++) VRJ_CUDA(d_in[i].alloc(npix * per[i]));
        VRJ_CUDA(d_colour.alloc(npix * 24));
        out_colour = d_colour.as<double>();
        if (srgb8) {
            VRJ_CUDA(d_srgb8.alloc(npix * 3));
            out_srgb8 = d_srgb8.as<uint8_t>();
        }
    }
    CallStream cs;
    VRJ_CUDA(cs.create());
    if (host) {
        for (int i = 0; i < 6; i++) VRJ_CUDA(cudaMemcpyAsync(d_in[i].p, src[i], npix * per[i], cudaMemcpyHostToDevice, cs.s));
        for (int i = 0; i < 6; i++) src[i] = d_in[i].p;
    }
    const DenoiseGuides g{static_cast<const double *>(src[3]), static_cast<const double *>(src[4]), static_cast<const int32_t *>(src[5])};
    const unsigned blocks = (unsigned)((npix + 255) / 256);
    VRJ_CUDA(cudaEventRecord(cs.e0, cs.s));
    k_denoise_init<<<blocks, 256, 0, cs.s>>>(static_cast<const double *>(src[0]), static_cast<const double *>(src[1]),
                                             static_cast<const double *>(src[2]), n32, buf[0]);
    const uint32_t bx = (uint32_t)((tile_width + 31) / 32), by = (uint32_t)((tile_height + 7) / 8);
    for (uint32_t i = 0; i < dp->iterations; i++)
        k_denoise_step<<<bx * by, 256, 0, cs.s>>>(buf[i & 1], buf[(i + 1) & 1], g, (uint32_t)tile_width, (uint32_t)tile_height, bx,
                                                   1 << i, dp->sigma_luminance, dp->sigma_normal, dp->sigma_depth);
    k_denoise_colour<<<blocks, 256, 0, cs.s>>>(buf[dp->iterations & 1], n32, out_colour);
    if (srgb8) k_tone_map<<<blocks, 256, 0, cs.s>>>(out_colour, out_srgb8, npix, VRJ_TONEMAP_XYZ);
    VRJ_CUDA(cudaGetLastError());
    VRJ_CUDA(cudaEventRecord(cs.e1, cs.s));
    if (host) {
        VRJ_CUDA(cudaMemcpyAsync(colour, out_colour, npix * 24, cudaMemcpyDeviceToHost, cs.s));
        if (srgb8) VRJ_CUDA(cudaMemcpyAsync(srgb8, out_srgb8, npix * 3, cudaMemcpyDeviceToHost, cs.s));
    }
    VRJ_CUDA(cudaStreamSynchronize(cs.s));
    float ms = 0.f;
    VRJ_CUDA(cudaEventElapsedTime(&ms, cs.e0, cs.e1));
    if (device_ms) *device_ms = ms;
    return VRJ_OK;
}

VrjStatus vrj_tone_map(int32_t device, uint32_t memory, uint32_t source, const double *colour, uint64_t n, uint8_t *rgb8) {
    DeviceGuard device_guard;
    if (n && (!colour || !rgb8)) return fail(VRJ_ERR_INVALID_ARGUMENT, "NULL argument");
    if (source > VRJ_TONEMAP_LINEAR_RGB || memory > VRJ_MEM_DEVICE) return fail(VRJ_ERR_INVALID_ARGUMENT, "unknown source / memory");
    if (n == 0) return VRJ_OK;
    VRJ_CUDA(cudaSetDevice(device));
    DeviceBuffer d_in, d_out;
    const double *src = colour;
    unsigned char *dst = rgb8;
    if (memory == VRJ_MEM_HOST) {
        VRJ_CUDA(d_in.alloc(n * 24));
        VRJ_CUDA(d_out.alloc(n * 3));
        VRJ_CUDA(cudaMemcpy(d_in.p, colour, n * 24, cudaMemcpyHostToDevice));
        src = d_in.as<double>(), dst = d_out.as<unsigned char>();
    }
    k_tone_map<<<(unsigned)((n + 255) / 256), 256>>>(src, dst, n, (int)source);
    VRJ_CUDA(cudaGetLastError());
    if (memory == VRJ_MEM_HOST) VRJ_CUDA(cudaMemcpy(rgb8, d_out.p, n * 3, cudaMemcpyDeviceToHost));
    else VRJ_CUDA(cudaDeviceSynchronize());
    return VRJ_OK;
}

VrjStatus vrj_trace_rays(const VrjScene *scene_c, uint64_t n, const double *origins, const double *directions,
                         uint32_t bvh_filter, int32_t *object_id, int32_t *prim_id, double *t, VrjStats *stats) {
    VrjScene *scene = const_cast<VrjScene *>(scene_c);
    if (!scene || (n && (!origins || !directions || !object_id || !prim_id || !t)))
        return fail(VRJ_ERR_INVALID_ARGUMENT, "NULL argument");
    if (bvh_filter > VRJ_FILTER_Q16) return fail(VRJ_ERR_INVALID_ARGUMENT, "unknown bvh_filter");
    if (stats) std::memset(stats, 0, sizeof(VrjStats));
    if (n == 0) return VRJ_OK;
    if (n > 0xfffffff0ull) return fail(VRJ_ERR_UNSUPPORTED, "more than 2^32 rays in one call");
    DeviceGuard device_guard;
    VRJ_CUDA(cudaSetDevice(scene->device));
    DeviceBuffer d_o, d_d, d_obj, d_prim, d_t, d_stats, d_q[3], d_hits, d_tbest, d_list;
    VRJ_CUDA(d_o.alloc(n * 24));
    VRJ_CUDA(d_d.alloc(n * 24));
    VRJ_CUDA(d_obj.alloc(n * 4));
    VRJ_CUDA(d_prim.alloc(n * 4));
    VRJ_CUDA(d_t.alloc(n * 8));
    for (int i = 0; i < 3; i++) VRJ_CUDA(d_q[i].alloc(n * 16));
    VRJ_CUDA(d_hits.alloc(n * 8));
    VRJ_CUDA(d_tbest.alloc(n * 8));
    VRJ_CUDA(d_list.alloc(n * 4));
    // the default filter walks ready-made records, as the render path does (the id gate then tests the kernel that renders)
    const bool records = bvh_filter == VRJ_FILTER_F32 && scene->trace_records && scene->dev.n_bvh_items > 0;
    DeviceBuffer d_recs;
    if (records) VRJ_CUDA(d_recs.alloc(n * sizeof(TraceRec)));
    VRJ_CUDA(d_stats.alloc((ST_COUNT + 1) * sizeof(unsigned long long)));
    cudaStream_t stream;
    VRJ_CUDA(cudaStreamCreateWithFlags(&stream, cudaStreamNonBlocking));
    cudaEvent_t e0, e1;
    cudaEventCreate(&e0), cudaEventCreate(&e1);
    struct Cleanup {
        cudaStream_t s;
        cudaEvent_t a, b;
        // runs before the DeviceBuffers above return to the pool: no kernel or copy may still be using them
        ~Cleanup() { cudaStreamSynchronize(s), cudaStreamDestroy(s), cudaEventDestroy(a), cudaEventDestroy(b); }
    } cleanup{stream, e0, e1};
    VRJ_CUDA(cudaMemcpyAsync(d_o.p, origins, n * 24, cudaMemcpyHostToDevice, stream));
    VRJ_CUDA(cudaMemcpyAsync(d_d.p, directions, n * 24, cudaMemcpyHostToDevice, stream));
    VRJ_CUDA(cudaMemsetAsync(d_stats.p, 0, (ST_COUNT + 1) * sizeof(unsigned long long), stream));
    unsigned long long *dstats = d_stats.as<unsigned long long>();
    uint32_t *d_lcount = reinterpret_cast<uint32_t *>(dstats + ST_COUNT), *d_work = d_lcount + 1;
    PathQueue q{};
    q.q0 = d_q[0].as<double2>(), q.q1 = d_q[1].as<double2>(), q.q2 = d_q[2].as<double2>();
    TraceBuffers tb{d_hits.as<int2>(), d_tbest.as<double>(), d_list.as<uint32_t>(), records ? d_recs.as<TraceRec>() : nullptr};
    const uint32_t n32 = (uint32_t)n;
    int grid_a = (int)std::min<uint64_t>((n + 127) / 128, (uint64_t)scene->sm_count * 16);
    VRJ_CUDA(cudaEventRecord(e0, stream));
    k_stage_ray_list<true><<<grid_a, 128, 0, stream>>>(scene->dev, n32, d_o.as<double>(), d_d.as<double>(), q, tb, d_lcount, dstats);
    uint64_t launches = 2;
    if (scene->dev.n_bvh_items) {
        launches++;
        if (bvh_filter == VRJ_FILTER_F64)
            k_trace<double, double, true><<<persistent_grid(scene, k_trace<double, double, true>), 128, 0, stream>>>(scene->dev, q, tb, d_lcount, d_work, dstats, nullptr);
        else if (bvh_filter == VRJ_FILTER_F32X4)
            k_trace4<true, false><<<persistent_grid(scene, k_trace4<true, false>), 128, 0, stream>>>(scene->dev, RenderConst{}, q, tb, d_lcount, d_work, dstats, nullptr);
        else if (bvh_filter == VRJ_FILTER_Q16)
            k_traceq<true, false><<<persistent_grid(scene, k_traceq<true, false>), 128, 0, stream>>>(scene->dev, RenderConst{}, q, tb, d_lcount, d_work, dstats, nullptr);
        else if (records)
            k_trace_rec<true><<<persistent_grid(scene, k_trace_rec<true>), 128, 0, stream>>>(scene->dev, tb, d_lcount, d_work, dstats, nullptr);
        else
            k_trace<float, double, true><<<persistent_grid(scene, k_trace<float, double, true>), 128, 0, stream>>>(scene->dev, q, tb, d_lcount, d_work, dstats, nullptr);
    }
    k_hit_ids<<<(n32 + 255) / 256, 256, 0, stream>>>(scene->dev, n32, tb, d_obj.as<int32_t>(), d_prim.as<int32_t>(), d_t.as<double>(), dstats);
    VRJ_CUDA(cudaGetLastError());
    VRJ_CUDA(cudaEventRecord(e1, stream));
    VRJ_CUDA(cudaMemcpyAsync(object_id, d_obj.p, n * 4, cudaMemcpyDeviceToHost, stream));
    VRJ_CUDA(cudaMemcpyAsync(prim_id, d_prim.p, n * 4, cudaMemcpyDeviceToHost, stream));
    VRJ_CUDA(cudaMemcpyAsync(t, d_t.p, n * 8, cudaMemcpyDeviceToHost, stream));
    unsigned long long hstats[ST_COUNT];
    VRJ_CUDA(cudaMemcpyAsync(hstats, d_stats.p, sizeof hstats, cudaMemcpyDeviceToHost, stream));
    VRJ_CUDA(cudaStreamSynchronize(stream));
    float ms = 0.f;
    VRJ_CUDA(cudaEventElapsedTime(&ms, e0, e1));
    if (stats) fill_stats(stats, hstats, launches, ms);
    return VRJ_OK;
}


// ------------------------------------------------------------------------------------------------
// Single-process multi-GPU: sample-index sharding + one NCCL reduce (SURVEY 8e)
} // extern "C"

namespace {
// the few NCCL entry points used, resolved from libnccl.so.2 at run time (ABI-stable across 2.x)
typedef void *nccl_comm_t;
struct NcclApi {
    void *lib = nullptr;
    int (*CommInitAll)(nccl_comm_t *, int, const int *) = nullptr;
    int (*CommDestroy)(nccl_comm_t) = nullptr;
    int (*GroupStart)() = nullptr;
    int (*GroupEnd)() = nullptr;
    int (*Reduce)(const void *, void *, size_t, int, int, int, nccl_comm_t, cudaStream_t) = nullptr;
    const char *(*GetErrorString)(int) = nullptr;
    bool load() {
        if (lib) return true;
        for (const char *name : {"libnccl.so.2", "libnccl.so"}) {
            lib = dlopen(name, RTLD_NOW | RTLD_GLOBAL);
            if (lib) break;
        }
        if (!lib) return false;
        CommInitAll = reinterpret_cast<decltype(CommInitAll)>(dlsym(lib, "ncclCommInitAll"));
        CommDestroy = reinterpret_cast<decltype(CommDestroy)>(dlsym(lib, "ncclCommDestroy"));
        GroupStart = reinterpret_cast<decltype(GroupStart)>(dlsym(lib, "ncclGroupStart"));
        GroupEnd = reinterpret_cast<decltype(GroupEnd)>(dlsym(lib, "ncclGroupEnd"));
        Reduce = reinterpret_cast<decltype(Reduce)>(dlsym(lib, "ncclReduce"));
        GetErrorString = reinterpret_cast<decltype(GetErrorString)>(dlsym(lib, "ncclGetErrorString"));
        return CommInitAll && CommDestroy && GroupStart && GroupEnd && Reduce && GetErrorString;
    }
};
NcclApi g_nccl;
const int kNcclDouble = 8, kNcclSum = 0; // nccl.h: ncclFloat64 = 8, ncclSum = 0

} // namespace

struct VrjComm {
    std::vector<int> devices;
    std::vector<nccl_comm_t> comms;
    std::vector<cudaStream_t> streams;
};
struct VrjMultiScene {
    VrjComm *comm = nullptr;
    std::vector<VrjScene *> scenes;
    std::vector<DeviceBuffer *> sum, weight; // per device
    DeviceBuffer colour;                      // on devices[0]
    size_t npix = 0;
};

extern "C" {

VrjStatus vrj_comm_create(int32_t n, const int32_t *devices, VrjComm **out) {
    if (!out || n < 1 || !devices) return fail(VRJ_ERR_INVALID_ARGUMENT, "vrj_comm_create: bad arguments");
    *out = nullptr;
    if (!g_nccl.load()) return fail(VRJ_ERR_UNSUPPORTED, "NCCL (libnccl.so.2) could not be loaded");
    DeviceGuard device_guard;
    VrjComm *c = new VrjComm();
    c->devices.assign(devices, devices + n);
    c->comms.assign(n, nullptr);
    int rc = g_nccl.CommInitAll(c->comms.data(), n, c->devices.data());
    if (rc != 0) {
        std::string msg = std::string("ncclCommInitAll: ") + g_nccl.GetErrorString(rc);
        delete c;
        return fail(VRJ_ERR_CUDA, msg);
    }
    for (int i = 0; i < n; i++) {
        cudaStream_t st = nullptr;
        if (cudaSetDevice(c->devices[i]) != cudaSuccess || cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking) != cudaSuccess) {
            vrj_comm_destroy(c);
            return fail(VRJ_ERR_CUDA, "vrj_comm_create: cannot create a stream on every device");
        }
        c->streams.push_back(st);
    }
    *out = c;
    return VRJ_OK;
}

void vrj_comm_destroy(VrjComm *c) {
    if (!c) return;
    DeviceGuard device_guard;
    for (size_t i = 0; i < c->streams.size(); i++) {
        cudaSetDevice(c->devices[i]);
        cudaStreamDestroy(c->streams[i]);
    }
    for (nccl_comm_t k : c->comms)
        if (k) g_nccl.CommDestroy(k);
    delete c;
}

void vrj_comm_scene_destroy(VrjMultiScene *m) {
    if (!m) return;
    DeviceGuard device_guard;
    for (size_t i = 0; i < m->scenes.size(); i++) {
        cudaSetDevice(m->comm->devices[i]);
        vrj_scene_destroy(m->scenes[i]);
        if (i < m->sum.size()) delete m->sum[i];
        if (i < m->weight.size()) delete m->weight[i];
    }
    cudaSetDevice(m->comm->devices[0]);
    delete m;
}

VrjStatus vrj_comm_scene_create(VrjComm *c, const VrjSceneDesc *desc, VrjMultiScene **out) {
    if (!c || !out) return fail(VRJ_ERR_INVALID_ARGUMENT, "vrj_comm_scene_create: NULL argument");
    *out = nullptr;
    VrjMultiScene *m = new VrjMultiScene();
    m->comm = c;
    // one thread per GPU: every device has its own staging block, preparation stream and lock, so the replicas upload and
    // build side by side
    const size_t n = c->devices.size();
    std::vector<VrjScene *> scenes(n, nullptr);
    std::vector<VrjStatus> status(n, VRJ_OK);
    std::vector<std::string> errors(n);
    std::vector<std::thread> workers;
    for (size_t i = 0; i < n; i++)
        workers.emplace_back([&, i] {
            status[i] = vrj_scene_create(desc, c->devices[i], &scenes[i]);
            if (status[i] != VRJ_OK) errors[i] = g_error; // the message is thread-local
        });
    for (auto &w : workers) w.join();
    for (size_t i = 0; i < n; i++) {
        m->scenes.push_back(scenes[i]);
        m->sum.push_back(new DeviceBuffer());
        m->weight.push_back(new DeviceBuffer());
    }
    for (size_t i = 0; i < n; i++)
        if (status[i] != VRJ_OK) {
            vrj_comm_scene_destroy(m);
            return fail(status[i], errors[i]);
        }
    *out = m;
    return VRJ_OK;
}

VrjStatus vrj_render_sharded(VrjMultiScene *m, const VrjTile *tile, uint64_t height, uint64_t width, const VrjRenderParams *p,
                             VrjAccumOut *out) {
    if (!m || !tile || !p || !out) return fail(VRJ_ERR_INVALID_ARGUMENT, "NULL argument");
    if (p->sample_stride > 1) return fail(VRJ_ERR_INVALID_ARGUMENT, "vrj_render_sharded shards the samples itself: sample_stride must be 0 or 1");
    if (out->accumulate || out->photons) return fail(VRJ_ERR_UNSUPPORTED, "vrj_render_sharded: accumulate / photons are not supported");
    if (tile->end_column < tile->start_column || tile->end_row < tile->start_row) return fail(VRJ_ERR_INVALID_ARGUMENT, "bad tile");
    VrjComm *c = m->comm;
    const int G = (int)c->devices.size();
    DeviceGuard device_guard;
    const size_t npix = (size_t)(tile->end_column - tile->start_column) * (tile->end_row - tile->start_row);
    if (out->stats) std::memset(out->stats, 0, sizeof(VrjStats));
    if (npix == 0 || p->spp == 0) return VRJ_OK;
    for (int g = 0; g < G; g++) {
        VRJ_CUDA(cudaSetDevice(c->devices[g]));
        if (m->sum[g]->bytes < npix * 24) {
            m->sum[g]->release();
            m->weight[g]->release();
            VRJ_CUDA(m->sum[g]->alloc(npix * 24));
            VRJ_CUDA(m->weight[g]->alloc(npix * 8));
        }
    }
    VRJ_CUDA(cudaSetDevice(c->devices[0]));
    if (m->colour.bytes < npix * 24) {
        m->colour.release();
        VRJ_CUDA(m->colour.alloc(npix * 24));
    }
    // ---- every device renders its share of the sample indices into its own device buffers ----
    std::vector<VrjStatus> status(G, VRJ_OK);
    std::vector<std::string> messages(G);
    std::vector<VrjStats> stats(G);
    std::vector<std::thread> threads;
    for (int g = 0; g < G; g++) {
        threads.emplace_back([&, g]() {
            VrjRenderParams q = *p;
            q.spp = p->spp > (uint32_t)g ? (p->spp - (uint32_t)g + (uint32_t)G - 1) / (uint32_t)G : 0; // samples g, g+G, ...
            q.sample_offset = p->sample_offset + (uint64_t)g;
            q.sample_stride = (uint32_t)G;
            VrjAccumOut o{};
            o.memory = VRJ_MEM_DEVICE;
            o.colour_sum = m->sum[g]->as<double>(), o.weight = m->weight[g]->as<double>();
            o.stats = &stats[g];
            std::memset(&stats[g], 0, sizeof(VrjStats));
            if (q.spp == 0) {
                cudaSetDevice(c->devices[g]);
                cudaMemset(m->sum[g]->p, 0, npix * 24);
                cudaMemset(m->weight[g]->p, 0, npix * 8);
                return;
            }
            status[g] = vrj_render_tile(m->scenes[g], tile, height, width, &q, &o);
            if (status[g] != VRJ_OK) messages[g] = vrj_last_error();
        });
    }
    for (auto &t : threads) t.join();
    for (int g = 0; g < G; g++)
        if (status[g] != VRJ_OK) return fail(status[g], "device " + std::to_string(c->devices[g]) + ": " + messages[g]);
    // ---- the one exchange step: ncclReduce(sum) of (sum XYZ, weight) into devices[0] ----
    if (G > 1) {
        int rc = g_nccl.GroupStart();
        for (int g = 0; g < G && rc == 0; g++) {
            cudaSetDevice(c->devices[g]);
            rc = g_nccl.Reduce(m->sum[g]->p, m->sum[g]->p, npix * 3, kNcclDouble, kNcclSum, 0, c->comms[g], c->streams[g]);
            if (rc == 0) rc = g_nccl.Reduce(m->weight[g]->p, m->weight[g]->p, npix, kNcclDouble, kNcclSum, 0, c->comms[g], c->streams[g]);
        }
        int rc2 = g_nccl.GroupEnd();
        if (rc != 0 || rc2 != 0) return fail(VRJ_ERR_CUDA, std::string("ncclReduce: ") + g_nccl.GetErrorString(rc ? rc : rc2));
        for (int g = 0; g < G; g++) {
            VRJ_CUDA(cudaSetDevice(c->devices[g]));
            VRJ_CUDA(cudaStreamSynchronize(c->streams[g]));
        }
    }
    VRJ_CUDA(cudaSetDevice(c->devices[0]));
    cudaStream_t s0 = c->streams[0];
    k_finalize<<<(unsigned)((npix + 255) / 256), 256, 0, s0>>>(m->sum[0]->as<double>(), m->weight[0]->as<double>(), m->colour.as<double>(), (uint32_t)npix);
    VRJ_CUDA(cudaGetLastError());
    const cudaMemcpyKind kind = out->memory == VRJ_MEM_DEVICE ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost;
    if (out->colour) VRJ_CUDA(cudaMemcpyAsync(out->colour, m->colour.p, npix * 24, kind, s0));
    if (out->colour_sum) VRJ_CUDA(cudaMemcpyAsync(out->colour_sum, m->sum[0]->p, npix * 24, kind, s0));
    if (out->weight) VRJ_CUDA(cudaMemcpyAsync(out->weight, m->weight[0]->p, npix * 8, kind, s0));
    DeviceBuffer srgb8;
    if (out->srgb8) {
        VRJ_CUDA(srgb8.alloc(npix * 3));
        k_tone_map<<<(unsigned)((npix + 255) / 256), 256, 0, s0>>>(m->colour.as<double>(), srgb8.as<unsigned char>(), npix, 0);
        VRJ_CUDA(cudaMemcpyAsync(out->srgb8, srgb8.p, npix * 3, kind, s0));
    }
    if (out->memory == VRJ_MEM_DEVICE) {
        if (out->colour_bias) VRJ_CUDA(cudaMemsetAsync(out->colour_bias, 0, npix * 24, s0));
        if (out->weight_bias) VRJ_CUDA(cudaMemsetAsync(out->weight_bias, 0, npix * 8, s0));
    } else {
        if (out->colour_bias) std::memset(out->colour_bias, 0, npix * 24);
        if (out->weight_bias) std::memset(out->weight_bias, 0, npix * 8);
    }
    VRJ_CUDA(cudaStreamSynchronize(s0));
    if (out->stats) {
        VrjStats &t = *out->stats;
        for (int g = 0; g < G; g++) {
            const VrjStats &a = stats[g];
            t.primary_rays += a.primary_rays, t.bounce_rays += a.bounce_rays, t.shadow_rays += a.shadow_rays;
            t.paths_missed += a.paths_missed, t.paths_escaped += a.paths_escaped, t.paths_depth_limited += a.paths_depth_limited;
            t.node_visits += a.node_visits, t.triangle_tests += a.triangle_tests, t.kernel_launches += a.kernel_launches;
            t.staged_rays += a.staged_rays;
            t.device_ms = std::max(t.device_ms, a.device_ms); // devices run concurrently
            t.primary_ms = std::max(t.primary_ms, a.primary_ms), t.bounce_ms = std::max(t.bounce_ms, a.bounce_ms);
            t.shade_ms = std::max(t.shade_ms, a.shade_ms), t.resolve_ms = std::max(t.resolve_ms, a.resolve_ms);
        }
        t.kernel_launches += 1;
    }
    return VRJ_OK;
}

} // extern "C"
