// bmo_host.cuh -- host-side state of libbmo.so: context, uploaded system, result tables, error
// handling and the BVH builder.  Shared by bmo_trace.cu and bmo_detector.cu.
#pragma once
#include <algorithm>
#include <cstdio>
#include <cstring>
#include <map>
#include <mutex>
#include <string>
#include <utility>
#include <vector>
#include <nvtx3/nvToolsExt.h>
#include "bmo_geom.cuh"

namespace bmo {

extern thread_local std::string g_last_error;
inline int32_t fail(int32_t code, const std::string& msg) { g_last_error = msg; return code; }

#define BMO_CUDA(call)                                                                              \
    do {                                                                                            \
        cudaError_t e_ = (call);                                                                    \
        if (e_ != cudaSuccess)                                                                      \
            return fail(BMO_ECUDA, std::string(#call) + ": " + cudaGetErrorString(e_) + " @" + __FILE__ + ":" + std::to_string(__LINE__)); \
    } while (0)

// NVTX range around a C-ABI call (header-only nvtx3: a no-op unless a profiler has injected itself)
struct NvtxRange {
    explicit NvtxRange(const char* name) { nvtxRangePushA(name); }
    ~NvtxRange() { nvtxRangePop(); }
    NvtxRange(const NvtxRange&) = delete;
    NvtxRange& operator=(const NvtxRange&) = delete;
};

// bad_ids: rays whose lambda_id / pose_id was out of range (init_queue, solve_rays_persistent).
// tiles, most_nseg: per-call words of solve_rays_persistent (zeroed by every such call): next tile of rays, largest nseg of a ray.
struct DevCounters { unsigned long long interactions, sdf, tri, bad_ids, tiles, most_nseg; };

}  // namespace bmo

struct bmo_ctx {
    int device = 0;
    cudaStream_t stream = nullptr;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr, evk0 = nullptr, evk1 = nullptr, evs0 = nullptr, evs1 = nullptr;
    std::vector<cudaEvent_t> ev_pool;        // 10 events per sub-batch slot
    std::vector<cudaStream_t> aux_streams;   // streams of the sub-batches of a pipelined trace call (created on demand)
    double k1_ms = 0, k3_ms = 0, k3_bytes = 0, k4_ms = 0;  // accumulated device time of trace_step / scatter_queue / pd_field
    int64_t k1_launches = 0, interactions_seen = 0, bad_ids_seen = 0;
    bmo::DevCounters* d_counters = nullptr;
    long long* d_totals = nullptr;   // [4] scratch for scans
    long long* h_totals = nullptr;   // pinned, 8 entries for the scans + 8 per sub-batch slot + the device counters (72..77)
    int64_t waves = 0, launches = 0, px_beamlets = 0, psf_pairs = 0;
    double psf_ms = 0;
    double trace_ms = 0, pd_ms = 0;
    int64_t pool_slack = 0;   // bytes by which bmo_retrace has grown the stream-ordered pool beyond its own needs (see there)
    int sm_count = 148;
    // solve_rays_persistent (bmo_trace.cu: persistent_blocks): the variant and table size last sized, its resident blocks per SM
    const void* persist_fn = nullptr;
    size_t persist_smem = 0;
    int persist_blocks = 0;
};

struct bmo_sys {
    bmo_ctx* ctx = nullptr;
    bmo::SysView view{};         // device pointers
    // host copies (needed for pose updates and detector metadata)
    std::vector<bmo_prim> prims;
    std::vector<bmo_part> parts;
    std::vector<bmo_object> objects;
    std::vector<bmo::MeshView> meshes;
    std::vector<double> lambdas;
    int64_t n_vertices = 0, n_faces = 0;
    bool has_rare = false;       // some primitive is a cylindrical / aspheric surface: the trace kernels compiled with them are used
    bool all_lean = false;       // every SDF part is a union of <= 4 plain primitives and no mesh has a BVH: the LEAN trace kernels are used
    // owned device buffers
    bmo_prim* d_prims = nullptr; bmo_part* d_parts = nullptr; bmo_object* d_objects = nullptr;
    bmo::MeshView* d_meshes = nullptr; double* d_vertices = nullptr; int32_t* d_faces = nullptr;
    bmo::BvhNode* d_nodes = nullptr; int32_t* d_bvh_faces = nullptr; double* d_ntable = nullptr;
    double* d_bounds = nullptr; double* d_detpose = nullptr; double* d_lambdas = nullptr; double* d_jones = nullptr; double* d_ext = nullptr;
    // pose-0 copies to restore after a sweep
    std::vector<double> h_vertices, h_bounds, h_detpose;
    // K5 (bmo_pose.cu): kinematic tree + the uploaded tables every pose starts from
    std::vector<bmo_kin_node> kin_nodes;
    bmo_kin_node* d_kin_nodes = nullptr; double* d_prim_bounds = nullptr;
    bmo_prim* d_prims0 = nullptr; double* d_vertices0 = nullptr; double* d_detpose0 = nullptr;
    // high-water marks of earlier branching traces, keyed by (mode, root beams): queue units, beams and scratch
    // units the call ended with.  The next call of the same shape allocates them up front (no growth copies,
    // identical request sizes for the pool).
    // first_chunk (splitter-free systems): waves to enqueue before the first look at the device -- 1 until a call of this
    // shape has shown that (almost) nobody dies on the first wave, then 4 (no early compaction decision to take).
    struct TraceHint { int64_t slots = 0, beams = 0, scr = 0; int first_chunk = 1; };
    std::map<std::pair<int, int64_t>, TraceHint> hints;
};

// One wave of segment records (wave-major), gathered into beam-major order at the end of a trace.
struct WaveBuf {
    double* d = nullptr;    // [nsd][count]
    int32_t* part = nullptr;
    int32_t* beam = nullptr;
    int32_t* seg = nullptr;
    int64_t count = 0;      // rays in this wave
};

struct bmo_result {
    bmo_sys* sys = nullptr;   // system the result was traced through (may be freed before the result: never dereferenced after the trace)
    bmo_ctx* ctx = nullptr;
    std::vector<int32_t> part_object;   // part -> object of that system (segment export, structure check of bmo_retrace)
    std::vector<int32_t> object_kind;   // bmo_obj_kind of every object of that system (bmo_spot_stats checks its detector)
    int32_t n_objects = 0;
    int32_t n_poses = 1;    // poses of that system at trace time (bmo_spot_stats_poses checks its argument against it)
    int mode = 0;           // 0 ray, 1 polarized ray, 2 gaussian beamlet
    int R = 1;              // rays per beam
    int nsd = 12;           // doubles per segment record
    int64_t n_roots = 0, n_beams = 0, n_segments = 0, interactions = 0;
    int32_t waves = 0;
    bool keep = false;
    // per-beam tables (device), capacity cap_beams
    int64_t cap_beams = 0;
    void* beam_slab = nullptr;    // splitter-free traces: the per-beam tables below are carved out of one allocation
    int32_t *parent = nullptr, *slot = nullptr, *nseg = nullptr, *status = nullptr, *lam = nullptr, *pose = nullptr;
    double *w0 = nullptr, *e0 = nullptr, *plen = nullptr, *popl = nullptr;
    int32_t* spot_obj = nullptr;  // [cap_beams * R]
    double* spot_xz = nullptr;    // [cap_beams * R * 2]
    long long* first_seg = nullptr;  // [n_beams + 1] after finalisation
    // beam-major segment table (device): rows = n_segments * R
    double* seg_d = nullptr;      // [rows][nsd]: one record per row
    int32_t* seg_part = nullptr;  // [rows]
    int64_t seg_rows = 0;
    std::vector<WaveBuf> wavebufs;
};

namespace bmo {

// ---- BVH (host build, median split on the longest centroid axis, <= 4 faces per leaf) ---------
struct BvhBuild {
    std::vector<BvhNode> nodes;
    std::vector<int32_t> order;
};
inline void bvh_build(const double* verts, const int32_t* faces, int64_t nf, BvhBuild& out) {
    out.nodes.clear();
    out.order.resize(nf);
    for (int64_t i = 0; i < nf; i++) out.order[i] = (int32_t)i;
    std::vector<double> cen(3 * nf), lo(3 * nf), hi(3 * nf);
    double glo[3] = {1e300, 1e300, 1e300}, ghi[3] = {-1e300, -1e300, -1e300};
    for (int64_t f = 0; f < nf; f++)
        for (int k = 0; k < 3; k++) {
            double a = verts[3 * faces[3 * f] + k], b = verts[3 * faces[3 * f + 1] + k], c = verts[3 * faces[3 * f + 2] + k];
            lo[3 * f + k] = std::min(a, std::min(b, c));
            hi[3 * f + k] = std::max(a, std::max(b, c));
            cen[3 * f + k] = (a + b + c) / 3;
            glo[k] = std::min(glo[k], lo[3 * f + k]);
            ghi[k] = std::max(ghi[k], hi[3 * f + k]);
        }
    // Moeller-Trumbore accepts (u, v) up to 1e-9 outside the triangle and the slab test rounds:
    // inflate every box by a margin far above both (SURVEY hard part 11).
    double diag = 0;
    for (int k = 0; k < 3; k++) diag = std::max(diag, ghi[k] - glo[k]);
    const double pad = 1e-6 * diag + 1e-12;
    struct Item { int64_t b, e; int32_t node; };
    std::vector<Item> stack;
    out.nodes.push_back(BvhNode{});
    stack.push_back({0, nf, 0});
    while (!stack.empty()) {
        Item it = stack.back(); stack.pop_back();
        BvhNode nd{};
        double clo[3] = {1e300, 1e300, 1e300}, chi[3] = {-1e300, -1e300, -1e300};
        for (int k = 0; k < 3; k++) { nd.lo[k] = 1e300; nd.hi[k] = -1e300; }
        for (int64_t i = it.b; i < it.e; i++) {
            int32_t f = out.order[i];
            for (int k = 0; k < 3; k++) {
                nd.lo[k] = std::min(nd.lo[k], lo[3 * f + k]); nd.hi[k] = std::max(nd.hi[k], hi[3 * f + k]);
                clo[k] = std::min(clo[k], cen[3 * f + k]); chi[k] = std::max(chi[k], cen[3 * f + k]);
            }
        }
        for (int k = 0; k < 3; k++) { nd.lo[k] -= pad; nd.hi[k] += pad; }
        int64_t cnt = it.e - it.b;
        int ax = 0;
        for (int k = 1; k < 3; k++) if (chi[k] - clo[k] > chi[ax] - clo[ax]) ax = k;
        if (cnt <= 4 || !(chi[ax] - clo[ax] > 0)) {
            nd.first = (int32_t)it.b; nd.count = (int32_t)cnt; nd.left = nd.right = -1;
            // keep the reference's face order inside a leaf
            std::sort(out.order.begin() + it.b, out.order.begin() + it.e);
            out.nodes[it.node] = nd;
            continue;
        }
        int64_t mid = (it.b + it.e) / 2;
        std::nth_element(out.order.begin() + it.b, out.order.begin() + mid, out.order.begin() + it.e,
                         [&](int32_t a, int32_t b) { return cen[3 * a + ax] < cen[3 * b + ax]; });
        nd.count = 0; nd.first = 0;
        nd.left = (int32_t)out.nodes.size(); out.nodes.push_back(BvhNode{});
        nd.right = (int32_t)out.nodes.size(); out.nodes.push_back(BvhNode{});
        out.nodes[it.node] = nd;
        stack.push_back({it.b, mid, nd.left});
        stack.push_back({mid, it.e, nd.right});
    }
}

// Stream-ordered allocation from the device's pool (release threshold = infinity, bmo_init).  Large requests
// are rounded up to size classes (8 per octave, <= 12.5 % slack): the wave loop of a branching trace asks for
// slightly different sizes on every call, and a pool that only holds blocks of other sizes has to map new
// physical memory, which blocks the host for milliseconds per gigabyte.
inline size_t size_class(size_t bytes) {
    if (bytes < (size_t)1 << 16) return bytes;
    int lg = 63 - __builtin_clzll((unsigned long long)bytes);
    const size_t step = (size_t)1 << (lg - 3);
    return (bytes + step - 1) & ~(step - 1);
}
// Blocks of 64 MiB and more (wave buffers and segment tables of large traces, queues of 10^7 rays) bypass the driver's pool:
// a pool that holds free blocks of other sizes satisfies a 25 GB request by remapping physical memory, which costs ~6 ms per
// gigabyte on every call (C4 with its segment table kept: 140 of 200 ms).  They are cudaMalloc'ed once and parked in a
// per-device free list when released; a request takes the smallest parked block that is large enough (and at most 25 % larger)
// and was released on the same stream (so that reuse is ordered behind the last user without an event).
struct BigBlocks {
    struct Blk { void* p; size_t bytes; cudaStream_t stream; };
    std::vector<Blk> parked;
    std::map<void*, size_t> live;
    std::mutex mu;   // contexts of the same device may live on different host threads
    static constexpr size_t kMin = (size_t)64 << 20;
    static BigBlocks& of_device() {
        static BigBlocks per_dev[64];
        int d = 0;
        cudaGetDevice(&d);
        return per_dev[d & 63];
    }
    size_t drop_parked() {
        std::lock_guard<std::mutex> g(mu);
        return drop_parked_locked();
    }
    size_t drop_parked_locked() {
        size_t bytes = 0;
        for (auto& b : parked) { bytes += b.bytes; cudaFree(b.p); }
        parked.clear();
        return bytes;
    }
    cudaError_t get(void** out, size_t bytes, cudaStream_t s) {
        std::lock_guard<std::mutex> g(mu);
        size_t best = parked.size();
        for (size_t i = 0; i < parked.size(); i++)
            if (parked[i].stream == s && parked[i].bytes >= bytes && parked[i].bytes <= bytes + bytes / 4 &&
                (best == parked.size() || parked[i].bytes < parked[best].bytes)) best = i;
        if (best < parked.size()) {
            *out = parked[best].p;
            live[*out] = parked[best].bytes;
            parked.erase(parked.begin() + best);
            return cudaSuccess;
        }
        cudaError_t e = cudaMalloc(out, bytes);
        if (e != cudaSuccess) {          // make room: parked blocks of other sizes, then whatever the stream-ordered pool caches
            cudaGetLastError();
            drop_parked_locked();
            int d = 0; cudaGetDevice(&d);
            cudaMemPool_t pool;
            if (cudaDeviceGetDefaultMemPool(&pool, d) == cudaSuccess) { cudaDeviceSynchronize(); cudaMemPoolTrimTo(pool, 0); }
            e = cudaMalloc(out, bytes);
        }
        if (e == cudaSuccess) live[*out] = bytes;
        return e;
    }
    bool put(void* p, cudaStream_t s) {
        std::lock_guard<std::mutex> g(mu);
        auto it = live.find(p);
        if (it == live.end()) return false;
        parked.push_back({p, it->second, s});
        live.erase(it);
        return true;
    }
};
template <class T> inline cudaError_t dev_alloc(T** p, size_t n, cudaStream_t s) {
    const size_t bytes = size_class(std::max<size_t>(n, 1) * sizeof(T));
    if (bytes >= BigBlocks::kMin) return BigBlocks::of_device().get((void**)p, bytes, s);
    return cudaMallocAsync((void**)p, bytes, s);
}
template <class T> inline void dev_free(T*& p, cudaStream_t s) {
    if (p && !BigBlocks::of_device().put((void*)p, s)) cudaFreeAsync((void*)p, s);
    p = nullptr;
}

}  // namespace bmo
