// bmo_trace.cu -- wavefront tracer (sm_100a) and the C ABI around it.
//
// One wave = one `tracing_step!` + `interact3d` of every live beam (System.jl:100-154, 274-318).
// Kernels per wave:
//   K1 intersect_wave     one thread per ray: trace_one / trace_all (SDF sphere tracing, Moeller-
//                         Trumbore behind the BVH) -> hit record (t, normal, part).  Two builds: LEAN (lens-stack systems:
//                         unions of <= 4 plain primitives, no BVH mesh; tracing_step_lean of bmo_lean.cuh with its cold state
//                         in shared-memory columns, 64 registers, 8 blocks per SM) and the general one (72-80 registers).
//                         Bound by the issue rate of its non-FP64 instructions (profiles/r02_k1_instruction_buckets.txt).
//   K2 interact_wave<MODE, NS> one thread per ray (Gaussian beamlets: chief/waist/divergence in adjacent
//                         lanes, 10 triples per warp): interact3d; the continuing ray overwrites its own queue
//                         slot, a dead one is flagged.  Systems with beamsplitters (NS = false): the children go
//                         to a scratch area in queue order (warp ballots + prefix sums), scan_counts + spawn_children
//                         number them deterministically and append the reflected ones to the queue.
//   K1+K2 fused_wave0     plain rays through a splitter-free system, all waves of a chunk in one launch: every wave of a
//                         pipelined host-input call with plain rays, where the number of launches is what limits.
//   K1r retrace_intersect_wave   K1 of a retrace call (stored path re-validated per beam).
//   K3 compact_fused      queue compaction in one cooperative launch once the dead slots are the majority.
// Plain rays through a splitter-free LEAN system whose segments are not kept need no waves at all: solve_rays_persistent
// carries every ray from the caller's inputs to its last interaction in one launch.
// With BMO_KEEP_SEGMENTS the segment records are written wave-major by K2 and gathered into
// beam-major row records at the end (gather_segments, a warp-level transposition through shared memory).
#include <chrono>
#include <cstdlib>
#include <cooperative_groups.h>
#include <type_traits>
#include "bmo_host.cuh"
#include "bmo_interact.cuh"
#include "bmo_lean.cuh"

namespace bmo {
thread_local std::string g_last_error;

// ---- queue layout -------------------------------------------------------------------------------
// double fields (SoA, stride = capacity): px py pz dx dy dz n | E0 re/im x3 (polarized) |
//                                         lsum lpar oplpar (gaussian chief accumulators)
enum { F_PX = 0, F_PY, F_PZ, F_DX, F_DY, F_DZ, F_N, F_X0 };
// int fields: lambda id, hinted part, beam (-1 = dead slot), segment index, pose, retrace cursor (beam of
// the previous solution whose stored path this beam re-validates, -1 = not retracing)
enum { I_LAM = 0, I_HINT, I_BEAM, I_SEG, I_POSE, I_RETR, NI_Q, I_PUNIT = NI_Q, NI_S };   // I_PUNIT (scratch only): queue unit of the parent
// segment record rows
enum { S_PX = 0, S_PY, S_PZ, S_DX, S_DY, S_DZ, S_N, S_T, S_NX, S_NY, S_NZ, S_E0 };

struct Queue {
    double* d = nullptr;
    int32_t* i = nullptr;
    int64_t cap = 0;  // rays
};

inline int nf_queue(int mode) { return mode == 1 ? 13 : (mode == 2 ? 10 : 7); }
inline int nf_scratch(int mode) { return mode == 2 ? 15 : nf_queue(mode); }
inline int nf_seg(int mode) { return mode == 1 ? 17 : 11; }

struct BeamTab {
    int32_t *parent, *slot, *nseg, *status, *lam, *pose, *spot_obj;
    double *w0, *e0, *plen, *popl, *spot_xz;
};

struct HitBuf {
    double* d = nullptr;      // [4][cap]: t, nx, ny, nz
    int32_t* part = nullptr;  // [cap]: -1 = miss
    int32_t* flag = nullptr;  // [cap], retrace calls only: 0 ordinary tracing_step!, 1 stored path re-validated, 2 path left
    int64_t cap = 0;
};

// Previous solution of the same beams (retrace_system!, System.jl:188-428): what the stored rays hit.
struct RetraceView {
    const int32_t* nseg = nullptr;         // [beams] stored rays per beam
    const long long* first_seg = nullptr;  // [beams] first row of the beam in the beam-major segment table
    const int32_t* seg_part = nullptr;     // [rows * R] part hit by each stored ray (-1: intersection === nothing)
    const int32_t* child = nullptr;        // [beams][2] stored children (transmitted, reflected), -1: none
    const double* w0 = nullptr;            // [beams] stored beamlet waists
    int32_t on = 0, pad = 0;
};

struct IntersectParams {
    SysView S;
    Queue cur;
    HitBuf hit;
    int64_t n_rays;
    int32_t r_max, pad;
    DevCounters* counters;
};

struct StepParams {
    SysView S;
    Queue cur, scr;
    HitBuf hit;
    int64_t count;       // beams in the current queue
    int32_t r_max, keep;
    WaveBuf wave;
    BeamTab B;
    int32_t* blk_cnt;    // [nblocks] spawn events per block
    unsigned long long* wave_totals;   // [2] units alive after this wave, spawn events of this wave
    DevCounters* counters;
    RetraceView rt;
    int32_t n_waves, pad2;   // fused_wave0: waves traced by one launch (the queue is updated in place between them)
};

template <int MODE> struct Cfg {
    static constexpr int R = MODE == 2 ? 3 : 1;
    static constexpr int BLOCK = 128;
    static constexpr int NWARP = BLOCK / 32;
    static constexpr int UNITS = MODE == 2 ? NWARP * 10 : BLOCK;  // beams per block
};

BMO_D unsigned lanemask_lt() { unsigned m; asm("mov.u32 %0, %%lanemask_lt;" : "=r"(m)); return m; }
BMO_D V3 shfl3(V3 v, int l) {
    return mk3(__shfl_sync(0xffffffffu, v.x, l), __shfl_sync(0xffffffffu, v.y, l), __shfl_sync(0xffffffffu, v.z, l));
}

// ---- K1: intersect ------------------------------------------------------------------------------
constexpr int IBLOCK = 128;
// Copies the small system tables into shared memory with the NT threads of the block: prims | parts | bounds, and for the LEAN
// kernels one packed word per part (lean_part_info).  The caller synchronises the block.
template <int NT, bool LEAN>
BMO_D void stage_tables(const SysView& S, unsigned char* smem) {
    const int nw = S.n_prims * (int)(sizeof(bmo_prim) / 8), nq = S.n_parts * (int)(sizeof(bmo_part) / 8);
    const double* src = reinterpret_cast<const double*>(S.prims);
    double* dst = reinterpret_cast<double*>(smem);
    for (int k = threadIdx.x; k < nw; k += NT) dst[k] = src[k];
    src = reinterpret_cast<const double*>(S.parts);
    dst = reinterpret_cast<double*>(smem + (size_t)S.n_prims * sizeof(bmo_prim));
    for (int k = threadIdx.x; k < nq; k += NT) dst[k] = src[k];
    double* s_bounds = reinterpret_cast<double*>(smem + (size_t)S.n_prims * sizeof(bmo_prim) + (size_t)S.n_parts * sizeof(bmo_part));
    for (int k = threadIdx.x; k < NBOUND * S.n_parts; k += NT) s_bounds[k] = S.bounds[k];
    if (LEAN) {
        unsigned long long* s_pinfo = reinterpret_cast<unsigned long long*>(s_bounds + NBOUND * S.n_parts);
        for (int k = threadIdx.x; k < S.n_parts; k += NT) s_pinfo[k] = lean_part_info(S.parts[k], S.objects[S.parts[k].object]);
    }
}
// STAGED: the small system tables (prims, parts, bounds) live in shared memory -- a compile-time fact,
// so that the marching loop reads them with LDS instead of generic loads.
// LEAN: every SDF part is a union of at most 4 plain primitives and every mesh is small (bmo_sys::all_lean): the union loop keeps
// its member bounds in shared memory (LeanBounds, bmo_geom.cuh) and the BVH traversal is compiled out.  LEAN implies STAGED and
// !RK (see k1_config).
// Resident blocks per SM K1 is compiled for (DESIGN §5): 8 for the lean build (64 registers, the fastest of 6 / 7 / 8 on C2),
// 7 for the general staged build (72 registers, the fastest of 4..8 on C2), 6 with the rare primitives, 4 without staged tables.
constexpr int k1_min_blocks(bool staged, bool rk, bool lean) { return !staged ? 4 : lean ? 8 : rk ? 6 : 7; }
template <bool STAGED, bool RK, bool LEAN = false>
__global__ void __launch_bounds__(IBLOCK, k1_min_blocks(STAGED, RK, LEAN)) intersect_wave(const IntersectParams P) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    __shared__ float s_lb[LEAN ? LB_ROWS * LB_STRIDE : 1];
    __shared__ double s_ls[LEAN ? LS_SLOTS * LB_STRIDE : 1];
    const SysView& S = P.S;
    // The ray state is requested first, every load at once and from a clamped slot so that none of them sits
    // behind a branch on another one's value: the DRAM round trip then overlaps the table staging below instead of
    // being paid three times in a row (alive? -> segment budget? -> position / direction).
    const int64_t ri = (int64_t)blockIdx.x * IBLOCK + threadIdx.x;
    const int64_t qs = P.cur.cap;
    const int64_t rl = ri < P.n_rays ? ri : 0;   // slot 0 exists whenever the kernel is launched
    const int q_beam = P.cur.i[I_BEAM * qs + rl], q_seg = P.cur.i[I_SEG * qs + rl];
    const int q_hint = P.cur.i[I_HINT * qs + rl], q_pose = P.cur.i[I_POSE * qs + rl];
    const double q_px = P.cur.d[F_PX * qs + rl], q_py = P.cur.d[F_PY * qs + rl], q_pz = P.cur.d[F_PZ * qs + rl];
    const double q_dx = P.cur.d[F_DX * qs + rl], q_dy = P.cur.d[F_DY * qs + rl], q_dz = P.cur.d[F_DZ * qs + rl];
    // shared-memory copies of the small system tables: prims | parts | bounds
    bmo_prim* s_prims = reinterpret_cast<bmo_prim*>(smem_raw);
    bmo_part* s_parts = reinterpret_cast<bmo_part*>(smem_raw + (size_t)S.n_prims * sizeof(bmo_prim));
    double* s_bounds = reinterpret_cast<double*>(smem_raw + (size_t)S.n_prims * sizeof(bmo_prim) + (size_t)S.n_parts * sizeof(bmo_part));
    if (STAGED) {
        stage_tables<IBLOCK, LEAN>(S, smem_raw);
        __syncthreads();
    }

    const bool active = ri < P.n_rays && q_beam >= 0;
    Stats st; st.sdf = 0; st.tri = 0;
    if (active) {
        const V3 pos = mk3(q_px, q_py, q_pz);
        const V3 dir = mk3(q_dx, q_dy, q_dz);
        const int hint = q_hint;
        const int pose = q_pose;
        const bool budget = q_seg + 1 < P.r_max;   // `while length(rays) < r_max` (System.jl:133)
        TraceCtx C;
        C.M.meshes = S.meshes; C.M.vertices = S.vertices; C.M.faces = S.faces; C.M.nodes = S.nodes; C.M.bvh_faces = S.bvh_faces;
        C.M.n_vertices = S.n_vertices; C.M.n_poses = S.n_poses; C.M.bvh_ok = S.bvh_ok;
        C.objects = S.objects; C.n_parts = S.n_parts; C.zr = S.zr;
        C.pose = pose;
        if (STAGED) { C.prims = s_prims; C.parts = s_parts; C.bounds = s_bounds; }
        else {
            C.prims = S.prims + (int64_t)pose * S.n_prims;
            C.parts = S.parts;
            C.bounds = S.bounds + NBOUND * (int64_t)pose * S.n_parts;
        }
        C.lb_addr = LEAN ? smem_u32(s_lb + threadIdx.x) : 0u;
        Hit h; h.part = -1; h.t = INFINITY; h.n = mk3(0, 0, 0);
        if (budget) {   // System.jl:100-110
            if (LEAN) h = tracing_step_lean(C, smem_u32(s_ls + threadIdx.x), C.lb_addr, smem_u32(s_bounds + NBOUND * S.n_parts), pos, dir, hint, st);
            else h = tracing_step<RK>(C, pos, dir, hint, st);
        }
        const int64_t hs = P.hit.cap;
        P.hit.d[ri] = h.t; P.hit.d[hs + ri] = h.n.x; P.hit.d[2 * hs + ri] = h.n.y; P.hit.d[3 * hs + ri] = h.n.z;
        P.hit.part[ri] = h.part;
    }
    unsigned sd = st.sdf, tr = st.tri;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        sd += __shfl_xor_sync(0xffffffffu, sd, o);
        tr += __shfl_xor_sync(0xffffffffu, tr, o);
    }
    if ((threadIdx.x & 31) == 0) {
        if (sd) atomicAdd(&P.counters->sdf, (unsigned long long)sd);
        if (tr) atomicAdd(&P.counters->tri, (unsigned long long)tr);
    }
}

// ---- K1r: intersect of a retrace call (retrace_system!, System.jl:188-255 / :326-428) ----------------
// Units are laid out like K2 (Gaussian: chief / waist / divergence in adjacent lanes, 10 triples per
// warp) because the decision "is the stored path still valid" is taken per beam.  A beam that carries a
// retrace cursor (I_RETR >= 0) intersects only what the reference intersects:
//   stored ray `seg` has no intersection                -> the stored solution ends here (cleanup, :200-206)
//   a hint came with the previous interaction           -> intersect3d(shape(_hint), ray)        (:213-218)
//   otherwise                                           -> intersect3d(object(_intersection), ray) (:209-211)
// pass 0 does that restricted intersection; if it misses (Gaussian: the three rays disagree,
// `_beams_hits_same_shape`, :367-381) the tail is dropped and solve_leaf! continues with trace_system!, whose
// first tracing_step! has no hint (:132-137): pass 1, the ordinary full trace, for exactly those beams and
// for the beams that are not retracing.  flag: 0 ordinary step, 1 re-validated (K2 must not apply the
// r_max test: retrace_system! has none), 2 stored path left in this wave.
template <int MODE, bool STAGED, bool RK, bool LEAN = false>
__global__ void __launch_bounds__(Cfg<MODE>::BLOCK, 6) retrace_intersect_wave(const StepParams P) {
    constexpr int R = Cfg<MODE>::R;
    constexpr int UNITS = Cfg<MODE>::UNITS;
    static_assert(Cfg<MODE>::BLOCK == LB_STRIDE, "the lean scratch columns are laid out for 128 threads per block");
    __shared__ float s_lb[LEAN ? LB_ROWS * LB_STRIDE : 1];
    __shared__ double s_ls[LEAN ? LS_SLOTS * LB_STRIDE : 1];
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const SysView& S = P.S;
    bmo_prim* s_prims = reinterpret_cast<bmo_prim*>(smem_raw);
    bmo_part* s_parts = reinterpret_cast<bmo_part*>(smem_raw + (size_t)S.n_prims * sizeof(bmo_prim));
    double* s_bounds = reinterpret_cast<double*>(smem_raw + (size_t)S.n_prims * sizeof(bmo_prim) + (size_t)S.n_parts * sizeof(bmo_part));
    if (STAGED) {
        stage_tables<Cfg<MODE>::BLOCK, LEAN>(S, smem_raw);
        __syncthreads();
    }
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    int uib, r;
    bool lane_ok = true;
    if (MODE == 2) { uib = warp * 10 + lane / 3; r = lane % 3; lane_ok = lane < 30; }
    else { uib = threadIdx.x; r = 0; }
    const int64_t unit = (int64_t)blockIdx.x * UNITS + uib;
    const int64_t ri = unit * R + r;
    const int64_t qs = P.cur.cap;
    const bool active = lane_ok && unit < P.count && P.cur.i[I_BEAM * qs + ri] >= 0;

    Stats st; st.sdf = 0; st.tri = 0;
    Hit h; h.part = -1; h.t = INFINITY; h.n = mk3(0, 0, 0);
    V3 pos = mk3(0, 0, 0), dir = mk3(0, 1, 0);
    int hint = -1, pose = 0, seg = 0, pb = -1;
    if (active) {
        const double* q = P.cur.d;
        pos = mk3(q[F_PX * qs + ri], q[F_PY * qs + ri], q[F_PZ * qs + ri]);
        dir = mk3(q[F_DX * qs + ri], q[F_DY * qs + ri], q[F_DZ * qs + ri]);
        hint = P.cur.i[I_HINT * qs + ri];
        pose = P.cur.i[I_POSE * qs + ri];
        seg = P.cur.i[I_SEG * qs + ri];
        pb = P.cur.i[I_RETR * qs + ri];
    }
    const bool budget = seg + 1 < P.r_max;   // `while length(rays) < r_max` (System.jl:133), trace_system! only
    TraceCtx C;
    C.M.meshes = S.meshes; C.M.vertices = S.vertices; C.M.faces = S.faces; C.M.nodes = S.nodes; C.M.bvh_faces = S.bvh_faces;
    C.M.n_vertices = S.n_vertices; C.M.n_poses = S.n_poses; C.M.bvh_ok = S.bvh_ok;
    C.objects = S.objects; C.n_parts = S.n_parts; C.zr = S.zr;
    C.pose = pose;
    C.lb_addr = 0u;
    if (STAGED) { C.prims = s_prims; C.parts = s_parts; C.bounds = s_bounds; }
    else {
        C.prims = S.prims + (int64_t)pose * S.n_prims;
        C.parts = S.parts;
        C.bounds = S.bounds + NBOUND * (int64_t)pose * S.n_parts;
    }
    const bool in_phase = active && pb >= 0;
    int lo = 0, hi = 0;
    bool restricted = false;
    if (in_phase && seg < P.rt.nseg[pb]) {
        const int ppart = P.rt.seg_part[(P.rt.first_seg[pb] + seg) * R];   // what the stored (chief) ray hit
        if (ppart >= 0) {
            restricted = true;
            if (hint >= 0) { lo = hint; hi = hint + 1; }
            else { const bmo_object& ob = S.objects[S.parts[ppart].object]; lo = ob.first_part; hi = lo + ob.n_parts; }
        }
    }
    bool ok = false;
    int flag = 0;
#pragma unroll 1
    for (int pass = 0; pass < 2; pass++) {
        bool run;
        int hp = -1, plo = lo, phi = hi;
        if (pass == 0) run = restricted;
        else { run = active && budget && !(in_phase && ok); hp = in_phase ? -1 : hint; plo = 0; phi = S.n_parts; }
        if (run) {
            if (LEAN) h = tracing_step_lean(C, smem_u32(s_ls + threadIdx.x), smem_u32(s_lb + threadIdx.x), smem_u32(s_bounds + NBOUND * S.n_parts), pos, dir, hp, st, plo, phi);
            else h = tracing_step<RK>(C, pos, dir, hp, st, plo, phi);
        }
        if (pass == 0) {
            ok = restricted && h.part >= 0;
            if (MODE == 2) {   // Gaussian.jl:171-180: all three rays must hit the same shape
                __syncwarp();
                const int base = lane - r, lw = min(base + 1, 31), ld = min(base + 2, 31);
                const int pc = __shfl_sync(0xffffffffu, h.part, base), pw = __shfl_sync(0xffffffffu, h.part, lw),
                          pd = __shfl_sync(0xffffffffu, h.part, ld);
                ok = restricted && pc >= 0 && pc == pw && pw == pd;
            }
            if (in_phase) {
                flag = ok ? 1 : 2;
                if (!ok) { h.part = -1; h.t = INFINITY; h.n = mk3(0, 0, 0); }
            }
        }
    }
    if (active) {
        const int64_t hs = P.hit.cap;
        P.hit.d[ri] = h.t; P.hit.d[hs + ri] = h.n.x; P.hit.d[2 * hs + ri] = h.n.y; P.hit.d[3 * hs + ri] = h.n.z;
        P.hit.part[ri] = h.part;
        P.hit.flag[ri] = flag;
    }
    unsigned sd = st.sdf, tr = st.tri;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        sd += __shfl_xor_sync(0xffffffffu, sd, o);
        tr += __shfl_xor_sync(0xffffffffu, tr, o);
    }
    if (lane == 0) {
        if (sd) atomicAdd(&P.counters->sdf, (unsigned long long)sd);
        if (tr) atomicAdd(&P.counters->tri, (unsigned long long)tr);
    }
}

// ---- interact3d without polarisation -------------------------------------------------------------------
// Spotdetector.jl:50-61: where the ray meets the detector plane, in the detector's (x, z)
struct SpotHit { int obj; double x, z; };
BMO_D void spot_hit(const SysView& S, int object, int pose, V3 pos, V3 dir, double t, SpotHit& sp) {
    const double* dp = S.det_pose + 12 * ((int64_t)pose * S.n_objects + object);
    V3 hp = pos + t * dir;
    V3 loc = hp - mk3(dp[0], dp[1], dp[2]);
    sp.obj = object;
    sp.x = dot(loc, mk3(dp[3], dp[6], dp[9]));     // orientation[:,1]
    sp.z = dot(loc, mk3(dp[5], dp[8], dp[11]));    // orientation[:,3]
}
// interact3d of a plain ray, or of one ray of a Gaussian triple, with part hit_part (pt of object ob) at distance t, normal nrm:
// the continuing ray goes to o (o.valid stays false when interact3d returns nothing), a Spotdetector hit to sp, and split is set
// when the part is a beamsplitter coating (the children are made by the caller).  The state is passed by value so that the
// wavefront kernels (interact_body) and the whole-solve kernel (solve_rays_persistent) run the same code on it.
BMO_D void interact_plain(const SysView& S, const bmo_part& pt, const bmo_object& ob, int hit_part, V3 pos, V3 dir, double rn, double t,
                          V3 nrm, int lam, int pose, RayOut& o, bool& split, SpotHit& sp) {
    const auto n_of_hit = [&]() { return S.n_table[pt.n_row * S.n_lambda + lam]; };   // only refractive parts have a row
    switch (ob.kind) {
        case BMO_OBJ_REFRACTIVE:
            interact_refractive_plain(pos, dir, rn, t, nrm, n_of_hit(), S.n_system, hit_part, o);
            break;
        case BMO_OBJ_DOUBLET:      // DoubletLenses.jl:66-76
            interact_refractive_plain(pos, dir, rn, t, nrm, n_of_hit(), S.n_system, hit_part, o);
            o.hint = ob.first_part + (1 - (hit_part - ob.first_part));
            break;
        case BMO_OBJ_MIRROR:
            interact_mirror_plain(pos, dir, rn, t, nrm, o);
            break;
        case BMO_OBJ_CUBE_BS:      // CubeBeamsplitter.jl:63-121
            if (pt.role == BMO_ROLE_COATING) split = true;
            else {
                interact_refractive_plain(pos, dir, rn, t, nrm, n_of_hit(), S.n_system, hit_part, o);
                o.hint = ob.first_part + 2;
            }
            break;
        case BMO_OBJ_PLATE_BS:     // PlateBeamsplitter.jl:189-275
            if (pt.role == BMO_ROLE_COATING) split = true;
            else {
                interact_refractive_plain(pos, dir, rn, t, nrm, n_of_hit(), S.n_system, hit_part, o);
                o.hint = ob.first_part + 1;
            }
            break;
        case BMO_OBJ_THIN_BS:
            split = true;
            break;
        case BMO_OBJ_SPOTDETECTOR:
            spot_hit(S, pt.object, pose, pos, dir, t, sp);
            break;
        default: break;  // PolarizationFilter (PolarizedRay only: no method -> nothing), Photodetector, IntersectableObject
    }
}

// ---- K2: interact + block-local compaction ----------------------------------------------------------
// The body is shared by the stand-alone kernel (hit records read from the buffer K1 wrote) and by the
// fused kernel of splitter-free plain-ray systems (hit still in registers, FUSED = true).
// NS: the system has no beamsplitter (host-side fact): no spawn events, so the block-level numbering of children, its two
// barriers and the scratch queue are compiled out and the units alive after the wave are counted per warp.
template <int MODE, bool FUSED, bool NS = false>
BMO_D void interact_body(const StepParams& P, const Hit& h_reg, const int wave_off = 0) {
    constexpr int R = Cfg<MODE>::R;
    constexpr int UNITS = Cfg<MODE>::UNITS;
    constexpr int NWARP = Cfg<MODE>::NWARP;
    __shared__ int s_wcnt[NWARP][2];
    __shared__ int s_woff[NWARP][2];

    const SysView& S = P.S;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    int uib, r;
    bool lane_ok = true;
    if (MODE == 2) { uib = warp * 10 + lane / 3; r = lane % 3; lane_ok = lane < 30; }
    else { uib = threadIdx.x; r = 0; }
    const int64_t unit = (int64_t)blockIdx.x * UNITS + uib;
    const bool in_queue = lane_ok && unit < P.count;
    const int64_t ri = unit * R + r;
    const int64_t qs = P.cur.cap;
    // All loads of the unit's state are issued at once from a clamped slot (slot 0 exists whenever the kernel runs):
    // behind `if (active)` they would wait for the alive flag's own DRAM round trip first.
    const int64_t rl = in_queue ? ri : 0;
    const int32_t* qi = P.cur.i;
    const double* q = P.cur.d;
    const int q_beam = qi[I_BEAM * qs + rl];
    int lam = qi[I_LAM * qs + rl], seg = qi[I_SEG * qs + rl], pose = qi[I_POSE * qs + rl];
    V3 pos = mk3(q[F_PX * qs + rl], q[F_PY * qs + rl], q[F_PZ * qs + rl]);
    V3 dir = mk3(q[F_DX * qs + rl], q[F_DY * qs + rl], q[F_DZ * qs + rl]);
    double rn = q[F_N * qs + rl];
    Cx E0[3];
    E0[0] = E0[1] = E0[2] = mkc(0, 0);
    if (MODE == 1) {
#pragma unroll
        for (int k = 0; k < 3; k++) E0[k] = mkc(q[(F_X0 + 2 * k) * qs + rl], q[(F_X0 + 2 * k + 1) * qs + rl]);
    }
    double acc_lsum = 0, acc_lpar = 0, acc_opl = 0;
    if (MODE == 2) { acc_lsum = q[F_X0 * qs + rl]; acc_lpar = q[(F_X0 + 1) * qs + rl]; acc_opl = q[(F_X0 + 2) * qs + rl]; }
    Hit h; h.part = -1; h.t = INFINITY; h.n = mk3(0, 0, 0);
    if (FUSED) h = h_reg;
    else {
        const int64_t hs = P.hit.cap;
        h.t = P.hit.d[rl]; h.n = mk3(P.hit.d[hs + rl], P.hit.d[2 * hs + rl], P.hit.d[3 * hs + rl]);
        h.part = P.hit.part[rl];
    }
    const bool active = in_queue && q_beam >= 0;   // dead slots wait for the next compaction
    const bool leader = active && r == 0;
    int beam = q_beam;
    if (!active) {   // the values a dead / absent lane carried before (they reach other lanes through the Gaussian shuffles)
        pos = mk3(0, 0, 0); dir = mk3(0, 1, 0); rn = 1.0; lam = 0; beam = 0; seg = 0; pose = 0;
        E0[0] = E0[1] = E0[2] = mkc(0, 0); acc_lsum = acc_lpar = acc_opl = 0;
        h.part = -1; h.t = INFINITY; h.n = mk3(0, 0, 0);
    }
    // retrace calls (K1r): how this wave's intersection was obtained, and the beam's retrace cursor
    int rflag = 0, pb = -1;
    if (!FUSED && P.rt.on && active) { rflag = P.hit.flag[ri]; pb = P.cur.i[I_RETR * qs + ri]; }

    // ---- outcome of tracing_step! (System.jl:100-110, intersect_wave) ----
    int status = BMO_ST_ACTIVE;
    if (active) {
        if (seg + 1 >= P.r_max && rflag != 1) {   // `while length(rays) < r_max`, System.jl:133 / :281: not traced (retrace_system! has no such test)
            status = BMO_ST_RMAX;
            h.part = -1; h.t = INFINITY; h.n = mk3(0, 0, 0);
        } else if (h.part < 0) status = BMO_ST_MISS;
    }
    double seg_t = h.t;       // t stored in this lane's segment record (Inf <=> intersection === nothing)
    int hit_part = h.part;    // part the interaction dispatches on (Gaussian: the chief's)

    // ---- Gaussian triple rules (System.jl:283-304) ----
    V3 c_pos = pos, c_dir = dir, c_nrm = h.n, w_pos = pos, w_dir = dir, d_pos = pos, d_dir = dir;
    double c_t = h.t, c_n = rn;
    int base = lane, lw = lane, ld = lane;
    if (MODE == 2) {
        __syncwarp();
        base = lane - r; lw = min(base + 1, 31); ld = min(base + 2, 31);
        const unsigned full = 0xffffffffu;
        const int pc = __shfl_sync(full, h.part, base), pw = __shfl_sync(full, h.part, lw), pd = __shfl_sync(full, h.part, ld);
        const int stc = __shfl_sync(full, status, base);
        c_pos = shfl3(pos, base); c_dir = shfl3(dir, base); c_nrm = shfl3(h.n, base);
        w_pos = shfl3(pos, lw); w_dir = shfl3(dir, lw);
        d_pos = shfl3(pos, ld); d_dir = shfl3(dir, ld);
        c_t = __shfl_sync(full, h.t, base);
        c_n = __shfl_sync(full, rn, base);
        hit_part = pc;
        if (active) {
            if (stc == BMO_ST_RMAX) { status = BMO_ST_RMAX; seg_t = INFINITY; }
            else if (pc < 0) { status = BMO_ST_MISS; seg_t = INFINITY; }                 // chief missed: the others are not traced
            else if (pw < 0) { status = BMO_ST_CLIPPED; if (r != 0) seg_t = INFINITY; }  // chief keeps its intersection (:288-291)
            else if (pd < 0) { status = BMO_ST_CLIPPED; if (r == 2) seg_t = INFINITY; }  // (:292-296)
            else if (!(pc == pw && pw == pd)) { status = BMO_ST_TORN; seg_t = INFINITY; }  // (:298-304)
            else status = BMO_ST_ACTIVE;
        }
    }

    // ---- interact (dispatch on the object kind / part role) ----
    int nsucc = 0;
    RayOut o1, o2;                 // continuing ray, or (transmitted, reflected) children
    o1.valid = o2.valid = false; o1.err = o2.err = false; o1.warn = o2.warn = false;
    o1.hint = o2.hint = -1;
    bool interacted = false;
    if (active && status == BMO_ST_ACTIVE && hit_part >= 0) {
        interacted = true;
        const bmo_part& pt = S.parts[hit_part];
        const bmo_object& ob = S.objects[pt.object];
        const bool pol = MODE == 1;
        const double t = h.t;
        bool split = false;
        // Plain rays and Gaussian triples (MODE 0 / 2) take the inlined interactions; whatever is out of line writes into
        // temporaries, so that o1 / o2 / E0 never have their address taken on this path and stay in registers.
        const auto n_of_hit = [&]() { return S.n_table[pt.n_row * S.n_lambda + lam]; };   // only refractive parts have a row
        RayOut ta, tb;
        ta.valid = tb.valid = false; ta.err = tb.err = false; ta.warn = tb.warn = false; ta.hint = tb.hint = -1;
        Cx Et[3];
        SpotHit sp; sp.obj = -1;
        if (!pol) interact_plain(S, pt, ob, hit_part, pos, dir, rn, t, h.n, lam, pose, o1, split, sp);
        else {
            Et[0] = E0[0]; Et[1] = E0[1]; Et[2] = E0[2];
            switch (ob.kind) {
                case BMO_OBJ_REFRACTIVE:
                    interact_refractive(pos, dir, rn, Et, true, t, h.n, n_of_hit(), S.n_system, hit_part, ta); o1 = ta;
                    break;
                case BMO_OBJ_MIRROR:
                    interact_mirror(pos, dir, rn, Et, true, t, h.n, ta); o1 = ta;
                    break;
                case BMO_OBJ_CUBE_BS:      // CubeBeamsplitter.jl:63-121
                    if (pt.role == BMO_ROLE_COATING) split = true;
                    else {
                        interact_refractive(pos, dir, rn, Et, true, t, h.n, n_of_hit(), S.n_system, hit_part, ta); o1 = ta;
                        o1.hint = ob.first_part + 2;
                    }
                    break;
                case BMO_OBJ_PLATE_BS:     // PlateBeamsplitter.jl:189-275
                    if (pt.role == BMO_ROLE_COATING) split = true;
                    else {
                        interact_refractive(pos, dir, rn, Et, true, t, h.n, n_of_hit(), S.n_system, hit_part, ta); o1 = ta;
                        o1.hint = ob.first_part + 1;
                    }
                    break;
                case BMO_OBJ_THIN_BS:
                    split = true;
                    break;
                case BMO_OBJ_POLFILTER: {   // PolarizationFilter.jl:31-47
                    const double* dp = S.det_pose + 12 * ((int64_t)pose * S.n_objects + pt.object);
                    interact_polfilter(pos, dir, rn, Et, t, dp + 3, S.jones + 10 * (int64_t)ob.pd_n, ta);
                    o1 = ta;
                    break;
                }
                case BMO_OBJ_SPOTDETECTOR:
                    spot_hit(S, pt.object, pose, pos, dir, t, sp);
                    break;
                default: break;  // Doublet (Ray only; a PolarizedRay has no method -> nothing), Photodetector, IntersectableObject
            }
        }
        if (sp.obj >= 0) {
            const int64_t bi = (int64_t)beam * R + r;
            P.B.spot_obj[bi] = sp.obj;
            P.B.spot_xz[2 * bi] = sp.x;
            P.B.spot_xz[2 * bi + 1] = sp.z;
        }
        if (!NS && split) {
            bs_children(pos, dir, Et, pol, t, h.n, pt.reflectance, pt.transmittance, ta, tb);
            o1 = ta; o2 = tb;
            if (ob.kind == BMO_OBJ_CUBE_BS) {          // CubeBeamsplitter.jl:80-82,110-112
                const double ng = S.n_table[S.parts[ob.first_part].n_row * S.n_lambda + lam];
                o1.n = ng; o2.n = ng;
            } else if (ob.kind == BMO_OBJ_PLATE_BS) {  // PlateBeamsplitter.jl:207-223,247-270
                const double n_opt = S.n_table[S.parts[ob.first_part].n_row * S.n_lambda + lam];
                const bool entering = (MODE == 2) ? (dot(c_dir, c_nrm) < 0) : (dot(dir, h.n) < 0);
                const double n2 = entering ? n_opt : S.n_system;
                bool tir, err = false;
                V3 nd = refraction3d_ray(dir, h.n, rn, n2, tir, err);
                o1.n = entering ? n_opt : S.n_system;
                o2.n = entering ? S.n_system : n_opt;
                o1.dir = normalize(nd);
                if (err) o1.err = true;
            }
            nsucc = 2;
            status = BMO_ST_SPLIT;
        } else if (o1.valid) {
            nsucc = 1;
        } else {
            status = BMO_ST_ABSORBED;
        }
        if ((o1.valid && o1.err) || (o2.valid && o2.err)) { status = BMO_ST_ERROR; nsucc = 0; }
    }

    // ---- Gaussian: triple-level agreement, chief hint, child beamlet parameters ----
    double g_w0 = 0, g_plen = 0, g_popl = 0;
    Cx g_et = mkc(0, 0), g_er = mkc(0, 0);
    double n_lsum = 0, n_lpar = 0, n_opl = 0;  // accumulators of the continuing / child rays
    if (MODE == 2) {
        __syncwarp();
        const unsigned full = 0xffffffffu;
        const int n0 = __shfl_sync(full, nsucc, base), n1 = __shfl_sync(full, nsucc, lw), n2 = __shfl_sync(full, nsucc, ld);
        const int s0 = __shfl_sync(full, status, base), s1 = __shfl_sync(full, status, lw), s2 = __shfl_sync(full, status, ld);
        const int hc = __shfl_sync(full, o1.hint, base);
        const double accl = __shfl_sync(full, acc_lsum, base), accp = __shfl_sync(full, acc_lpar, base),
                     acco = __shfl_sync(full, acc_opl, base);
        if (interacted) {
            int nm = min(n0, min(n1, n2));
            if (s0 == BMO_ST_ERROR || s1 == BMO_ST_ERROR || s2 == BMO_ST_ERROR) { status = BMO_ST_ERROR; nm = 0; }
            else if (nm == 0) status = BMO_ST_ABSORBED;   // any(isnothing, (i_c, i_w, i_d)) -> nothing (Gaussian.jl:131-133)
            nsucc = nm;
            o1.hint = hc;                                  // hint(i::GaussianBeamletInteraction) = hint(i.chief), Gaussian.jl:80
            if (nm == 1) {                                 // Beam.jl:125-205 running sums (association kept)
                n_lsum = accl + c_t; n_lpar = accp + c_t; n_opl = acco + c_t * c_n;
            } else if (nm == 2) {                          // ThinBeamsplitter.jl:117-168
                const bmo_part& pt = S.parts[hit_part];
                const double plen_parent = P.B.plen[beam];
                const double L = (accl + c_t) + plen_parent;              // length(gauss) = l + l0
                V3 p0 = c_pos + (L - accp) * c_dir;                        // point_on_beam(gauss, length(gauss)), Beam.jl:201-204
                double w, Rc, psi, w0n;
                gauss_parameters(p0, c_dir, c_n, w_pos, w_dir, d_pos, d_dir, S.lambdas[lam], w, Rc, psi, w0n);
                const double w0b = P.B.w0[beam];
                const Cx e0b = mkc(P.B.e0[2 * beam], P.B.e0[2 * beam + 1]);
                g_w0 = w0n;
                g_et = (pt.transmittance * e0b) * (w0b / w0n);
                g_er = (pt.reflectance * e0b) * (w0b / w0n);
                const double phi = (dot(c_dir, c_nrm) < 0) ? kPi : 0.0;  // reflection phase jump, :151-158
                g_er = g_er * cis(phi);
                g_plen = L;
                g_popl = acco + c_t * c_n;
                n_lsum = 0.0; n_lpar = L; n_opl = g_popl;
            }
        }
    }

    // ---- retrace cursor (System.jl:238-247 / :402-411) ----
    // A re-validated ray whose successor exists in the stored solution replaces that successor and the
    // beam keeps retracing; if it was the last stored ray the new ray is pushed, the children are dropped
    // and solve_leaf! continues with trace_system!, whose first tracing_step! has no hint.  Children of a
    // re-validated splitter hit keep their stored paths (children!, AbstractBeam.jl:59-76): they start
    // with the cursor of the stored child; Gaussian children also keep their stored w0
    // (_modify_beam_head!, Gaussian.jl:154-162, copies wavelength and E0 only).
    int retr_next = -1, retr_child0 = -1, retr_child1 = -1;
    if (rflag == 1 && pb >= 0) {
        const int np = P.rt.nseg[pb];
        if (nsucc == 1) {
            if (seg + 1 < np) retr_next = pb;
            else o1.hint = -1;
        } else if (nsucc == 2 && seg + 1 == np) {
            retr_child0 = P.rt.child[2 * pb]; retr_child1 = P.rt.child[2 * pb + 1];
        }
        // replace! (Beam.jl:81-95) and _modify_beam_head! (Beam.jl:97-112) write through direction!, which
        // normalises (AbstractRay.jl:83-86); push! of a fresh ray does not
        if (retr_next >= 0) o1.dir = normalize(o1.dir);
        if (retr_child0 >= 0) o1.dir = normalize(o1.dir);
        if (retr_child1 >= 0) o2.dir = normalize(o2.dir);
    }

    // ---- bookkeeping: counters, segment record, per-beam state ----
    if (P.keep && in_queue && !active) P.wave.beam[ri] = -1;
    if (P.keep && active) {
        const int64_t ws = P.wave.count;
        double* w = P.wave.d;
        w[S_PX * ws + ri] = pos.x; w[S_PY * ws + ri] = pos.y; w[S_PZ * ws + ri] = pos.z;
        w[S_DX * ws + ri] = dir.x; w[S_DY * ws + ri] = dir.y; w[S_DZ * ws + ri] = dir.z;
        w[S_N * ws + ri] = rn; w[S_T * ws + ri] = seg_t;
        w[S_NX * ws + ri] = h.n.x; w[S_NY * ws + ri] = h.n.y; w[S_NZ * ws + ri] = h.n.z;
        if (MODE == 1) {
#pragma unroll
            for (int k = 0; k < 3; k++) { w[(S_E0 + 2 * k) * ws + ri] = E0[k].re; w[(S_E0 + 2 * k + 1) * ws + ri] = E0[k].im; }
        }
        P.wave.part[ri] = isinf(seg_t) ? -1 : h.part;
        P.wave.beam[ri] = beam;
        P.wave.seg[ri] = seg;
    }
    if (leader) {
        P.B.nseg[beam] = seg + 1;
        // bit 8: the reference's E0-orthogonality check (atol 1e-14) failed somewhere along this beam
        const bool warn = (o1.valid && o1.warn) || (o2.valid && o2.warn);
        if (nsucc != 1 || warn) {   // a continuing beam without a new warning keeps its word: no read-modify-write
            const int old = P.B.status[beam];
            const int wbit = (old & 0x100) | (warn ? 0x100 : 0);
            P.B.status[beam] = ((nsucc != 1) ? status : (old & 0xff)) | wbit;
        }
    }

    // ---- successors ----
    // nsucc == 1: the continuing ray overwrites its own queue slot (no data movement between waves);
    // nsucc == 0: the slot is marked dead (beam = -1) and removed by the next compaction (K3);
    // nsucc == 2: beamsplitter children go to the block's scratch area in queue order (warp ballot +
    //             prefix sums), spawn_children numbers them deterministically and puts the transmitted
    //             child into the parent's slot, the reflected child at the tail of the queue.
    const unsigned full = 0xffffffffu;
    int wsoff = 0;
    if (NS) {
        const unsigned alive = __popc(__ballot_sync(full, leader && nsucc >= 1));
        const unsigned ia = __popc(__ballot_sync(full, interacted));
        if (lane == 0) {
            if (ia) atomicAdd(&P.counters->interactions, (unsigned long long)ia);
            if (alive) atomicAdd(P.wave_totals + 2 * wave_off, (unsigned long long)alive);   // units alive in the next wave
        }
    } else {
        const unsigned b2 = __ballot_sync(full, leader && nsucc == 2);
        const unsigned lt = lanemask_lt();
        wsoff = __popc(b2 & lt);                     // spawn events of lower lanes
        const unsigned alive = __popc(__ballot_sync(full, leader && nsucc >= 1)) + __popc(b2);
        if (lane == 0) { s_wcnt[warp][0] = (int)alive; s_wcnt[warp][1] = __popc(b2); }
        const unsigned ia = __popc(__ballot_sync(full, interacted));
        if (lane == 0 && ia) atomicAdd(&P.counters->interactions, (unsigned long long)ia);
        __syncthreads();
        if (threadIdx.x == 0) {
            int a = 0, b = 0;
            for (int k = 0; k < NWARP; k++) { s_woff[k][1] = b; a += s_wcnt[k][0]; b += s_wcnt[k][1]; }
            P.blk_cnt[blockIdx.x] = b;
            if (a) atomicAdd(P.wave_totals + 2 * wave_off, (unsigned long long)a);        // units alive in the next wave
            if (b) atomicAdd(P.wave_totals + 2 * wave_off + 1, (unsigned long long)b);    // spawn events
        }
        __syncthreads();
    }
    if (MODE == 2) wsoff = __shfl_sync(full, wsoff, base);
    if (active) {
        int32_t* qi = P.cur.i;
        if (nsucc == 1) {
            double* d = P.cur.d;
            d[F_PX * qs + ri] = o1.pos.x; d[F_PY * qs + ri] = o1.pos.y; d[F_PZ * qs + ri] = o1.pos.z;
            d[F_DX * qs + ri] = o1.dir.x; d[F_DY * qs + ri] = o1.dir.y; d[F_DZ * qs + ri] = o1.dir.z;
            d[F_N * qs + ri] = o1.n;
            if (MODE == 1) {
#pragma unroll
                for (int c = 0; c < 3; c++) { d[(F_X0 + 2 * c) * qs + ri] = o1.E0[c].re; d[(F_X0 + 2 * c + 1) * qs + ri] = o1.E0[c].im; }
            }
            if (MODE == 2) { d[F_X0 * qs + ri] = n_lsum; d[(F_X0 + 1) * qs + ri] = n_lpar; d[(F_X0 + 2) * qs + ri] = n_opl; }
            qi[I_HINT * qs + ri] = o1.hint;
            qi[I_SEG * qs + ri] = seg + 1;
            if (P.rt.on) qi[I_RETR * qs + ri] = retr_next;
        } else {
            qi[I_BEAM * qs + ri] = -1;
        }
        if (!NS && nsucc == 2) {
            const int64_t ss = P.scr.cap;
            const int lspawn = s_woff[warp][1] + wsoff;
            for (int k = 0; k < 2; k++) {
                const RayOut& o = (k == 0) ? o1 : o2;
                const int64_t si = (((int64_t)blockIdx.x * UNITS + lspawn) * 2 + k) * R + r;
                double* d = P.scr.d;
                d[F_PX * ss + si] = o.pos.x; d[F_PY * ss + si] = o.pos.y; d[F_PZ * ss + si] = o.pos.z;
                d[F_DX * ss + si] = o.dir.x; d[F_DY * ss + si] = o.dir.y; d[F_DZ * ss + si] = o.dir.z;
                d[F_N * ss + si] = o.n;
                if (MODE == 1) {
#pragma unroll
                    for (int c = 0; c < 3; c++) { d[(F_X0 + 2 * c) * ss + si] = o.E0[c].re; d[(F_X0 + 2 * c + 1) * ss + si] = o.E0[c].im; }
                }
                if (MODE == 2) {
                    d[F_X0 * ss + si] = n_lsum; d[(F_X0 + 1) * ss + si] = n_lpar; d[(F_X0 + 2) * ss + si] = n_opl;
                    const Cx e = (k == 0) ? g_et : g_er;
                    const int rc = (k == 0) ? retr_child0 : retr_child1;
                    d[(F_X0 + 3) * ss + si] = rc >= 0 ? P.rt.w0[rc] : g_w0; d[(F_X0 + 4) * ss + si] = e.re; d[(F_X0 + 5) * ss + si] = e.im;
                    d[(F_X0 + 6) * ss + si] = g_plen; d[(F_X0 + 7) * ss + si] = g_popl;
                }
                int32_t* iq = P.scr.i;
                iq[I_LAM * ss + si] = lam;
                iq[I_BEAM * ss + si] = beam;       // parent beam
                iq[I_POSE * ss + si] = pose;
                iq[I_RETR * ss + si] = (k == 0) ? retr_child0 : retr_child1;
                iq[I_PUNIT * ss + si] = (int32_t)unit;
            }
        }
    }
}

template <int MODE, bool NS = false>
__global__ void __launch_bounds__(Cfg<MODE>::BLOCK, MODE == 0 ? 6 : 1) interact_wave(const StepParams P) {
    Hit none; none.part = -1; none.t = INFINITY; none.n = mk3(0, 0, 0);
    interact_body<MODE, false, NS>(P, none);
}

// ---- K1+K2 fused: plain rays through a system without beamsplitters (the sequential lens-stack path) --
// One thread per ray does tracing_step! and interact3d back to back: the hit record never leaves the
// registers and the ray state is read once.  Needs IBLOCK == Cfg<0>::BLOCK == Cfg<0>::UNITS.
// Resident blocks per SM it is compiled for: 6 with staged tables (the lean build included), 4 without.
constexpr int fused_min_blocks(bool staged) { return staged ? 6 : 4; }
template <bool STAGED, bool RK, bool LEAN = false>
__global__ void __launch_bounds__(IBLOCK, fused_min_blocks(STAGED)) fused_wave0(const StepParams P) {
    static_assert(IBLOCK == Cfg<0>::BLOCK && Cfg<0>::UNITS == IBLOCK, "fused_wave0 maps one thread to one ray like interact_wave<0>");
    __shared__ float s_lb[LEAN ? LB_ROWS * LB_STRIDE : 1];
    __shared__ double s_ls[LEAN ? LS_SLOTS * LB_STRIDE : 1];
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const SysView& S = P.S;
    bmo_prim* s_prims = reinterpret_cast<bmo_prim*>(smem_raw);
    bmo_part* s_parts = reinterpret_cast<bmo_part*>(smem_raw + (size_t)S.n_prims * sizeof(bmo_prim));
    double* s_bounds = reinterpret_cast<double*>(smem_raw + (size_t)S.n_prims * sizeof(bmo_prim) + (size_t)S.n_parts * sizeof(bmo_part));
    if (STAGED) {
        stage_tables<IBLOCK, LEAN>(S, smem_raw);
        __syncthreads();
    }
    const int64_t ri = (int64_t)blockIdx.x * IBLOCK + threadIdx.x;
    const int64_t qs = P.cur.cap;
    // Splitter-free systems never grow the queue and every continuing ray overwrites its own slot, so one launch
    // can run several waves back to back: the thread re-reads the slot it wrote (L1 / L2 hits), the hit record and
    // the table staging are not repeated, and the host gets the per-wave totals exactly as from separate launches.
    unsigned sd = 0, tr = 0;
#pragma unroll 1
    for (int w = 0; w < P.n_waves; w++) {
        const bool active = ri < P.count && P.cur.i[I_BEAM * qs + ri] >= 0;
        if (w > 0 && !__syncthreads_or(active)) break;      // the whole block is done
        Stats st; st.sdf = 0; st.tri = 0;
        Hit h; h.part = -1; h.t = INFINITY; h.n = mk3(0, 0, 0);
        if (active) {
            const double* q = P.cur.d;
            const V3 pos = mk3(q[F_PX * qs + ri], q[F_PY * qs + ri], q[F_PZ * qs + ri]);
            const V3 dir = mk3(q[F_DX * qs + ri], q[F_DY * qs + ri], q[F_DZ * qs + ri]);
            const int hint = P.cur.i[I_HINT * qs + ri];
            const int pose = P.cur.i[I_POSE * qs + ri];
            const bool budget = P.cur.i[I_SEG * qs + ri] + 1 < P.r_max;
            TraceCtx C;
            C.M.meshes = S.meshes; C.M.vertices = S.vertices; C.M.faces = S.faces; C.M.nodes = S.nodes; C.M.bvh_faces = S.bvh_faces;
            C.M.n_vertices = S.n_vertices; C.M.n_poses = S.n_poses; C.M.bvh_ok = S.bvh_ok;
            C.objects = S.objects; C.n_parts = S.n_parts; C.zr = S.zr;
            C.pose = pose;
            if (STAGED) { C.prims = s_prims; C.parts = s_parts; C.bounds = s_bounds; }
            else {
                C.prims = S.prims + (int64_t)pose * S.n_prims;
                C.parts = S.parts;
                C.bounds = S.bounds + NBOUND * (int64_t)pose * S.n_parts;
            }
            C.lb_addr = LEAN ? smem_u32(s_lb + threadIdx.x) : 0u;
            if (budget) {
                if (LEAN) h = tracing_step_lean(C, smem_u32(s_ls + threadIdx.x), C.lb_addr, smem_u32(s_bounds + NBOUND * S.n_parts), pos, dir, hint, st);
                else h = tracing_step<RK>(C, pos, dir, hint, st);
            }
        }
        sd += st.sdf; tr += st.tri;
        interact_body<0, true, true>(P, h, w);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        sd += __shfl_xor_sync(0xffffffffu, sd, o);
        tr += __shfl_xor_sync(0xffffffffu, tr, o);
    }
    if ((threadIdx.x & 31) == 0) {
        if (sd) atomicAdd(&P.counters->sdf, (unsigned long long)sd);
        if (tr) atomicAdd(&P.counters->tri, (unsigned long long)tr);
    }
}

// ---- whole solve of plain rays through a splitter-free LEAN system in one launch ---------------------------
// Without beamsplitters no ray ever makes or meets another one, so the wave structure (queue, hit records, one launch per wave,
// compaction) has nothing to coordinate: each thread carries its ray from the caller's inputs through tracing_step! and
// interact3d until it dies, misses, reaches a detector or has r_max rays, and writes its beam-table entry once.  As many
// blocks as are resident at once stage the tables once; each warp takes tiles of 32 rays from a global counter, so rays
// with more interactions than others do not leave a tail.  The march and interact_plain are the device functions the wave
// kernels run, in the same order, so every per-ray result and counter is the wave path's bit for bit.
struct SolveParams {
    SysView S;
    const double *pos, *dir;        // [n][3]; dir [3] with dir_uniform (BMO_UNIFORM_DIR)
    const int32_t *lam, *pose;      // [n] or NULL (0 for every ray)
    int64_t n;
    int32_t r_max, dir_uniform;
    BeamTab B;
    DevCounters* counters;          // tiles and most_nseg zeroed by the caller
};
// Per-thread scratch columns besides the march's (s_ls): the ray's refractive index (s_pn), wavelength id and segment index
// (s_pi rows 0 / 1) are not needed by the march and would otherwise hold registers through it.  2 KB on top of the 22 KB of
// intersect_wave's static scratch: with the LEAN gate's 24 KB of tables (staged_smem) a block stays within the 48 KB it gets
// without opting in (checked at launch, persistent_blocks).  6 resident blocks per SM: the fastest on C2 (DESIGN §5).
__global__ void __launch_bounds__(IBLOCK, 6) solve_rays_persistent(const SolveParams P) {
    __shared__ float s_lb[LB_ROWS * LB_STRIDE];
    __shared__ double s_ls[LS_SLOTS * LB_STRIDE];
    __shared__ double s_pn[LB_STRIDE];
    __shared__ int s_pi[2 * LB_STRIDE];
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const SysView& S = P.S;
    bmo_prim* s_prims = reinterpret_cast<bmo_prim*>(smem_raw);
    bmo_part* s_parts = reinterpret_cast<bmo_part*>(smem_raw + (size_t)S.n_prims * sizeof(bmo_prim));
    double* s_bounds = reinterpret_cast<double*>(smem_raw + (size_t)S.n_prims * sizeof(bmo_prim) + (size_t)S.n_parts * sizeof(bmo_part));
    stage_tables<IBLOCK, true>(S, smem_raw);
    __syncthreads();
    TraceCtx C;
    C.M.meshes = S.meshes; C.M.vertices = S.vertices; C.M.faces = S.faces; C.M.nodes = S.nodes; C.M.bvh_faces = S.bvh_faces;
    C.M.n_vertices = S.n_vertices; C.M.n_poses = S.n_poses; C.M.bvh_ok = S.bvh_ok;
    C.objects = S.objects; C.n_parts = S.n_parts; C.zr = S.zr;
    C.pose = 0;   // the tables are staged: one pose (a ray with another pose_id is rejected below)
    C.prims = s_prims; C.parts = s_parts; C.bounds = s_bounds;
    C.lb_addr = smem_u32(s_lb + threadIdx.x);
    const unsigned sc = smem_u32(s_ls + threadIdx.x), pinfo = smem_u32(s_bounds + NBOUND * S.n_parts);
    const unsigned a_n = smem_u32(s_pn + threadIdx.x), a_lam = smem_u32(s_pi + threadIdx.x), a_seg = a_lam + 4u * LB_STRIDE;
    const unsigned full = 0xffffffffu;
    const int lane = threadIdx.x & 31;
    const long long n_tiles = (P.n + 31) / 32;
    Stats st; st.sdf = 0; st.tri = 0;
    unsigned n_int = 0, n_bad = 0, most = 0;
#pragma unroll 1
    for (;;) {
        long long tile = 0;
        if (lane == 0) tile = (long long)atomicAdd(&P.counters->tiles, 1ull);
        tile = __shfl_sync(full, tile, 0);
        if (tile >= n_tiles) break;
        const int64_t ri = tile * 32 + lane;
        if (ri < P.n) {
            // the ray as init_queue makes it: Ray(pos, dir, lambda) has n = 1 (Rays.jl:32-42)
            const int64_t di = P.dir_uniform ? 0 : ri;
            V3 pos = mk3(P.pos[3 * ri], P.pos[3 * ri + 1], P.pos[3 * ri + 2]);
            V3 dir = mk3(P.dir[3 * di], P.dir[3 * di + 1], P.dir[3 * di + 2]);
            int lam = P.lam ? P.lam[ri] : 0, pose = P.pose ? P.pose[ri] : 0;
            // an id outside the tables is parked (status ERROR, no segment) and counted; the call then returns BMO_EINVAL
            const bool bad = (unsigned)lam >= (unsigned)S.n_lambda || (unsigned)pose >= (unsigned)S.n_poses;
            if (bad) { lam = 0; pose = 0; n_bad++; }
            int hint = -1, nseg = 0, status = BMO_ST_ERROR;
            bool warn = false;
            SpotHit sp; sp.obj = -1; sp.x = sp.z = __longlong_as_double(0x7ff8000000000000ll);   // NaN until a Spotdetector is hit
            sts_f64(a_n, 1.0);
            sts_f32(a_lam, __int_as_float(lam));
            sts_f32(a_seg, __int_as_float(0));
    #pragma unroll 1
            while (!bad) {
                // one wave: tracing_step! (intersect_wave), then the outcome and interact3d (interact_body<0, *, true>)
                const int seg = __float_as_int(lds_f32(a_seg));
                Hit h; h.part = -1; h.t = INFINITY; h.n = mk3(0, 0, 0);
                const bool budget = seg + 1 < P.r_max;   // `while length(rays) < r_max` (System.jl:133)
                if (budget) h = tracing_step_lean(C, sc, C.lb_addr, pinfo, pos, dir, hint, st);
                int s = budget ? (h.part < 0 ? BMO_ST_MISS : BMO_ST_ACTIVE) : BMO_ST_RMAX;
                RayOut o;
                o.valid = false; o.err = false; o.warn = false; o.hint = -1;
                if (s == BMO_ST_ACTIVE) {
                    n_int++;
                    // the ray as the march left it in its scratch column (not carried through the march in registers)
                    pos = ls_load3(sc, LS_POS); dir = ls_load3(sc, LS_DIR);
                    const double rn = lds_f64(a_n);
                    const int lm = __float_as_int(lds_f32(a_lam));
                    const bmo_part& pt = s_parts[h.part];
                    const bmo_object& ob = S.objects[pt.object];
                    bool split = false;   // never set: the system has no beamsplitter
                    interact_plain(S, pt, ob, h.part, pos, dir, rn, h.t, h.n, lm, 0, o, split, sp);
                    if (!o.valid) s = BMO_ST_ABSORBED;
                    if (o.valid && o.err) s = BMO_ST_ERROR;
                    warn |= o.valid && o.warn;
                }
                if (s != BMO_ST_ACTIVE) { nseg = seg + 1; status = s; break; }
                pos = o.pos; dir = o.dir; hint = o.hint;
                sts_f64(a_n, o.n);
                sts_f32(a_seg, __int_as_float(seg + 1));
            }
            // the beam-table entry init_queue and the waves would have left (bit 8 of status: see interact_body)
            P.B.parent[ri] = -1; P.B.slot[ri] = -1; P.B.nseg[ri] = nseg; P.B.status[ri] = status | (warn ? 0x100 : 0);
            P.B.lam[ri] = lam; P.B.pose[ri] = pose;
            P.B.spot_obj[ri] = sp.obj; P.B.spot_xz[2 * ri] = sp.x; P.B.spot_xz[2 * ri + 1] = sp.z;
            most = max(most, (unsigned)nseg);
        }
    }
    unsigned sd = st.sdf, tr = st.tri;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        sd += __shfl_xor_sync(full, sd, o);
        tr += __shfl_xor_sync(full, tr, o);
        n_int += __shfl_xor_sync(full, n_int, o);
        n_bad += __shfl_xor_sync(full, n_bad, o);
        most = max(most, __shfl_xor_sync(full, most, o));
    }
    if (lane == 0) {
        if (sd) atomicAdd(&P.counters->sdf, (unsigned long long)sd);
        if (tr) atomicAdd(&P.counters->tri, (unsigned long long)tr);
        if (n_int) atomicAdd(&P.counters->interactions, (unsigned long long)n_int);
        if (n_bad) atomicAdd(&P.counters->bad_ids, (unsigned long long)n_bad);
        if (most) atomicMax(&P.counters->most_nseg, (unsigned long long)most);
    }
}

// ---- K2: exclusive scan of int32 counts with stride (single block, chunked) -----------------------
// in[i*stride + which] for which in [0, nwhich) -> out (long long), totals[which]
// Tiles of 1024 coalesced elements: warp shuffle scan, 32 warp totals scanned by warp 0, running carry.
__global__ void __launch_bounds__(1024) scan_counts(const int32_t* in, int64_t n, int stride, int nwhich, long long* out,
                                                    long long* totals) {
    __shared__ long long s_warp[32];
    __shared__ long long s_carry;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int w = 0; w < nwhich; w++) {
        if (threadIdx.x == 0) s_carry = 0;
        __syncthreads();
        for (int64_t base = 0; base < n; base += 1024) {
            const int64_t i = base + threadIdx.x;
            const long long v = i < n ? (long long)in[i * stride + w] : 0;
            long long x = v;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const long long y = __shfl_up_sync(0xffffffffu, x, o);
                if (lane >= o) x += y;
            }
            if (lane == 31) s_warp[warp] = x;
            __syncthreads();
            if (warp == 0) {
                long long t = s_warp[lane];
#pragma unroll
                for (int o = 1; o < 32; o <<= 1) {
                    const long long y = __shfl_up_sync(0xffffffffu, t, o);
                    if (lane >= o) t += y;
                }
                s_warp[lane] = t;   // inclusive totals of warps 0..lane
            }
            __syncthreads();
            const long long carry = s_carry;
            const long long excl = carry + (warp ? s_warp[warp - 1] : 0) + (x - v);
            if (i < n) out[i * nwhich + w] = excl;
            __syncthreads();
            if (threadIdx.x == 1023) s_carry = carry + s_warp[31];
            __syncthreads();
        }
        if (threadIdx.x == 0) totals[w] = s_carry;
        __syncthreads();
    }
}

// Large inputs: per-block local scan (1024 elements) + scan of the block sums + offset add.
__global__ void __launch_bounds__(1024) scan_local(const int32_t* in, int64_t n, long long* out, int32_t* blk_sum) {
    __shared__ long long s_warp[32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t i = (int64_t)blockIdx.x * 1024 + threadIdx.x;
    const long long v = i < n ? (long long)in[i] : 0;
    long long x = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const long long y = __shfl_up_sync(0xffffffffu, x, o); if (lane >= o) x += y; }
    if (lane == 31) s_warp[warp] = x;
    __syncthreads();
    if (warp == 0) {
        long long t = s_warp[lane];
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const long long y = __shfl_up_sync(0xffffffffu, t, o); if (lane >= o) t += y; }
        s_warp[lane] = t;
    }
    __syncthreads();
    if (i < n) out[i] = (warp ? s_warp[warp - 1] : 0) + (x - v);
    if (threadIdx.x == 0) blk_sum[blockIdx.x] = (int32_t)s_warp[31];
}
__global__ void scan_add(long long* out, int64_t n, const long long* blk_off) {
    const int64_t i = (int64_t)blockIdx.x * 1024 + threadIdx.x;
    if (i < n) out[i] += blk_off[blockIdx.x];
}

// ---- beamsplitter children: deterministic numbering in queue order ---------------------------------
struct SpawnParams {
    Queue scr, q;
    const int32_t* blk_cnt;
    const long long* blk_off;  // exclusive scan of blk_cnt
    BeamTab B;
    int64_t n_beams;           // beams that exist before this wave's spawns
    int64_t n_slots;           // queue units before this wave's spawns
    int32_t nf, mode, units, R;
};
__global__ void __launch_bounds__(256) spawn_children(const SpawnParams P) {
    const int b = blockIdx.x;
    const int cnt = P.blk_cnt[b];
    if (cnt == 0) return;
    const long long off = P.blk_off[b];
    const int64_t ss = P.scr.cap, qs = P.q.cap;
    const int R = P.R;
    for (int j = threadIdx.x; j < cnt * 2 * R; j += blockDim.x) {
        const int ls = j / (2 * R), k = (j / R) & 1, r = j % R;
        const int64_t si = (((int64_t)b * P.units + ls) * 2 + k) * R + r;
        const long long rank = off + ls;
        const int32_t* iq = P.scr.i;
        const int64_t du = (k == 0) ? (int64_t)iq[I_PUNIT * ss + si] : P.n_slots + rank;
        const int64_t di = du * R + r;
        for (int f = 0; f < P.nf; f++) P.q.d[f * qs + di] = P.scr.d[f * ss + si];
        const int parent = iq[I_BEAM * ss + si];
        const int lam = iq[I_LAM * ss + si], pose = iq[I_POSE * ss + si];
        const int beam = (int)(P.n_beams + 2 * rank + k);
        if (r == 0) {
            P.B.parent[beam] = parent; P.B.slot[beam] = k; P.B.nseg[beam] = 0; P.B.status[beam] = BMO_ST_ACTIVE;
            P.B.lam[beam] = lam; P.B.pose[beam] = pose;
            if (P.mode == 2) {
                P.B.w0[beam] = P.scr.d[(F_X0 + 3) * ss + si];
                P.B.e0[2 * beam] = P.scr.d[(F_X0 + 4) * ss + si];
                P.B.e0[2 * beam + 1] = P.scr.d[(F_X0 + 5) * ss + si];
                P.B.plen[beam] = P.scr.d[(F_X0 + 6) * ss + si];
                P.B.popl[beam] = P.scr.d[(F_X0 + 7) * ss + si];
            }
        }
        P.B.spot_obj[(int64_t)beam * R + r] = -1;
        P.B.spot_xz[2 * ((int64_t)beam * R + r)] = P.B.spot_xz[2 * ((int64_t)beam * R + r) + 1] = __longlong_as_double(0x7ff8000000000000ll);
        int32_t* nq = P.q.i;
        nq[I_LAM * qs + di] = lam;
        nq[I_HINT * qs + di] = -1;
        nq[I_BEAM * qs + di] = beam;
        nq[I_SEG * qs + di] = 0;
        nq[I_POSE * qs + di] = pose;
        nq[I_RETR * qs + di] = iq[I_RETR * ss + si];
    }
}

// ---- K3: queue compaction (HBM-bound) ----------------------------------------------------------------
// Dead slots are squeezed out when they make up more than half of the queue: the live units move to the front of the other
// queue buffer, order preserved.
constexpr int CBLOCK = 256;
// One cooperative launch (one CTA slice per resident block, one contiguous sub-slice per warp): every warp counts
// the live units of its sub-slice, grid-wide barrier, own offset = sum of the lower blocks' counts (a few hundred values, L2
// hits) + the lower warps of the block, then every warp scatters its sub-slice on its own, two 32-slot rows per step, all loads
// of both rows issued before the first store -- no block barrier inside the copy loop, so the 8 warps of a block and the two
// rows of a step keep independent DRAM requests in flight (the previous version walked 256-slot rows between two barriers and was
// bound by the latency of one row at a time: 36 % of the HBM peak).  The alive flags are read twice (the second time from L2),
// every surviving ray is read and written once; order is preserved (sub-slices are contiguous and ordered).
template <int NF>
BMO_D void compact_copy_unit(const Queue& src, const Queue& dst, int64_t ss, int64_t ds, int64_t si, int64_t di) {
    double v[NF];
    int w[NI_Q];
#pragma unroll
    for (int k = 0; k < NF; k++) v[k] = src.d[k * ss + si];
#pragma unroll
    for (int f = 0; f < NI_Q; f++) w[f] = src.i[f * ss + si];
#pragma unroll
    for (int k = 0; k < NF; k++) dst.d[k * ds + di] = v[k];
#pragma unroll
    for (int f = 0; f < NI_Q; f++) dst.i[f * ds + di] = w[f];
}
__global__ void __launch_bounds__(CBLOCK) compact_fused(Queue src, Queue dst, int64_t n_slots, int64_t per, int R, int nf, int32_t* blk_cnt) {
    namespace cg = cooperative_groups;
    constexpr int NW = CBLOCK / 32;
    __shared__ int s_w[NW];
    __shared__ long long s_red[NW];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t ss = src.cap, ds = dst.cap;
    const int64_t lo = (int64_t)blockIdx.x * per, hi = min(lo + per, n_slots);
    const int64_t wper = per / NW;                         // per is a multiple of CBLOCK: whole 32-slot rows per warp
    const int64_t wlo = min(lo + warp * wper, hi), whi = min(wlo + wper, hi);
    const int32_t* alive = src.i + I_BEAM * ss;
    int cnt = 0;
    for (int64_t u = wlo + lane; u < whi; u += 32) cnt += alive[u * R] >= 0;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
    if (lane == 0) s_w[warp] = cnt;
    __syncthreads();
    if (threadIdx.x == 0) {
        int a = 0;
        for (int k = 0; k < NW; k++) a += s_w[k];
        blk_cnt[blockIdx.x] = a;
    }
    cg::this_grid().sync();
    long long part = 0;
    for (int k = threadIdx.x; k < (int)blockIdx.x; k += CBLOCK) part += __ldcg(blk_cnt + k);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) part += __shfl_xor_sync(0xffffffffu, part, o);
    if (lane == 0) s_red[warp] = part;
    __syncthreads();
    long long off = 0;
    for (int k = 0; k < NW; k++) off += s_red[k];
    for (int k = 0; k < warp; k++) off += s_w[k];
    for (int64_t base = wlo; base < whi; base += 64) {
        const int64_t u0 = base + lane, u1 = base + 32 + lane;
        const bool l0 = u0 < whi && alive[u0 * R] >= 0, l1 = u1 < whi && alive[u1 * R] >= 0;
        const unsigned b0 = __ballot_sync(0xffffffffu, l0), b1 = __ballot_sync(0xffffffffu, l1);
        const int64_t d0 = off + __popc(b0 & lanemask_lt()), d1 = off + __popc(b0) + __popc(b1 & lanemask_lt());
        off += __popc(b0) + __popc(b1);
        if (R == 1 && nf == 7) {                            // plain rays: both rows' loads in flight before the stores
            double v0[7], v1[7];
            int w0[NI_Q], w1[NI_Q];
            if (l0) {
#pragma unroll
                for (int k = 0; k < 7; k++) v0[k] = src.d[k * ss + u0];
#pragma unroll
                for (int f = 0; f < NI_Q; f++) w0[f] = src.i[f * ss + u0];
            }
            if (l1) {
#pragma unroll
                for (int k = 0; k < 7; k++) v1[k] = src.d[k * ss + u1];
#pragma unroll
                for (int f = 0; f < NI_Q; f++) w1[f] = src.i[f * ss + u1];
            }
            if (l0) {
#pragma unroll
                for (int k = 0; k < 7; k++) dst.d[k * ds + d0] = v0[k];
#pragma unroll
                for (int f = 0; f < NI_Q; f++) dst.i[f * ds + d0] = w0[f];
            }
            if (l1) {
#pragma unroll
                for (int k = 0; k < 7; k++) dst.d[k * ds + d1] = v1[k];
#pragma unroll
                for (int f = 0; f < NI_Q; f++) dst.i[f * ds + d1] = w1[f];
            }
        } else {
            for (int r = 0; r < R; r++) {
                if (nf == 13) {
                    if (l0) compact_copy_unit<13>(src, dst, ss, ds, u0 * R + r, d0 * R + r);
                    if (l1) compact_copy_unit<13>(src, dst, ss, ds, u1 * R + r, d1 * R + r);
                } else if (nf == 10) {
                    if (l0) compact_copy_unit<10>(src, dst, ss, ds, u0 * R + r, d0 * R + r);
                    if (l1) compact_copy_unit<10>(src, dst, ss, ds, u1 * R + r, d1 * R + r);
                } else {
                    if (l0) compact_copy_unit<7>(src, dst, ss, ds, u0 * R + r, d0 * R + r);
                    if (l1) compact_copy_unit<7>(src, dst, ss, ds, u1 * R + r, d1 * R + r);
                }
            }
        }
    }
}

// ---- init / gather ---------------------------------------------------------------------------------
struct InitParams {
    Queue q;
    int64_t n, beam0;   // beam0: global id of this sub-batch's first root beam
    int mode;
    const double *pos, *dir, *E0, *grays, *w0, *ge0;
    const int32_t *lam, *pose;
    BeamTab B;
    int32_t retrace, pad;   // retrace: root beam g re-validates beam g of the previous solution
    int32_t n_lambda, n_poses;   // valid ranges of lambda_id / pose_id
    DevCounters* counters;
    int32_t dir_uniform, pad2;   // BMO_UNIFORM_DIR: dir holds one direction shared by every ray of the bundle
};
__global__ void init_queue(const InitParams P) {
    const int R = P.mode == 2 ? 3 : 1;
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= P.n * R) return;
    const int64_t u = i / R;
    const int r = (int)(i % R);
    const int64_t s = P.q.cap;
    double* d = P.q.d;
    if (P.mode == 2) {
        const double* g = P.grays + (u * 3 + r) * 6;
        d[F_PX * s + i] = g[0]; d[F_PY * s + i] = g[1]; d[F_PZ * s + i] = g[2];
        d[F_DX * s + i] = g[3]; d[F_DY * s + i] = g[4]; d[F_DZ * s + i] = g[5];
        d[F_X0 * s + i] = 0; d[(F_X0 + 1) * s + i] = 0; d[(F_X0 + 2) * s + i] = 0;
    } else {
        d[F_PX * s + i] = P.pos[3 * u]; d[F_PY * s + i] = P.pos[3 * u + 1]; d[F_PZ * s + i] = P.pos[3 * u + 2];
        const int64_t du = P.dir_uniform ? 0 : u;
        d[F_DX * s + i] = P.dir[3 * du]; d[F_DY * s + i] = P.dir[3 * du + 1]; d[F_DZ * s + i] = P.dir[3 * du + 2];
        if (P.mode == 1)
            for (int k = 0; k < 6; k++) d[(F_X0 + k) * s + i] = P.E0[6 * u + k];
    }
    d[F_N * s + i] = 1.0;  // Ray(pos, dir, lambda): n = 1 (Rays.jl:32-42)
    int32_t* q = P.q.i;
    int lam = P.lam ? P.lam[u] : 0, pose = P.pose ? P.pose[u] : 0;
    const int64_t g = P.beam0 + u;   // global beam id; inputs are this sub-batch's slices, tables are global
    // An id outside the tables would index n_table / lambdas / the pose-stacked tables out of bounds: the ray is parked
    // (dead slot, status ERROR) and counted; the trace call then returns BMO_EINVAL instead of faulting the context.
    const bool bad = (unsigned)lam >= (unsigned)P.n_lambda || (unsigned)pose >= (unsigned)P.n_poses;
    if (bad) { lam = 0; pose = 0; if (r == 0) atomicAdd(&P.counters->bad_ids, 1ull); }
    q[I_LAM * s + i] = lam; q[I_HINT * s + i] = -1; q[I_BEAM * s + i] = bad ? -1 : (int)g; q[I_SEG * s + i] = 0; q[I_POSE * s + i] = pose;
    q[I_RETR * s + i] = P.retrace ? (int)g : -1;
    P.B.spot_obj[g * R + r] = -1;
    P.B.spot_xz[2 * (g * R + r)] = P.B.spot_xz[2 * (g * R + r) + 1] = __longlong_as_double(0x7ff8000000000000ll);   // NaN until a Spotdetector is hit
    if (r == 0) {
        P.B.parent[g] = -1; P.B.slot[g] = -1; P.B.nseg[g] = 0; P.B.status[g] = bad ? BMO_ST_ERROR : BMO_ST_ACTIVE; P.B.lam[g] = lam; P.B.pose[g] = pose;
        if (P.mode == 2) { P.B.w0[g] = P.w0[u]; P.B.e0[2 * g] = P.ge0[2 * u]; P.B.e0[2 * g + 1] = P.ge0[2 * u + 1]; P.B.plen[g] = 0; P.B.popl[g] = 0; }
    }
}
// ---- retrace: roots and children of the previous solution --------------------------------------------
// The root beams of a retrace call start from the first stored ray of the previous solution's roots
// (retrace_system! keeps ray 1 as it is, System.jl:198).
struct PrevRoots {
    const double* seg_d; const long long* first_seg; int64_t rows; int nsd;   // previous segment table, row records [rows][nsd]
    const int32_t *lam, *pose; const double *w0, *e0;
    int64_t n; int mode;
    double *pos, *dir, *E0, *grays, *ow0, *oe0; int32_t *olam, *opose;
};
__global__ void gather_prev_roots(const PrevRoots P) {
    const int R = P.mode == 2 ? 3 : 1;
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= P.n * R) return;
    const int64_t b = i / R;
    const int r = (int)(i % R);
    const int64_t row = P.first_seg[b] * R + r;
    double v[6];
    for (int k = 0; k < 6; k++) v[k] = P.seg_d[(size_t)row * P.nsd + (S_PX + k)];
    if (P.mode == 2) { for (int k = 0; k < 6; k++) P.grays[i * 6 + k] = v[k]; }
    else {
        for (int k = 0; k < 3; k++) { P.pos[3 * b + k] = v[k]; P.dir[3 * b + k] = v[3 + k]; }
        if (P.mode == 1) for (int k = 0; k < 6; k++) P.E0[6 * b + k] = P.seg_d[(size_t)row * P.nsd + (S_E0 + k)];
    }
    if (r == 0) {
        P.olam[b] = P.lam[b]; P.opose[b] = P.pose[b];
        if (P.mode == 2) { P.ow0[b] = P.w0[b]; P.oe0[2 * b] = P.e0[2 * b]; P.oe0[2 * b + 1] = P.e0[2 * b + 1]; }
    }
}
// child[2 * parent + slot] = beam (children are numbered after the roots; slot 0 transmitted, 1 reflected)
__global__ void build_child_table(const int32_t* parent, const int32_t* slot, int64_t n_roots, int64_t n_beams, int32_t* child) {
    const int64_t i = n_roots + (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_beams) return;
    const int p = parent[i], k = slot[i];
    if (p >= 0 && (k == 0 || k == 1)) child[2 * (int64_t)p + k] = (int32_t)i;
}

// wave-major records -> row records of the beam-major table.  A warp takes 32 consecutive slots of the wave: the fields are read
// plane by plane (coalesced), transposed through shared memory, and written so that consecutive lanes store consecutive doubles
// of a row record (runs of NSD doubles): ~3 rows per store instruction instead of one 8-byte piece of 32 different rows.
template <int NSD>
__global__ void __launch_bounds__(256) gather_segments(WaveBuf w, int R, const long long* first_seg, double* seg_d, int32_t* seg_part) {
    __shared__ double s_val[8][32 * NSD];
    __shared__ long long s_row[8][32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x;
    const bool valid = i < w.count && w.beam[i] >= 0;
    long long row = -1;
    if (valid) {
        row = (first_seg[w.beam[i]] + w.seg[i]) * R + (int)(i % R);
        seg_part[row] = w.part[i];
#pragma unroll
        for (int f = 0; f < NSD; f++) s_val[warp][lane * NSD + f] = w.d[(size_t)f * w.count + i];
    }
    s_row[warp][lane] = row;
    __syncwarp();
#pragma unroll
    for (int k = 0; k < NSD; k++) {
        const int flat = k * 32 + lane, ray = flat / NSD, field = flat - ray * NSD;
        const long long rr = s_row[warp][ray];
        if (rr >= 0) seg_d[(size_t)rr * NSD + field] = s_val[warp][flat];
    }
}

}  // namespace bmo

using namespace bmo;

// =================================================================================================
// host side
// =================================================================================================
// (exported functions get C linkage from their declarations in include/bmo.h)

const char* bmo_last_error(void) { return g_last_error.c_str(); }

int32_t bmo_init(int32_t device, bmo_ctx** out) {
    if (!out) return fail(BMO_EINVAL, "bmo_init: ctx is NULL");
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0)
        return fail(BMO_ECUDA, std::string("bmo_init: no CUDA device (") + cudaGetErrorString(e) + "); libbmo has no CPU fallback");
    if (device < 0 || device >= ndev) return fail(BMO_EINVAL, "bmo_init: bad device index");
    BMO_CUDA(cudaSetDevice(device));
    cudaDeviceProp prop;
    BMO_CUDA(cudaGetDeviceProperties(&prop, device));
    if (prop.major < 10) return fail(BMO_ECUDA, std::string("bmo_init: ") + prop.name + " is not an sm_100-class device");
    std::unique_ptr<bmo_ctx, FreeWith<bmo_shutdown>> c(new bmo_ctx());
    c->device = device;
    c->sm_count = prop.multiProcessorCount;
    BMO_CUDA(cudaEventCreate(&c->ev0));
    BMO_CUDA(cudaEventCreate(&c->ev1));
    BMO_CUDA(cudaEventCreate(&c->evk0)); BMO_CUDA(cudaEventCreate(&c->evk1));
    BMO_CUDA(cudaEventCreate(&c->evs0)); BMO_CUDA(cudaEventCreate(&c->evs1));
    BMO_CUDA(cudaMalloc((void**)&c->d_counters, sizeof(DevCounters)));
    BMO_CUDA(cudaMemset(c->d_counters, 0, sizeof(DevCounters)));
    BMO_CUDA(cudaMalloc((void**)&c->d_totals, 4 * sizeof(long long)));
    BMO_CUDA(cudaMallocHost((void**)&c->h_totals, 8 * 10 * sizeof(long long)));   // scans + 8 sub-batch slots + the device counters
    cudaMemPool_t pool;
    BMO_CUDA(cudaDeviceGetDefaultMemPool(&pool, device));
    uint64_t thr = UINT64_MAX;  // keep freed blocks cached: the wave loop reuses them every call
    BMO_CUDA(cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &thr));
    *out = c.release();
    return BMO_OK;
}
int32_t bmo_shutdown(bmo_ctx* c) {
    if (!c) return BMO_OK;
    cudaSetDevice(c->device);
    cudaStreamSynchronize(c->stream);
    BigBlocks::of_device().drop_parked();
    cudaFree(c->d_counters); cudaFree(c->d_totals); cudaFreeHost(c->h_totals);
    std::vector<cudaEvent_t> evs = c->ev_pool;
    evs.insert(evs.end(), {c->ev0, c->ev1, c->evk0, c->evk1, c->evs0, c->evs1});
    for (cudaEvent_t e : evs)
        if (e) cudaEventDestroy(e);   // (a context that bmo_init gave up on may lack some)
    for (cudaStream_t s : c->aux_streams) cudaStreamDestroy(s);
    delete c;
    return BMO_OK;
}
int32_t bmo_trim(bmo_ctx* c, int64_t* released) {
    if (!c) return fail(BMO_EINVAL, "ctx NULL");
    BMO_CUDA(cudaSetDevice(c->device));
    BMO_CUDA(cudaStreamSynchronize(c->stream));
    const size_t bytes = BigBlocks::of_device().drop_parked();
    cudaMemPool_t pool;
    if (cudaDeviceGetDefaultMemPool(&pool, c->device) == cudaSuccess) cudaMemPoolTrimTo(pool, 0);
    c->pool_slack = 0;        // the slack bmo_retrace grew the pool by is gone with the trim
    if (released) *released = (int64_t)bytes;
    return BMO_OK;
}
int32_t bmo_set_stream(bmo_ctx* c, void* s) { if (!c) return fail(BMO_EINVAL, "ctx NULL"); c->stream = (cudaStream_t)s; return BMO_OK; }
int32_t bmo_counters_get(bmo_ctx* c, bmo_counters* o) {
    if (!c || !o) return fail(BMO_EINVAL, "bmo_counters_get: NULL");
    BMO_CUDA(cudaSetDevice(c->device));
    DevCounters h;
    BMO_CUDA(cudaStreamSynchronize(c->stream));
    BMO_CUDA(cudaMemcpy(&h, c->d_counters, sizeof(h), cudaMemcpyDeviceToHost));
    o->interactions = (int64_t)h.interactions; o->sdf_evals = (int64_t)h.sdf; o->tri_tests = (int64_t)h.tri;
    o->waves = c->waves; o->kernel_launches = c->launches; o->px_beamlets = c->px_beamlets;
    o->trace_ms = c->trace_ms; o->pd_ms = c->pd_ms;
    o->trace_step_ms = c->k1_ms; o->trace_step_launches = c->k1_launches; o->scatter_ms = c->k3_ms; o->scatter_bytes = c->k3_bytes;
    o->pd_field_ms = c->k4_ms;
    o->psf_pairs = c->psf_pairs; o->psf_ms = c->psf_ms;
    return BMO_OK;
}
int32_t bmo_counters_reset(bmo_ctx* c) {
    if (!c) return fail(BMO_EINVAL, "ctx NULL");
    BMO_CUDA(cudaSetDevice(c->device));
    BMO_CUDA(cudaStreamSynchronize(c->stream));
    BMO_CUDA(cudaMemset(c->d_counters, 0, sizeof(DevCounters)));
    c->waves = c->launches = c->px_beamlets = 0; c->psf_pairs = 0; c->psf_ms = 0;
    c->k1_ms = c->k3_ms = c->k3_bytes = c->k4_ms = 0; c->k1_launches = 0; c->interactions_seen = 0; c->bad_ids_seen = 0;
    return BMO_OK;
}

// ---- system upload ------------------------------------------------------------------------------
static int32_t validate_tables(const bmo_tables* t) {
    if (!t) return fail(BMO_EINVAL, "tables NULL");
    if (t->n_objects <= 0 || t->n_parts <= 0) return fail(BMO_EINVAL, "system has no objects");
    if (t->n_lambda <= 0 || !t->lambdas) return fail(BMO_EINVAL, "n_lambda must be >= 1");
    for (int p = 0; p < t->n_parts; p++) {
        const bmo_part& pt = t->parts[p];
        if (pt.object < 0 || pt.object >= t->n_objects) return fail(BMO_EINVAL, "part.object out of range");
        if (pt.shape_kind == BMO_SHAPE_SDF) {
            if (pt.first < 0 || pt.count <= 0 || pt.first + pt.count > t->n_prims) return fail(BMO_EINVAL, "part prim range out of bounds");
        } else if (pt.shape_kind == BMO_SHAPE_MESH) {
            if (pt.first < 0 || pt.first >= t->n_meshes) return fail(BMO_EINVAL, "part mesh index out of range");
        } else return fail(BMO_EINVAL, "unknown shape kind");
        if (pt.n_row >= t->n_rows) return fail(BMO_EINVAL, "part.n_row out of range");
        if (pt.n_row >= 0 && !t->n_table) return fail(BMO_EINVAL, "part.n_row set but n_table is NULL");
        if (pt.role < BMO_ROLE_SINGLE || pt.role > BMO_ROLE_COATING) return fail(BMO_EINVAL, "unknown part role");
    }
    for (int p = 0; p < t->n_prims; p++) {
        const int ty = t->prims[p].type;
        if (ty < BMO_PRIM_PLANO || ty > BMO_PRIM_CONCAVE_ACYL) return fail(BMO_EINVAL, "unknown primitive type");
    }
    for (int o = 0; o < t->n_objects; o++) {
        const bmo_object& ob = t->objects[o];
        if (ob.first_part < 0 || ob.n_parts <= 0 || ob.first_part + ob.n_parts > t->n_parts) return fail(BMO_EINVAL, "object part range out of bounds");
        const int need = ob.kind == BMO_OBJ_CUBE_BS ? 3 : ((ob.kind == BMO_OBJ_PLATE_BS || ob.kind == BMO_OBJ_DOUBLET) ? 2 : 1);
        if (ob.n_parts != need) return fail(BMO_EINVAL, "object has the wrong number of parts for its kind");
        if (ob.kind < BMO_OBJ_REFRACTIVE || ob.kind > BMO_OBJ_POLFILTER) return fail(BMO_EINVAL, "unknown object kind");
        // every part whose interaction reads n_table needs a row: lens / prism, both lenses of a doublet, the substrate of a
        // plate splitter, both prisms of a cube splitter (interact_wave: n_of_hit, the children's n of CUBE_BS / PLATE_BS)
        const int n_refr = ob.kind == BMO_OBJ_REFRACTIVE ? 1 : (ob.kind == BMO_OBJ_DOUBLET || ob.kind == BMO_OBJ_CUBE_BS) ? 2 : (ob.kind == BMO_OBJ_PLATE_BS ? 1 : 0);
        for (int k = 0; k < n_refr; k++)
            if (t->parts[ob.first_part + k].n_row < 0) return fail(BMO_EINVAL, "refractive part without a row of n_table (n_row < 0)");
        if (ob.kind == BMO_OBJ_POLFILTER && (!t->jones || ob.pd_n < 0 || ob.pd_n >= t->n_jones)) return fail(BMO_EINVAL, "PolarizationFilter without a row of tables.jones");
    }
    for (int m = 0; m < t->n_meshes; m++) {
        const bmo_mesh& me = t->meshes[m];
        if (me.first_vertex < 0 || me.first_vertex + me.n_vertices > t->n_vertices || me.first_face < 0 || me.first_face + me.n_faces > t->n_faces)
            return fail(BMO_EINVAL, "mesh range out of bounds");
        for (int64_t f = 3 * me.first_face; f < 3 * (me.first_face + me.n_faces); f++)
            if (t->faces[f] < 0 || t->faces[f] >= me.n_vertices) return fail(BMO_EINVAL, "face vertex index out of range");
    }
    for (int p = 0; p < t->n_prims; p++) {
        const bmo_prim& pr = t->prims[p];
        if (pr.type >= BMO_PRIM_CONVEX_ASPH && (!t->ext || pr.ext_first < 0 || pr.ext_count < 7 || (int64_t)pr.ext_first + pr.ext_count > t->n_ext))
            return fail(BMO_EINVAL, "aspheric primitive without a parameter block in tables.ext");
    }
    return BMO_OK;
}

// bit 0 of bmo_prim.reserved: transposed_orientation is exactly the identity (w2s_f skips the products)
static int32_t prim_flags(const bmo_prim& p) {
    static const double I[9] = {1, 0, 0, 0, 1, 0, 0, 0, 1};
    for (int k = 0; k < 9; k++) if (p.tdir[k] != I[k]) return 0;
    return 1;
}

// aspheric primitives carry the device address of their parameter block in par[0] (see asph_block, bmo_geom.cuh)
// bit 1 of the first prim record of an SDF part: the union has cylindrical / aspheric members (part_intersect, bmo_geom.cuh)
static void flag_rare_parts(bmo_prim* p, size_t n_prims_per_pose, size_t n_poses, const std::vector<bmo_part>& parts) {
    for (size_t q = 0; q < n_poses; q++)
        for (const bmo_part& pt : parts) {
            if (pt.shape_kind != BMO_SHAPE_SDF) continue;
            bool rare = false;
            for (int k = 0; k < pt.count; k++) rare |= p[q * n_prims_per_pose + pt.first + k].type >= BMO_PRIM_CONVEX_CYL;
            if (rare) p[q * n_prims_per_pose + pt.first].reserved |= 2;
        }
}
// every SDF part is a union of at most 4 plain primitives (no meniscus frame, no cylindrical / aspheric member) and every mesh
// is small enough to have no BVH: the LEAN builds of the trace kernels apply (bmo_geom.cuh: LeanBounds, mesh_intersect_small)
static bool system_is_lean(const std::vector<bmo_prim>& prims, const std::vector<bmo_part>& parts, const std::vector<MeshView>& meshes) {
    for (const bmo_part& pt : parts) {
        if (pt.shape_kind != BMO_SHAPE_SDF) continue;
        if (pt.count < 1 || pt.count > 4) return false;
        for (int k = 0; k < pt.count; k++) {
            const int ty = prims[pt.first + k].type;
            if (ty == BMO_PRIM_MENISCUS || ty >= BMO_PRIM_CONVEX_CYL) return false;
        }
    }
    for (const MeshView& mv : meshes) if (mv.n_nodes != 0) return false;
    return true;
}
static void patch_asph(bmo_prim* p, size_t n, const double* d_ext) {
    for (size_t i = 0; i < n; i++)
        if (p[i].type >= BMO_PRIM_CONVEX_ASPH && p[i].type <= BMO_PRIM_CONCAVE_ACYL) {
            const unsigned long long a = (unsigned long long)(uintptr_t)(d_ext + p[i].ext_first);
            std::memcpy(&p[i].par[0], &a, sizeof(double));
        }
}

int32_t bmo_system_upload(bmo_ctx* ctx, const bmo_tables* t, bmo_sys** out) {
    NvtxRange nvtx_("bmo_system_upload");
    if (!ctx || !out) return fail(BMO_EINVAL, "bmo_system_upload: NULL argument");
    int32_t rc = validate_tables(t);
    if (rc) return rc;
    BMO_CUDA(cudaSetDevice(ctx->device));
    std::unique_ptr<bmo_sys, FreeWith<bmo_system_free>> s(new bmo_sys());
    s->ctx = ctx;
    s->prims.assign(t->prims, t->prims + t->n_prims);
    for (auto& pr : s->prims) pr.reserved = prim_flags(pr);
    s->parts.assign(t->parts, t->parts + t->n_parts);
    s->objects.assign(t->objects, t->objects + t->n_objects);
    s->lambdas.assign(t->lambdas, t->lambdas + t->n_lambda);
    s->n_vertices = t->n_vertices; s->n_faces = t->n_faces;
    s->h_vertices.assign(t->vertices, t->vertices + 3 * t->n_vertices);
    // meshes + BVH
    std::vector<BvhNode> nodes;
    std::vector<int32_t> order(std::max<int64_t>(t->n_faces, 1), 0);
    for (int m = 0; m < t->n_meshes; m++) {
        const bmo_mesh& me = t->meshes[m];
        MeshView mv{};
        mv.first_vertex = me.first_vertex; mv.n_vertices = me.n_vertices; mv.first_face = me.first_face; mv.n_faces = me.n_faces;
        mv.f32 = me.f32;
        mv.first_node = (int64_t)nodes.size(); mv.n_nodes = 0;
        if (me.n_faces > 16) {
            BvhBuild bb;
            bvh_build(t->vertices + 3 * me.first_vertex, t->faces + 3 * me.first_face, me.n_faces, bb);
            mv.n_nodes = (int64_t)bb.nodes.size();
            nodes.insert(nodes.end(), bb.nodes.begin(), bb.nodes.end());
            std::copy(bb.order.begin(), bb.order.end(), order.begin() + me.first_face);
        }
        s->meshes.push_back(mv);
    }
    // detector poses + bounds (pose 0)
    s->h_detpose.assign((size_t)12 * t->n_objects, 0.0);
    for (int o = 0; o < t->n_objects; o++) {
        for (int k = 0; k < 3; k++) s->h_detpose[12 * o + k] = t->objects[o].pos[k];
        for (int k = 0; k < 9; k++) s->h_detpose[12 * o + 3 + k] = t->objects[o].dir[k];
    }
    s->h_bounds.assign((size_t)NBOUND * t->n_parts, 0.0);
    for (int p = 0; p < t->n_parts; p++)
        for (int k = 0; k < NBOUND; k++) s->h_bounds[NBOUND * p + k] = t->parts[p].bound[k];
    std::vector<double> ntab(t->n_table, t->n_table + (size_t)std::max(t->n_rows, 0) * t->n_lambda);
    if (t->n_ext > 0 && (rc = upload(s->d_ext, t->ext, (size_t)t->n_ext))) return rc;
    patch_asph(s->prims.data(), s->prims.size(), s->d_ext.get());
    flag_rare_parts(s->prims.data(), s->prims.size(), 1, s->parts);
    for (const bmo_prim& pr : s->prims) s->has_rare |= pr.type >= BMO_PRIM_CONVEX_CYL;
    s->all_lean = system_is_lean(s->prims, s->parts, s->meshes);
    if ((rc = upload(s->d_prims, s->prims.data(), s->prims.size()))) return rc;
    if ((rc = upload(s->d_parts, s->parts.data(), s->parts.size()))) return rc;
    if ((rc = upload(s->d_objects, s->objects.data(), s->objects.size()))) return rc;
    if ((rc = upload(s->d_meshes, s->meshes.data(), s->meshes.size()))) return rc;
    if ((rc = upload(s->d_vertices, s->h_vertices.data(), s->h_vertices.size()))) return rc;
    if ((rc = upload(s->d_faces, t->faces, (size_t)3 * t->n_faces))) return rc;
    if ((rc = upload(s->d_nodes, nodes.data(), nodes.size()))) return rc;
    if ((rc = upload(s->d_bvh_faces, order.data(), (size_t)t->n_faces))) return rc;
    if ((rc = upload(s->d_ntable, ntab.data(), ntab.size()))) return rc;
    if ((rc = upload(s->d_bounds, s->h_bounds.data(), s->h_bounds.size()))) return rc;
    if ((rc = upload(s->d_detpose, s->h_detpose.data(), s->h_detpose.size()))) return rc;
    if ((rc = upload(s->d_lambdas, s->lambdas.data(), s->lambdas.size()))) return rc;
    if (t->n_jones > 0 && (rc = upload(s->d_jones, t->jones, (size_t)10 * t->n_jones))) return rc;
    SysView& v = s->view;
    v.prims = s->d_prims.get(); v.parts = s->d_parts.get(); v.objects = s->d_objects.get(); v.meshes = s->d_meshes.get();
    v.vertices = s->d_vertices.get(); v.faces = s->d_faces.get(); v.nodes = s->d_nodes.get(); v.bvh_faces = s->d_bvh_faces.get();
    v.n_table = s->d_ntable.get(); v.bounds = s->d_bounds.get(); v.det_pose = s->d_detpose.get(); v.lambdas = s->d_lambdas.get();
    v.jones = s->d_jones.get(); v.ext = s->d_ext.get();
    v.n_prims = t->n_prims; v.n_parts = t->n_parts; v.n_objects = t->n_objects; v.n_meshes = t->n_meshes;
    v.n_lambda = t->n_lambda; v.n_poses = 1; v.bvh_ok = 1; v.zr = t->norm_zero_rule; v.n_vertices = t->n_vertices;
    v.n_system = t->n_system;
    *out = s.release();
    return BMO_OK;
}
int32_t bmo_system_free(bmo_sys* s) {
    if (!s) return BMO_OK;
    cudaSetDevice(s->ctx->device);
    cudaStreamSynchronize(s->ctx->stream);
    delete s;   // the device tables go with it
    return BMO_OK;
}
int32_t bmo_system_set_poses(bmo_sys* s, int32_t n_poses, const bmo_prim* prims, const double* vertices, const double* bounds,
                             const double* det_pos, const double* det_dir) {
    if (!s || n_poses < 1) return fail(BMO_EINVAL, "bmo_system_set_poses: bad arguments");
    BMO_CUDA(cudaSetDevice(s->ctx->device));
    BMO_CUDA(cudaStreamSynchronize(s->ctx->stream));
    const size_t np = (size_t)n_poses;
    // the new tables replace the live ones only once all of them are on the device
    DevTable<bmo_prim> d_prims; DevTable<double> d_vertices, d_bounds, d_detpose;
    int32_t rc;
    if (n_poses == 1 && !prims) {  // restore the uploaded tables
        if ((rc = upload(d_prims, s->prims.data(), s->prims.size()))) return rc;
        if ((rc = upload(d_vertices, s->h_vertices.data(), s->h_vertices.size()))) return rc;
        if ((rc = upload(d_bounds, s->h_bounds.data(), s->h_bounds.size()))) return rc;
        if ((rc = upload(d_detpose, s->h_detpose.data(), s->h_detpose.size()))) return rc;
    } else {
        if (!prims || !bounds || (!vertices && s->n_vertices > 0) || !det_pos || !det_dir) return fail(BMO_EINVAL, "bmo_system_set_poses: NULL table");
        std::vector<bmo_prim> pp(prims, prims + np * s->prims.size());
        for (auto& pr : pp) pr.reserved = prim_flags(pr);
        patch_asph(pp.data(), pp.size(), s->d_ext.get());
        flag_rare_parts(pp.data(), s->prims.size(), np, s->parts);
        if ((rc = upload(d_prims, pp.data(), pp.size()))) return rc;
        if ((rc = upload(d_vertices, vertices, np * 3 * (size_t)s->n_vertices))) return rc;
        if ((rc = upload(d_bounds, bounds, np * NBOUND * s->parts.size()))) return rc;
        std::vector<double> dp(np * 12 * s->objects.size());
        for (size_t i = 0; i < np * s->objects.size(); i++) {
            for (int k = 0; k < 3; k++) dp[12 * i + k] = det_pos[3 * i + k];
            for (int k = 0; k < 9; k++) dp[12 * i + 3 + k] = det_dir[9 * i + k];
        }
        if ((rc = upload(d_detpose, dp.data(), dp.size()))) return rc;
    }
    s->d_prims = std::move(d_prims); s->d_vertices = std::move(d_vertices); s->d_bounds = std::move(d_bounds); s->d_detpose = std::move(d_detpose);
    SysView& v = s->view;
    v.prims = s->d_prims.get(); v.vertices = s->d_vertices.get(); v.bounds = s->d_bounds.get(); v.det_pose = s->d_detpose.get();
    v.n_poses = n_poses;
    v.bvh_ok = (n_poses == 1 && !prims) ? 1 : 0;   // moved vertices: the BVH boxes are stale, meshes fall back to the face loop
    return BMO_OK;
}

// ---- trace driver -----------------------------------------------------------------------------------
struct EventDestroy { void operator()(cudaEvent_t e) const { cudaEventDestroy(e); } };
static void free_wavebuf(WaveBuf& w, cudaStream_t st) { dev_free(w.d, st); dev_free(w.part, st); dev_free(w.beam, st); dev_free(w.seg, st); }
static int32_t alloc_queue(Queue& q, int64_t cap, int nf, int ni, cudaStream_t st) {
    q.cap = cap;
    BMO_CUDA(dev_alloc(&q.d, (size_t)nf * cap, st));
    BMO_CUDA(dev_alloc(&q.i, (size_t)ni * cap, st));
    return BMO_OK;
}
// enlarge a queue (SoA planes of stride cap) keeping its contents
static int32_t grow_queue(Queue& q, int64_t new_cap, int nf, int ni, cudaStream_t st) {
    DevBuf<double> d;
    DevBuf<int32_t> i;
    BMO_CUDA(d.alloc((size_t)nf * new_cap, st));
    BMO_CUDA(i.alloc((size_t)ni * new_cap, st));
    if (q.cap) {
        BMO_CUDA(cudaMemcpy2DAsync(d.get(), (size_t)new_cap * sizeof(double), q.d, (size_t)q.cap * sizeof(double), (size_t)q.cap * sizeof(double), nf,
                                   cudaMemcpyDeviceToDevice, st));
        BMO_CUDA(cudaMemcpy2DAsync(i.get(), (size_t)new_cap * sizeof(int32_t), q.i, (size_t)q.cap * sizeof(int32_t), (size_t)q.cap * sizeof(int32_t), ni,
                                   cudaMemcpyDeviceToDevice, st));
    }
    dev_free(q.d, st); dev_free(q.i, st);
    q.d = d.release(); q.i = i.release(); q.cap = new_cap;
    return BMO_OK;
}
static void free_queue(Queue& q, cudaStream_t st) { dev_free(q.d, st); dev_free(q.i, st); q.cap = 0; }

static BeamTab beamtab(bmo_result* r) {
    BeamTab b;
    b.parent = r->parent; b.slot = r->slot; b.nseg = r->nseg; b.status = r->status; b.lam = r->lam; b.pose = r->pose;
    b.spot_obj = r->spot_obj; b.w0 = r->w0; b.e0 = r->e0; b.plen = r->plen; b.popl = r->popl; b.spot_xz = r->spot_xz;
    return b;
}
template <class T> static int32_t grow(T*& p, int64_t old_n, int64_t new_n, cudaStream_t st) {
    DevBuf<T> np_;
    BMO_CUDA(np_.alloc((size_t)new_n, st));
    if (p && old_n) BMO_CUDA(cudaMemcpyAsync(np_.get(), p, (size_t)old_n * sizeof(T), cudaMemcpyDeviceToDevice, st));
    dev_free(p, st);
    p = np_.release();
    return BMO_OK;
}
// Per-beam tables of a trace that cannot add beams (no beamsplitter in the system): one allocation instead of 8-12.
static int32_t alloc_beams_slab(bmo_result* r, int64_t n, cudaStream_t st) {
    const int64_t R = r->R;
    auto pad = [](size_t b) { return (b + 255) / 256 * 256; };
    const size_t b_xz = pad((size_t)n * R * 2 * 8), b_d = r->mode == 2 ? pad((size_t)n * 8) : 0, b_i = pad((size_t)n * 4), b_so = pad((size_t)n * R * 4);
    const size_t total = b_xz + (r->mode == 2 ? 3 * b_d + pad((size_t)n * 16) : 0) + 6 * b_i + b_so;
    unsigned char* p = nullptr;
    BMO_CUDA(dev_alloc(&p, total, st));
    r->beam_slab = p;
    auto take = [&](size_t b) { unsigned char* q = p; p += b; return q; };
    r->spot_xz = (double*)take(b_xz);
    if (r->mode == 2) {
        r->w0 = (double*)take(b_d); r->plen = (double*)take(b_d); r->popl = (double*)take(b_d); r->e0 = (double*)take(pad((size_t)n * 16));
    }
    r->parent = (int32_t*)take(b_i); r->slot = (int32_t*)take(b_i); r->nseg = (int32_t*)take(b_i); r->status = (int32_t*)take(b_i);
    r->lam = (int32_t*)take(b_i); r->pose = (int32_t*)take(b_i); r->spot_obj = (int32_t*)take(b_so);
    r->cap_beams = n;
    return BMO_OK;
}
static int32_t ensure_beams(bmo_result* r, int64_t need, cudaStream_t st) {
    if (need <= r->cap_beams) return BMO_OK;
    if (r->beam_slab) return fail(BMO_ESTATE, "trace: a splitter-free trace asked for more beams than it started with");
    int64_t nc = std::max<int64_t>(need, r->cap_beams + r->cap_beams / 2);
    const int64_t oc = r->cap_beams, R = r->R;
    int32_t rc;
    if ((rc = grow(r->parent, oc, nc, st))) return rc;
    if ((rc = grow(r->slot, oc, nc, st))) return rc;
    if ((rc = grow(r->nseg, oc, nc, st))) return rc;
    if ((rc = grow(r->status, oc, nc, st))) return rc;
    if ((rc = grow(r->lam, oc, nc, st))) return rc;
    if ((rc = grow(r->pose, oc, nc, st))) return rc;
    if ((rc = grow(r->spot_obj, oc * R, nc * R, st))) return rc;
    if ((rc = grow(r->spot_xz, oc * R * 2, nc * R * 2, st))) return rc;
    if (r->mode == 2) {
        if ((rc = grow(r->w0, oc, nc, st))) return rc;
        if ((rc = grow(r->e0, oc * 2, nc * 2, st))) return rc;
        if ((rc = grow(r->plen, oc, nc, st))) return rc;
        if ((rc = grow(r->popl, oc, nc, st))) return rc;
    }
    r->cap_beams = nc;
    return BMO_OK;
}

// first_seg[b] = exclusive scan of nseg; n_segments = total.  Lazy for traces that keep no segments.
static int32_t ensure_first_seg(bmo_result* res) {
    if (res->first_seg) return BMO_OK;
    bmo_ctx* ctx = res->ctx;
    cudaStream_t st = ctx->stream;
    const int64_t nb = res->n_beams;
    BMO_CUDA(dev_alloc(&res->first_seg, (size_t)nb + 1, st));
    if (nb <= 16384) {
        scan_counts<<<1, 1024, 0, st>>>(res->nseg, nb, 1, 1, res->first_seg, ctx->d_totals);
        BMO_LAUNCH(ctx, "scan_counts(nseg)");
    } else {
        const int64_t nblk = (nb + 1023) / 1024;
        DevBuf<int32_t> bsum;
        DevBuf<long long> boff;
        BMO_CUDA(bsum.alloc((size_t)nblk, st));
        BMO_CUDA(boff.alloc((size_t)nblk, st));
        scan_local<<<(unsigned)nblk, 1024, 0, st>>>(res->nseg, nb, res->first_seg, bsum.get());
        BMO_LAUNCH(ctx, "scan_local");
        scan_counts<<<1, 1024, 0, st>>>(bsum.get(), nblk, 1, 1, boff.get(), ctx->d_totals);
        BMO_LAUNCH(ctx, "scan_counts(blocks)");
        scan_add<<<(unsigned)nblk, 1024, 0, st>>>(res->first_seg, nb, boff.get());
        BMO_LAUNCH(ctx, "scan_add");
    }
    BMO_CUDA(cudaMemcpyAsync(ctx->h_totals, ctx->d_totals, sizeof(long long), cudaMemcpyDeviceToHost, st));
    BMO_CUDA(cudaMemcpyAsync(res->first_seg + nb, ctx->d_totals, sizeof(long long), cudaMemcpyDeviceToDevice, st));
    BMO_CUDA(cudaStreamSynchronize(st));
    res->n_segments = ctx->h_totals[0];
    return BMO_OK;
}

struct TraceInputs {
    int64_t n;
    const double *pos, *dir, *E0, *grays, *w0, *ge0;
    const int32_t *lam, *pose;
    bool dir_uniform = false;   // BMO_UNIFORM_DIR
};

// *out = the device copy of a host input (owned by tmp), or the input itself when it is on the device already
template <class T> static int32_t stage_in(const T* h, size_t n, bool on_device, cudaStream_t st, const T** out, std::vector<DevBuf<char>>& tmp) {
    if (!h) { *out = nullptr; return BMO_OK; }
    if (on_device) { *out = h; return BMO_OK; }
    DevBuf<char> d;
    BMO_CUDA(d.alloc(n * sizeof(T), st));
    BMO_CUDA(cudaMemcpyAsync(d.get(), h, n * sizeof(T), cudaMemcpyHostToDevice, st));
    *out = (const T*)d.get();
    tmp.push_back(std::move(d));
    return BMO_OK;
}

// One sub-batch of a trace call: a contiguous range of root beams with its own queue, hit buffer and
// stream.  Device-resident inputs and systems with beamsplitters use a single sub-batch; host inputs of
// splitter-free systems are cut into several, so that the host->device copy of batch k+1 and the
// device->host copy of the Spotdetector hits of batch k-1 overlap the waves of batch k (rays are
// independent; without splitters beam ids are the ray indices, so the sub-batches write disjoint
// slices of the result tables).
struct SubTrace {
    bmo_sys* sys = nullptr; bmo_ctx* ctx = nullptr; bmo_result* res = nullptr;
    cudaStream_t st = nullptr;
    int mode = 0, R = 1, nfq = 0, nfs = 0, nsd = 0, units = 0;
    int32_t r_max = 0;
    bool has_splitter = false, staged = false, on_dev = false, pipelined = false;
    int64_t beam0 = 0, n = 0;              // global id of the first root beam, number of root beams
    TraceInputs in{};                      // device pointers of this sub-batch's inputs
    std::vector<DevBuf<char>> tmp;         // staged input copies
    Queue cur, next, scr;
    HitBuf hit;
    int32_t* blk_cnt = nullptr; long long* blk_off = nullptr; int64_t blk_cap = 0;
    unsigned long long* d_wtot = nullptr;  // [max_waves() + 8][2]: units alive after wave w, spawn events of wave w
    unsigned long long* h_wtot = nullptr;  // pinned, 2 * 4 entries
    long long* d_scan_tot = nullptr;       // scratch total of scan_counts
    std::vector<cudaEvent_t> ev;           // (start, stop) of intersect_wave for each wave of a chunk
    cudaEvent_t evs0 = nullptr, evs1 = nullptr;
    int64_t n_slots = 0, alive = 0, n_beams = 0;
    int wave = 0, waves_done = 0, launched = 0, slot = 0;
    int first_chunk = 1;                   // waves before the first look (bmo_sys::TraceHint)
    int64_t alive_after_w0 = -1;           // units alive after the first wave (feeds the hint)
    int32_t* spot_obj_out = nullptr; double* spot_xz_out = nullptr;   // host destinations of the Spotdetector hits (optional)
    double host_wait_ms = 0;
    RetraceView rt;                        // retrace calls: the previous solution

    // A beam holds at most r_max rays (`while length(rays) < r_max`, System.jl:133), but the children of a beamsplitter
    // start counting afresh (System.jl:141-150): a tree of g generations needs up to g * r_max waves.  The host gives up
    // after 64 generations' worth (the reference would recurse as deep as the tree is).
    int64_t max_waves() const { return has_splitter ? (int64_t)64 * (r_max + 1) : (int64_t)r_max + 1; }
    SubTrace() = default;
    SubTrace(const SubTrace&) = delete;
    SubTrace& operator=(const SubTrace&) = delete;
    ~SubTrace();
    int32_t begin(const TraceInputs& in_h);
    int32_t enqueue_chunk();
    int32_t finish_chunk();
};

static double tnow_ms() { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count(); }

int32_t SubTrace::begin(const TraceInputs& in_h) {
    int32_t rc;
    in = in_h;
    const int64_t o = beam0;
    if (mode == 2) {
        if ((rc = stage_in(in_h.grays ? in_h.grays + o * 18 : nullptr, (size_t)n * 18, on_dev, st, &in.grays, tmp))) return rc;
        if ((rc = stage_in(in_h.w0 ? in_h.w0 + o : nullptr, (size_t)n, on_dev, st, &in.w0, tmp))) return rc;
        if ((rc = stage_in(in_h.ge0 ? in_h.ge0 + o * 2 : nullptr, (size_t)n * 2, on_dev, st, &in.ge0, tmp))) return rc;
    } else {
        if ((rc = stage_in(in_h.pos + o * 3, (size_t)n * 3, on_dev, st, &in.pos, tmp))) return rc;
        if ((rc = stage_in(in_h.dir_uniform ? in_h.dir : in_h.dir + o * 3, in_h.dir_uniform ? 3 : (size_t)n * 3, on_dev, st, &in.dir, tmp))) return rc;
        if (mode == 1 && (rc = stage_in(in_h.E0 + o * 6, (size_t)n * 6, on_dev, st, &in.E0, tmp))) return rc;
    }
    if ((rc = stage_in(in_h.lam ? in_h.lam + o : nullptr, (size_t)n, on_dev, st, &in.lam, tmp))) return rc;
    if ((rc = stage_in(in_h.pose ? in_h.pose + o : nullptr, (size_t)n, on_dev, st, &in.pose, tmp))) return rc;
    if ((rc = alloc_queue(cur, n * R, nfq, NI_Q, st))) return rc;
    InitParams ip{};
    ip.q = cur; ip.n = n; ip.beam0 = beam0; ip.mode = mode; ip.pos = in.pos; ip.dir = in.dir; ip.E0 = in.E0; ip.grays = in.grays;
    ip.w0 = in.w0; ip.ge0 = in.ge0; ip.lam = in.lam; ip.pose = in.pose; ip.B = beamtab(res); ip.retrace = rt.on;
    ip.n_lambda = sys->view.n_lambda; ip.n_poses = sys->view.n_poses; ip.counters = ctx->d_counters; ip.dir_uniform = in.dir_uniform;
    const int64_t tot = n * R;
    init_queue<<<(unsigned)((tot + 255) / 256), 256, 0, st>>>(ip);
    BMO_LAUNCH(ctx, "init_queue");
    const int max_chunk = has_splitter ? 1 : 4;
    // events and the pinned read-back slots come from per-context pools (slot = index of the sub-batch)
    const size_t e0 = (size_t)slot * 10;
    while (ctx->ev_pool.size() < e0 + 10) {
        cudaEvent_t e;
        BMO_CUDA(cudaEventCreate(&e));
        ctx->ev_pool.push_back(e);
    }
    ev.assign(ctx->ev_pool.begin() + e0, ctx->ev_pool.begin() + e0 + 2 * max_chunk);
    evs0 = ctx->ev_pool[e0 + 8]; evs1 = ctx->ev_pool[e0 + 9];
    const size_t n_wtot = (size_t)2 * (max_waves() + 8);
    BMO_CUDA(dev_alloc(&d_wtot, n_wtot, st));
    BMO_CUDA(cudaMemsetAsync(d_wtot, 0, n_wtot * sizeof(unsigned long long), st));
    BMO_CUDA(dev_alloc(&d_scan_tot, 4, st));
    h_wtot = (unsigned long long*)ctx->h_totals + 8 * (1 + slot);   // slot 0 of h_totals stays with the scans
    n_slots = n; alive = n; n_beams = 0;   // n_beams is only meaningful for the single sub-batch of splitter systems (set by the caller)
    return BMO_OK;
}

// Dynamic shared memory of the trace kernels (0 unless the tables are staged); lean: the LEAN builds apply (bmo_lean.cuh).
static size_t staged_smem(const bmo_sys* sys, bool staged, bool& lean) {
    const SysView& V = sys->view;
    const size_t tab_bytes = (size_t)V.n_prims * sizeof(bmo_prim) + (size_t)V.n_parts * (sizeof(bmo_part) + NBOUND * sizeof(double));
    // kernels compiled for lean unions + small meshes only; their tables live in shared memory next to 22 KB of per-thread
    // scratch (static), so the tables + part words have to fit in what is left of the 48 KB a block gets without opting in
    lean = sys->all_lean && !sys->has_rare && staged && tab_bytes + (size_t)V.n_parts * 8 <= 24 * 1024;
    return staged ? tab_bytes + (lean ? (size_t)V.n_parts * 8 : 0) : 0;
}

// Calls f(STAGED, RK, LEAN) with the build of the trace kernels a call runs, as std::bool_constant arguments: staged tables,
// the rare (cylindrical / aspheric) primitives compiled in, the LEAN build.  LEAN implies STAGED and !RK.
template <class F> static void k1_config(bool staged, bool rk, bool lean, F&& f) {
    using Y = std::true_type;
    using N = std::false_type;
    if (lean) f(Y{}, N{}, Y{});
    else if (staged && rk) f(Y{}, Y{}, N{});
    else if (staged) f(Y{}, N{}, N{});
    else if (rk) f(N{}, Y{}, N{});
    else f(N{}, N{}, N{});
}

// enqueue the next waves on this sub-batch's stream and the read-back of their totals
int32_t SubTrace::enqueue_chunk() {
    int32_t rc;
    launched = 0;
    // waves per look at the device: 1 (most rays that miss everything die on the first wave, so the
    // compaction decision is worth an early look), then 3, then 4, 4, ...
    // (pipelined sub-batches enqueue 4 at once: an idle stream costs more than a late compaction)
    const int chunk = has_splitter ? 1 : (pipelined ? 4 : (wave == 0 ? first_chunk : (wave == 1 ? 3 : 4)));
    for (int c = 0; c < chunk; c++) {
        const int64_t nblocks = (n_slots + units - 1) / units;
        if (has_splitter) {
            // every live unit may add one unit (the reflected child) and two beams in this wave
            if (cur.cap < (n_slots + alive) * R) {
                if ((rc = grow_queue(cur, 2 * (n_slots + alive) * R, nfq, NI_Q, st))) return rc;
            }
            const int64_t scr_cap = nblocks * 2 * units * R;
            if (scr.cap < scr_cap) { free_queue(scr, st); if ((rc = alloc_queue(scr, scr_cap, nfs, NI_S, st))) return rc; }
            if ((rc = ensure_beams(res, n_beams + 2 * alive, st))) return rc;
        }
        if (blk_cap < nblocks) {
            dev_free(blk_cnt, st); dev_free(blk_off, st);
            BMO_CUDA(dev_alloc(&blk_cnt, (size_t)nblocks, st));
            BMO_CUDA(dev_alloc(&blk_off, (size_t)nblocks, st));
            blk_cap = nblocks;
        }
        WaveBuf wb{};
        if (res->keep) {     // owned by the result from the first allocation on
            res->wavebufs.push_back(WaveBuf{});
            WaveBuf& w = res->wavebufs.back();
            w.count = n_slots * R;
            BMO_CUDA(dev_alloc(&w.d, (size_t)nsd * w.count, st));
            BMO_CUDA(dev_alloc(&w.part, (size_t)w.count, st));
            BMO_CUDA(dev_alloc(&w.beam, (size_t)w.count, st));
            BMO_CUDA(dev_alloc(&w.seg, (size_t)w.count, st));
            wb = w;
        }
        if (hit.cap < n_slots * R) {
            dev_free(hit.d, st); dev_free(hit.part, st); dev_free(hit.flag, st);
            hit.cap = n_slots * R;
            BMO_CUDA(dev_alloc(&hit.d, (size_t)4 * hit.cap, st));
            BMO_CUDA(dev_alloc(&hit.part, (size_t)hit.cap, st));
            if (rt.on) BMO_CUDA(dev_alloc(&hit.flag, (size_t)hit.cap, st));
        }
        StepParams sp{};
        sp.S = sys->view; sp.cur = cur; sp.scr = scr; sp.hit = hit; sp.count = n_slots; sp.r_max = r_max; sp.keep = res->keep;
        sp.wave = wb; sp.B = beamtab(res); sp.blk_cnt = blk_cnt; sp.wave_totals = d_wtot + 2 * wave; sp.counters = ctx->d_counters;
        sp.rt = rt;
        // Pipelined (launch-bound) calls run K1 and K2 fused, every wave of the chunk in one launch: the hit records stay in
        // registers.  Measured on C2, the fused kernel carries the interaction's registers through the march (0.282 vs
        // 0.209 + 0.058 ms per wave), so it only pays where the number of launches is what limits the call.  Pipelined calls
        // have no beamsplitter, no retrace and no segment table.
        const bool fused = pipelined && mode == 0;
        const int nw = fused ? chunk - c : 1;   // waves of this launch
        sp.n_waves = nw;
        IntersectParams xp{};
        xp.S = sys->view; xp.cur = cur; xp.hit = hit; xp.n_rays = n_slots * R; xp.r_max = r_max;
        xp.counters = ctx->d_counters;
        const unsigned grid = (unsigned)((n_slots * R + IBLOCK - 1) / IBLOCK);
        bool lean;
        const size_t smem = staged_smem(sys, staged, lean);
        BMO_CUDA(cudaEventRecord(ev[2 * c], st));
        k1_config(staged, sys->has_rare, lean, [&](auto S, auto K, auto L) {
            if (fused) fused_wave0<S, K, L><<<(unsigned)nblocks, IBLOCK, smem, st>>>(sp);
            // retrace call: K1r re-validates the stored path where there is one, ordinary tracing_step! elsewhere
            else if (rt.on && mode == 0) retrace_intersect_wave<0, S, K, L><<<(unsigned)nblocks, Cfg<0>::BLOCK, smem, st>>>(sp);
            else if (rt.on && mode == 1) retrace_intersect_wave<1, S, K, L><<<(unsigned)nblocks, Cfg<1>::BLOCK, smem, st>>>(sp);
            else if (rt.on) retrace_intersect_wave<2, S, K, L><<<(unsigned)nblocks, Cfg<2>::BLOCK, smem, st>>>(sp);
            else intersect_wave<S, K, L><<<grid, IBLOCK, smem, st>>>(xp);
        });
        BMO_LAUNCH(ctx, fused ? "fused_wave0" : rt.on ? "retrace_intersect_wave" : "intersect_wave");
        BMO_CUDA(cudaEventRecord(ev[2 * c + 1], st));
        if (fused) {
            for (int k = 1; k < nw; k++) {      // the waves folded into this launch: empty timing brackets, same bookkeeping
                BMO_CUDA(cudaEventRecord(ev[2 * (c + k)], st));
                BMO_CUDA(cudaEventRecord(ev[2 * (c + k) + 1], st));
            }
            wave += nw - 1; launched += nw - 1; c += nw - 1;
        } else {
            if (!has_splitter) {
                if (mode == 0) interact_wave<0, true><<<(unsigned)nblocks, Cfg<0>::BLOCK, 0, st>>>(sp);
                else if (mode == 1) interact_wave<1, true><<<(unsigned)nblocks, Cfg<1>::BLOCK, 0, st>>>(sp);
                else interact_wave<2, true><<<(unsigned)nblocks, Cfg<2>::BLOCK, 0, st>>>(sp);
            } else if (mode == 0) interact_wave<0><<<(unsigned)nblocks, Cfg<0>::BLOCK, 0, st>>>(sp);
            else if (mode == 1) interact_wave<1><<<(unsigned)nblocks, Cfg<1>::BLOCK, 0, st>>>(sp);
            else interact_wave<2><<<(unsigned)nblocks, Cfg<2>::BLOCK, 0, st>>>(sp);
            BMO_LAUNCH(ctx, "interact_wave");
        }
        wave++;
        launched++;
        if (wave > max_waves()) break;
    }
    BMO_CUDA(cudaMemcpyAsync(h_wtot, d_wtot + 2 * (wave - launched), (size_t)2 * launched * sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
    // single-stream calls: the cumulative counters ride along, so that the call needs no blocking read-back at its end
    if (!pipelined) BMO_CUDA(cudaMemcpyAsync(ctx->h_totals + 72, ctx->d_counters, sizeof(DevCounters), cudaMemcpyDeviceToHost, st));
    return BMO_OK;
}

// one look at the device: units alive / spawn events of the waves just launched; children, compaction
int32_t SubTrace::finish_chunk() {
    int32_t rc;
    const double tw0 = tnow_ms();
    BMO_CUDA(cudaStreamSynchronize(st));
    host_wait_ms += tnow_ms() - tw0;
    int64_t prev_alive = alive;
    if (wave == launched) alive_after_w0 = (int64_t)h_wtot[0];   // this chunk began with wave 0
    for (int c = 0; c < launched; c++) {
        if (prev_alive > 0) {       // waves launched on an already empty queue are no-ops and not counted
            float kms = 0;
            BMO_CUDA(cudaEventElapsedTime(&kms, ev[2 * c], ev[2 * c + 1]));
            ctx->k1_ms += kms; ctx->k1_launches++;
            waves_done++;
        }
        prev_alive = (int64_t)h_wtot[2 * c];
    }
    alive = (int64_t)h_wtot[2 * (launched - 1)];
    const int64_t spawns = (int64_t)h_wtot[2 * (launched - 1) + 1];   // chunk == 1 whenever spawns are possible
    if (spawns > 0) {
        const int64_t nblocks = (n_slots + units - 1) / units;
        scan_counts<<<1, 1024, 0, st>>>(blk_cnt, nblocks, 1, 1, blk_off, d_scan_tot);
        BMO_LAUNCH(ctx, "scan_counts");
        SpawnParams cp{};
        cp.scr = scr; cp.q = cur; cp.blk_cnt = blk_cnt; cp.blk_off = blk_off; cp.B = beamtab(res); cp.n_beams = n_beams; cp.n_slots = n_slots;
        cp.nf = nfq; cp.mode = mode; cp.units = units; cp.R = R;
        spawn_children<<<(unsigned)nblocks, 256, 0, st>>>(cp);
        BMO_LAUNCH(ctx, "spawn_children");
        n_slots += spawns;
        n_beams += 2 * spawns;
    }
    // K3: squeeze the dead slots out once they are the majority
    if (alive > 0 && 2 * alive <= n_slots && n_slots >= 4096) {
        const int64_t cblocks = (n_slots + CBLOCK - 1) / CBLOCK;
        if (blk_cap < cblocks) {
            dev_free(blk_cnt, st); dev_free(blk_off, st);
            BMO_CUDA(dev_alloc(&blk_cnt, (size_t)cblocks, st));
            BMO_CUDA(dev_alloc(&blk_off, (size_t)cblocks, st));
            blk_cap = cblocks;
        }
        const int64_t want = has_splitter ? 2 * alive * R : alive * R;
        if (next.cap < want) { free_queue(next, st); if ((rc = alloc_queue(next, want, nfq, NI_Q, st))) return rc; }
        BMO_CUDA(cudaEventRecord(evs0, st));
        // one cooperative launch, as many blocks as are resident at once on this device
        static int coop_blocks = -1;
        if (coop_blocks < 0) {
            int per_sm = 0, sms = 0;
            BMO_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, compact_fused, CBLOCK, 0));
            BMO_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, ctx->device));
            coop_blocks = std::max(1, per_sm * sms);
        }
        int64_t nb = std::min<int64_t>(coop_blocks, cblocks);
        int64_t per = ((n_slots + nb - 1) / nb + CBLOCK - 1) / CBLOCK * CBLOCK;   // slots per block, whole rows
        nb = (n_slots + per - 1) / per;
        int R_ = R, nf_ = nfq;
        int64_t ns_ = n_slots;
        void* args[] = {&cur, &next, &ns_, &per, &R_, &nf_, &blk_cnt};
        BMO_CUDA(cudaLaunchCooperativeKernel((const void*)compact_fused, dim3((unsigned)nb), dim3(CBLOCK), args, 0, st));
        BMO_LAUNCH(ctx, "compact_fused");
        BMO_CUDA(cudaEventRecord(evs1, st));
        BMO_CUDA(cudaStreamSynchronize(st));
        float sms = 0;
        BMO_CUDA(cudaEventElapsedTime(&sms, evs0, evs1));
        ctx->k3_ms += sms;
        // algorithmic bytes: the alive flag of every slot, then read + write of every surviving ray
        ctx->k3_bytes += (double)n_slots * 4 * 2 + (double)alive * R * 2.0 * (nfq * 8 + NI_Q * 4);
        std::swap(cur, next);
        n_slots = alive;
    }
    if (alive == 0 && spot_xz_out) {   // this sub-batch is done: its Spotdetector hits go home while the others still trace
        const int64_t o = beam0 * R, m = n * R;
        if (spot_obj_out) BMO_CUDA(cudaMemcpyAsync(spot_obj_out + o, res->spot_obj + o, (size_t)m * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
        BMO_CUDA(cudaMemcpyAsync(spot_xz_out + 2 * o, res->spot_xz + 2 * o, (size_t)2 * m * sizeof(double), cudaMemcpyDeviceToHost, st));
    }
    return BMO_OK;
}

// The host waits for an auxiliary stream before its buffers go: after a failed call it may still write to the result, which
// is freed on the caller's stream.
SubTrace::~SubTrace() {
    if (ctx && st != ctx->stream) cudaStreamSynchronize(st);
    free_queue(cur, st); free_queue(next, st); free_queue(scr, st);
    dev_free(hit.d, st); dev_free(hit.part, st); dev_free(hit.flag, st);
    dev_free(blk_cnt, st); dev_free(blk_off, st);
    dev_free(d_wtot, st); dev_free(d_scan_tot, st);
}

// Resident blocks per SM of solve_rays_persistent with smem bytes of tables, 0 if a block would not fit the 48 KB of shared
// memory it gets without opting in (static scratch + tables): such a call keeps the waves.  Cached per context.
static int32_t persistent_blocks(bmo_ctx* ctx, size_t smem, int* blocks) {
    if (ctx->persist_blocks < 0 || ctx->persist_smem != smem) {
        cudaFuncAttributes fa;
        BMO_CUDA(cudaFuncGetAttributes(&fa, solve_rays_persistent));
        int b = 0;
        if (fa.sharedSizeBytes + smem <= (size_t)48 * 1024)
            BMO_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&b, solve_rays_persistent, IBLOCK, smem));
        ctx->persist_smem = smem; ctx->persist_blocks = b;
    }
    *blocks = ctx->persist_blocks;
    return BMO_OK;
}

// The whole solve of a `persistent` call (trace_common) on the caller's stream: the result tables are written by the kernel, the
// counters (with the largest nseg, from which the caller derives the wave count) come back with one copy into h_totals.
// blocks: resident blocks per SM (persistent_blocks).
static int32_t solve_persistent(bmo_sys* sys, const TraceInputs& in_h, int32_t r_max, bool on_dev, size_t smem, int blocks, bmo_result* res,
                                int32_t* spot_obj_out, double* spot_xz_out) {
    bmo_ctx* ctx = sys->ctx;
    cudaStream_t st = ctx->stream;
    const int64_t n = in_h.n;
    int32_t rc;
    std::vector<DevBuf<char>> tmp;
    SolveParams sp{};
    sp.S = sys->view; sp.n = n; sp.r_max = r_max; sp.dir_uniform = in_h.dir_uniform; sp.B = beamtab(res); sp.counters = ctx->d_counters;
    if ((rc = stage_in(in_h.pos, (size_t)n * 3, on_dev, st, &sp.pos, tmp))) return rc;
    if ((rc = stage_in(in_h.dir, in_h.dir_uniform ? 3 : (size_t)n * 3, on_dev, st, &sp.dir, tmp))) return rc;
    if ((rc = stage_in(in_h.lam, (size_t)n, on_dev, st, &sp.lam, tmp))) return rc;
    if ((rc = stage_in(in_h.pose, (size_t)n, on_dev, st, &sp.pose, tmp))) return rc;
    BMO_CUDA(cudaMemsetAsync(&ctx->d_counters->tiles, 0, 2 * sizeof(unsigned long long), st));   // tiles, most_nseg
    const int64_t grid = std::min<int64_t>((int64_t)blocks * ctx->sm_count, (n + IBLOCK - 1) / IBLOCK);
    BMO_CUDA(cudaEventRecord(ctx->evk0, st));
    solve_rays_persistent<<<(unsigned)grid, IBLOCK, smem, st>>>(sp);
    BMO_LAUNCH(ctx, "solve_rays_persistent");
    BMO_CUDA(cudaEventRecord(ctx->evk1, st));
    BMO_CUDA(cudaMemcpyAsync(ctx->h_totals + 72, ctx->d_counters, sizeof(DevCounters), cudaMemcpyDeviceToHost, st));
    if (spot_xz_out) {
        if (spot_obj_out) BMO_CUDA(cudaMemcpyAsync(spot_obj_out, res->spot_obj, (size_t)n * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
        BMO_CUDA(cudaMemcpyAsync(spot_xz_out, res->spot_xz, (size_t)2 * n * sizeof(double), cudaMemcpyDeviceToHost, st));
    }
    return BMO_OK;
}

static int32_t trace_common(bmo_sys* sys, int mode, const TraceInputs& in_h, int32_t r_max, uint32_t flags, bmo_result** out,
                            int32_t* spot_obj_out = nullptr, double* spot_xz_out = nullptr, const RetraceView* prev_rt = nullptr) {
    NvtxRange nvtx_("bmo_trace");
    if (!sys) return fail(BMO_EINVAL, "trace: NULL argument");
    if (in_h.n <= 0) return fail(BMO_EINVAL, "trace: n must be > 0");
    if (r_max < 1) return fail(BMO_EINVAL, "trace: r_max must be >= 1");
    bmo_ctx* ctx = sys->ctx;
    BMO_CUDA(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    const bool on_dev = flags & BMO_INPUT_DEVICE;
    const int R = mode == 2 ? 3 : 1;
    const int64_t n = in_h.n;

    std::unique_ptr<bmo_result, FreeWith<bmo_result_free>> res(new bmo_result());
    res->sys = sys; res->ctx = sys->ctx; res->part_object.resize(sys->parts.size()); for (size_t i = 0; i < sys->parts.size(); i++) res->part_object[i] = sys->parts[i].object;
    for (const bmo_object& ob : sys->objects) res->object_kind.push_back(ob.kind);
    res->n_objects = (int32_t)sys->objects.size(); res->n_poses = sys->view.n_poses; res->mode = mode; res->R = R; res->nsd = nf_seg(mode); res->n_roots = n; res->keep = flags & BMO_KEEP_SEGMENTS;
    static const bool prof = getenv("BMO_HOST_PROFILE") != nullptr;
    const double tp0 = tnow_ms();
    BMO_CUDA(cudaEventRecord(ctx->ev0, st));
    int32_t rc;
    // Beamsplitters are the only objects that add beams: without them the queue never grows, the
    // continuing rays are updated in place and the host only looks at the device every few waves.
    bool has_splitter = false;
    for (const bmo_object& ob : sys->objects)
        has_splitter |= ob.kind == BMO_OBJ_THIN_BS || ob.kind == BMO_OBJ_PLATE_BS || ob.kind == BMO_OBJ_CUBE_BS;
    if ((rc = has_splitter ? ensure_beams(res.get(), n, st) : alloc_beams_slab(res.get(), n, st))) return rc;
    const SysView& V = sys->view;
    const size_t table_bytes = (size_t)V.n_prims * sizeof(bmo_prim) + (size_t)V.n_parts * (sizeof(bmo_part) + NBOUND * sizeof(double));
    const bool staged = V.n_poses == 1 && table_bytes <= 40 * 1024;

    // sub-batches (see SubTrace): only host inputs of splitter-free systems are pipelined, in up to 4 (6 and 8 measured slower)
    constexpr int max_sub = 4;
    int n_sub = 1;
    if (!on_dev && !has_splitter && !res->keep) n_sub = (int)std::min<int64_t>(max_sub, std::max<int64_t>(1, n / (128 * 1024)));
    // Plain rays through a splitter-free LEAN system whose segments are not kept, in one stream: one launch solves them all
    // (solve_rays_persistent); BMO_PERSIST=0 runs them through the waves instead (A/B timing).
    static const bool persist_ok = !(getenv("BMO_PERSIST") && atoi(getenv("BMO_PERSIST")) == 0);
    bool lean;
    const size_t smem = staged_smem(sys, staged, lean);
    int pblocks = 0;
    if (persist_ok && mode == 0 && !has_splitter && !prev_rt && !res->keep && lean && n_sub == 1 && (rc = persistent_blocks(ctx, smem, &pblocks)))
        return rc;
    const bool persistent = pblocks > 0;
    int wave = 0;
    double tp1 = tp0, tp2 = tp0, tp_wave_sync = 0;   // host timeline (BMO_HOST_PROFILE)
    if (persistent) {
        if ((rc = solve_persistent(sys, in_h, r_max, on_dev, smem, pblocks, res.get(), spot_obj_out, spot_xz_out))) return rc;
        res->n_beams = n;
        tp1 = tp2 = tnow_ms();
    } else {
        while ((int)ctx->aux_streams.size() < n_sub - 1) {
            cudaStream_t s2;
            BMO_CUDA(cudaStreamCreateWithFlags(&s2, cudaStreamNonBlocking));
            ctx->aux_streams.push_back(s2);
        }
        std::unique_ptr<CUevent_st, EventDestroy> ev_fork;
        if (n_sub > 1) {   // the auxiliary streams start after everything already queued on the caller's stream (result tables included)
            cudaEvent_t e;
            BMO_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
            ev_fork.reset(e);
            BMO_CUDA(cudaEventRecord(ev_fork.get(), st));
        }
        // released at the end of this block, before the segment gather allocates the segment table
        std::vector<SubTrace> subs((size_t)n_sub);
        for (int k = 0; k < n_sub; k++) {
            SubTrace& s = subs[k];
            s.sys = sys; s.ctx = ctx; s.res = res.get(); s.st = k == 0 ? st : ctx->aux_streams[k - 1]; s.slot = k;
            s.mode = mode; s.R = R; s.nfq = nf_queue(mode); s.nfs = nf_scratch(mode); s.nsd = res->nsd;
            s.units = mode == 2 ? Cfg<2>::UNITS : Cfg<0>::UNITS;
            s.r_max = r_max; s.has_splitter = has_splitter; s.staged = staged; s.on_dev = on_dev; s.pipelined = n_sub > 1;
            s.beam0 = n * k / n_sub; s.n = n * (k + 1) / n_sub - s.beam0;
            s.spot_obj_out = spot_obj_out; s.spot_xz_out = spot_xz_out;
            if (prev_rt) s.rt = *prev_rt;
            if (k > 0) BMO_CUDA(cudaStreamWaitEvent(s.st, ev_fork.get(), 0));
            if (!has_splitter && n_sub == 1 && !prev_rt) {
                auto it = sys->hints.find({mode, n});
                if (it != sys->hints.end()) s.first_chunk = it->second.first_chunk;
            }
            if ((rc = s.begin(in_h))) return rc;
            s.n_beams = n;
            if (has_splitter) {     // sizes the previous call of this shape ended with (see bmo_sys::hints)
                auto it = sys->hints.find({mode, n});
                if (it != sys->hints.end()) {
                    const bmo_sys::TraceHint& hh = it->second;
                    if (hh.slots * R > s.cur.cap && (rc = grow_queue(s.cur, hh.slots * R, s.nfq, NI_Q, s.st))) return rc;
                    if (hh.scr > s.scr.cap) { free_queue(s.scr, s.st); if ((rc = alloc_queue(s.scr, hh.scr, s.nfs, NI_S, s.st))) return rc; }
                    if ((rc = ensure_beams(res.get(), hh.beams, s.st))) return rc;
                }
            }
            if ((rc = s.enqueue_chunk())) return rc;     // the first sub-batch is already copying / tracing while the others are set up
        }
        tp1 = tnow_ms();
        // Every sub-batch always has its next chunk of waves in flight: as soon as the host has looked at
        // the totals of one chunk it enqueues the next one on that stream, before it waits for the
        // following sub-batch (they finish roughly in order: their input copies are serialised on the link).
        for (bool any = true; any;) {
            any = false;
            for (auto& s : subs) {
                if (s.launched == 0) continue;
                if ((rc = s.finish_chunk())) return rc;
                s.launched = 0;
                if (prof) fprintf(stderr, "[bmo]   sub-batch %d: chunk done at %.3f ms (waited %.3f), alive %lld\n", s.slot, tnow_ms() - tp0, s.host_wait_ms, (long long)s.alive);
                if (s.alive > 0) {
                    if (s.wave > s.max_waves()) return fail(BMO_ESTATE, "trace: wave loop did not terminate (more than 64 generations of r_max rays)");
                    if ((rc = s.enqueue_chunk())) return rc;
                    any = true;
                }
            }
        }
        tp2 = tnow_ms();
        for (auto& s : subs) { wave = std::max(wave, s.waves_done); tp_wave_sync += s.host_wait_ms; }
        ctx->waves += wave;
        res->n_beams = has_splitter ? subs[0].n_beams : n;
        res->waves = wave;
        if (!has_splitter && n_sub == 1 && !prev_rt && subs[0].alive_after_w0 >= 0)   // would the look after wave 0 have compacted?
            sys->hints[{mode, n}].first_chunk = (2 * subs[0].alive_after_w0 > n || n < 4096) ? 4 : 1;
        if (has_splitter) {
            bmo_sys::TraceHint& hh = sys->hints[{mode, n}];
            hh.slots = std::max(hh.slots, subs[0].cur.cap / R); hh.scr = std::max(hh.scr, subs[0].scr.cap); hh.beams = std::max(hh.beams, res->cap_beams);
        }
        // join: the caller's stream continues after every sub-batch (copies of the Spotdetector hits included); the host
        // waits for each auxiliary stream as its sub-batch is released
        for (int k = 1; k < n_sub; k++) {
            BMO_CUDA(cudaEventRecord(ev_fork.get(), subs[k].st));
            BMO_CUDA(cudaStreamWaitEvent(st, ev_fork.get(), 0));
        }
    }
    const int nsd = res->nsd;
    // segment table: first_seg = exclusive scan of nseg, then gather wave-major -> beam-major
    // (spot-only traces compute first_seg lazily, see ensure_first_seg)
    if (res->keep) {
        const double tf0 = tnow_ms();
        if ((rc = ensure_first_seg(res.get()))) return rc;
        if (prof) { cudaStreamSynchronize(st); fprintf(stderr, "[bmo]   finalize: first_seg scan %.3f ms\n", tnow_ms() - tf0); }
        res->seg_rows = res->n_segments * R;
        BMO_CUDA(dev_alloc(&res->seg_d, (size_t)nsd * res->seg_rows, st));
        BMO_CUDA(dev_alloc(&res->seg_part, (size_t)res->seg_rows, st));
        if (prof) { cudaStreamSynchronize(st); fprintf(stderr, "[bmo]   finalize: + table allocation (%.1f MB) %.3f ms\n", nsd * res->seg_rows * 8e-6, tnow_ms() - tf0); }
        for (auto& wb : res->wavebufs) {
            if (nsd == 17) gather_segments<17><<<(unsigned)((wb.count + 255) / 256), 256, 0, st>>>(wb, R, res->first_seg, res->seg_d, res->seg_part);
            else gather_segments<11><<<(unsigned)((wb.count + 255) / 256), 256, 0, st>>>(wb, R, res->first_seg, res->seg_d, res->seg_part);
            BMO_LAUNCH(ctx, "gather_segments");
            free_wavebuf(wb, st);   // as soon as it is gathered: peak memory
        }
        res->wavebufs.clear();
        if (prof) { cudaStreamSynchronize(st); fprintf(stderr, "[bmo]   finalize: + gather %.3f ms\n", tnow_ms() - tf0); }
    }
    BMO_CUDA(cudaEventRecord(ctx->ev1, st));
    BMO_CUDA(cudaStreamSynchronize(st));
    float ms = 0;
    BMO_CUDA(cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1));
    ctx->trace_ms = ms;
    {
        DevCounters h;
        if (n_sub == 1) memcpy(&h, ctx->h_totals + 72, sizeof(h));   // copied behind the last chunk of waves or the solve, stream synchronised since
        else BMO_CUDA(cudaMemcpy(&h, ctx->d_counters, sizeof(h), cudaMemcpyDeviceToHost));
        if (persistent) {
            // the waves the wave loop would have counted: one per segment of the longest beam, at least one
            wave = (int)std::max<unsigned long long>(1, h.most_nseg);
            ctx->waves += wave;
            res->waves = wave;
            float kms = 0;
            BMO_CUDA(cudaEventElapsedTime(&kms, ctx->evk0, ctx->evk1));
            ctx->k1_ms += kms; ctx->k1_launches++;
        }
        res->interactions = (int64_t)h.interactions - ctx->interactions_seen;  // the counter is cumulative since the last reset
        ctx->interactions_seen = (int64_t)h.interactions;
        const int64_t bad = (int64_t)h.bad_ids - ctx->bad_ids_seen;
        ctx->bad_ids_seen = (int64_t)h.bad_ids;
        if (bad > 0)
            return fail(BMO_EINVAL, "trace: " + std::to_string(bad) + " beam(s) carry a lambda_id outside [0, n_lambda) or a pose_id outside [0, n_poses)");
    }
    if (prof) fprintf(stderr, "[bmo] trace n=%lld waves=%d sub-batches=%d: setup %.3f ms, wave loop %.3f ms (of which waiting %.3f), finalize %.3f ms\n",
                      (long long)n, wave, n_sub, tp1 - tp0, tp2 - tp1, tp_wave_sync, tnow_ms() - tp2);
    if (out) *out = res.release();
    return BMO_OK;
}

int32_t bmo_trace_rays(bmo_sys* sys, int64_t n, const double* pos, const double* dir, const int32_t* lambda_id, const double* E0,
                       const int32_t* pose_id, int32_t r_max, uint32_t flags, bmo_result** out) {
    if (!pos || !dir) return fail(BMO_EINVAL, "bmo_trace_rays: pos/dir NULL");
    TraceInputs in{};
    in.n = n; in.pos = pos; in.dir = dir; in.E0 = E0; in.lam = lambda_id; in.pose = pose_id; in.dir_uniform = (flags & BMO_UNIFORM_DIR) != 0;
    if (!sys) return fail(BMO_EINVAL, "sys NULL");
    return trace_common(sys, E0 ? 1 : 0, in, r_max, flags, out);
}
int32_t bmo_trace_rays_spots(bmo_sys* sys, int64_t n, const double* pos, const double* dir, const int32_t* lambda_id, const double* E0,
                             const int32_t* pose_id, int32_t r_max, uint32_t flags, int32_t* det_object, double* xz, bmo_result** out) {
    if (!pos || !dir) return fail(BMO_EINVAL, "bmo_trace_rays_spots: pos/dir NULL");
    if (!xz) return fail(BMO_EINVAL, "bmo_trace_rays_spots: xz NULL");
    if (!sys) return fail(BMO_EINVAL, "sys NULL");
    for (const bmo_object& ob : sys->objects)
        if (ob.kind == BMO_OBJ_THIN_BS || ob.kind == BMO_OBJ_PLATE_BS || ob.kind == BMO_OBJ_CUBE_BS)
            return fail(BMO_EINVAL, "bmo_trace_rays_spots: the system has beamsplitters (beams != rays); use bmo_trace_rays + bmo_result_spots");
    TraceInputs in{};
    in.n = n; in.pos = pos; in.dir = dir; in.E0 = E0; in.lam = lambda_id; in.pose = pose_id; in.dir_uniform = (flags & BMO_UNIFORM_DIR) != 0;
    return trace_common(sys, E0 ? 1 : 0, in, r_max, flags & ~BMO_KEEP_SEGMENTS, out, det_object, xz);
}
// solve_system!(system, beam; retrace = true) on beams that already hold a solution (System.jl:444-461 with
// retrace_system!, :188-255 / :326-428): the roots restart from their stored first rays and every beam of
// the previous tree re-validates its stored path against the previously hit objects / hinted shapes.
int32_t bmo_retrace(bmo_sys* sys, bmo_result* prev, int32_t r_max, uint32_t flags, bmo_result** out) {
    NvtxRange nvtx_("bmo_retrace");
    if (!sys || !prev) return fail(BMO_EINVAL, "bmo_retrace: NULL argument");
    if (!prev->keep || !prev->seg_part || !prev->seg_d) return fail(BMO_ESTATE, "bmo_retrace: the previous result has no segment table (trace it with BMO_KEEP_SEGMENTS)");
    if (sys->ctx != prev->ctx) return fail(BMO_EINVAL, "bmo_retrace: system and previous result live on different contexts");
    // the stored intersections name parts and objects by index: the system must have the same structure
    // (kinematics between the solves change poses, not the object list)
    if (sys->parts.size() != prev->part_object.size() || (int32_t)sys->objects.size() != prev->n_objects)
        return fail(BMO_EINVAL, "bmo_retrace: the system's objects / parts differ from those of the previous solution");
    for (size_t i = 0; i < sys->parts.size(); i++)
        if (sys->parts[i].object != prev->part_object[i]) return fail(BMO_EINVAL, "bmo_retrace: part/object layout differs from the previous solution");
    bmo_ctx* ctx = sys->ctx;
    BMO_CUDA(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    int32_t rc;
    if ((rc = ensure_first_seg(prev))) return rc;
    const int mode = prev->mode, R = prev->R;
    const int64_t n = prev->n_roots;
    // A retrace allocates the same buffers as a fresh trace plus its own temporaries (root rays, child table) while the
    // previous solution is still alive.  In a pool that holds just enough memory for the fresh trace these extra requests
    // shift every later one onto blocks that have to be split / remapped: cudaMallocAsync then takes milliseconds, erratically
    // (measured: 3.5 - 22 ms per call against 2.5 ms, pool size constant).  Growing the pool once by the footprint of a
    // call (allocate + free; the release threshold keeps it) gives the allocator the slack it needs.
    {
        const int64_t want = (int64_t)n * R * 1024;
        if (ctx->pool_slack < want) {
            void* w = nullptr;
            if (cudaMallocAsync(&w, (size_t)want, st) == cudaSuccess) cudaFreeAsync(w, st);
            else cudaGetLastError();
            ctx->pool_slack = want;
        }
    }
    PrevRoots pr{};
    pr.seg_d = prev->seg_d; pr.first_seg = prev->first_seg; pr.rows = prev->seg_rows; pr.nsd = prev->nsd; pr.lam = prev->lam; pr.pose = prev->pose;
    pr.w0 = prev->w0; pr.e0 = prev->e0; pr.n = n; pr.mode = mode;
    DevBuf<double> grays, ow0, oe0, pos, dir, E0;
    DevBuf<int32_t> olam, opose, child;
    if (mode == 2) {
        BMO_CUDA(grays.alloc((size_t)n * 18, st)); BMO_CUDA(ow0.alloc((size_t)n, st)); BMO_CUDA(oe0.alloc((size_t)n * 2, st));
    } else {
        BMO_CUDA(pos.alloc((size_t)n * 3, st)); BMO_CUDA(dir.alloc((size_t)n * 3, st));
        if (mode == 1) BMO_CUDA(E0.alloc((size_t)n * 6, st));
    }
    BMO_CUDA(olam.alloc((size_t)n, st)); BMO_CUDA(opose.alloc((size_t)n, st));
    pr.grays = grays.get(); pr.ow0 = ow0.get(); pr.oe0 = oe0.get(); pr.pos = pos.get(); pr.dir = dir.get(); pr.E0 = E0.get();
    pr.olam = olam.get(); pr.opose = opose.get();
    gather_prev_roots<<<(unsigned)((n * R + 255) / 256), 256, 0, st>>>(pr);
    BMO_LAUNCH(ctx, "gather_prev_roots");
    BMO_CUDA(child.alloc((size_t)2 * prev->n_beams, st));
    BMO_CUDA(cudaMemsetAsync(child.get(), 0xff, (size_t)2 * prev->n_beams * sizeof(int32_t), st));
    if (prev->n_beams > n) {
        build_child_table<<<(unsigned)((prev->n_beams - n + 255) / 256), 256, 0, st>>>(prev->parent, prev->slot, n, prev->n_beams, child.get());
        BMO_LAUNCH(ctx, "build_child_table");
    }
    RetraceView rt;
    rt.nseg = prev->nseg; rt.first_seg = prev->first_seg; rt.seg_part = prev->seg_part; rt.child = child.get(); rt.w0 = prev->w0; rt.on = 1;
    TraceInputs in{};
    in.n = n; in.pos = pr.pos; in.dir = pr.dir; in.E0 = pr.E0; in.grays = pr.grays; in.w0 = pr.ow0; in.ge0 = pr.oe0; in.lam = pr.olam; in.pose = pr.opose;
    uint32_t f = (flags | BMO_INPUT_DEVICE);
    if (mode == 2) f |= BMO_KEEP_SEGMENTS;
    return trace_common(sys, mode, in, r_max, f, out, nullptr, nullptr, &rt);
}
int32_t bmo_trace_beamlets(bmo_sys* sys, int64_t n, const double* rays, const int32_t* lambda_id, const double* w0, const double* E0,
                           const int32_t* pose_id, int32_t r_max, uint32_t flags, bmo_result** out) {
    if (!rays || !w0 || !E0) return fail(BMO_EINVAL, "bmo_trace_beamlets: rays/w0/E0 NULL");
    TraceInputs in{};
    in.n = n; in.grays = rays; in.w0 = w0; in.ge0 = E0; in.lam = lambda_id; in.pose = pose_id;
    if (!sys) return fail(BMO_EINVAL, "sys NULL");
    return trace_common(sys, 2, in, r_max, flags | BMO_KEEP_SEGMENTS, out);
}

// ---- result access ----------------------------------------------------------------------------------
int32_t bmo_result_get_info(bmo_result* r, bmo_result_info* info) {
    if (!r || !info) return fail(BMO_EINVAL, "bmo_result_get_info: NULL");
    info->n_roots = r->n_roots; info->n_beams = r->n_beams; info->n_segments = r->first_seg ? r->n_segments : -1; info->interactions = r->interactions;
    info->rays_per_beam = r->R; info->polarized = r->mode == 1; info->waves = r->waves; info->reserved = 0;
    return BMO_OK;
}
template <class T> static int32_t d2h(T* dst, const T* src, size_t n, cudaStream_t st) {
    if (!dst || !n) return BMO_OK;
    BMO_CUDA(cudaMemcpyAsync(dst, src, n * sizeof(T), cudaMemcpyDeviceToHost, st));
    return BMO_OK;
}
int32_t bmo_result_beams(bmo_result* r, int32_t* parent, int32_t* child_slot, int32_t* n_seg, int32_t* status, int64_t* first_seg,
                         double* w0, double* E0, int32_t* lambda_id) {
    if (!r) return fail(BMO_EINVAL, "result NULL");
    BMO_CUDA(cudaSetDevice(r->ctx->device));
    cudaStream_t st = r->ctx->stream;
    const size_t nb = (size_t)r->n_beams;
    int32_t rc;
    if ((rc = ensure_first_seg(r))) return rc;
    if ((rc = d2h(parent, r->parent, nb, st))) return rc;
    if ((rc = d2h(child_slot, r->slot, nb, st))) return rc;
    if ((rc = d2h(n_seg, r->nseg, nb, st))) return rc;
    if ((rc = d2h(status, r->status, nb, st))) return rc;
    if ((rc = d2h((long long*)first_seg, r->first_seg, nb, st))) return rc;
    if ((rc = d2h(lambda_id, r->lam, nb, st))) return rc;
    if (r->mode == 2) {
        if ((rc = d2h(w0, r->w0, nb, st))) return rc;
        if ((rc = d2h(E0, r->e0, 2 * nb, st))) return rc;
    }
    BMO_CUDA(cudaStreamSynchronize(st));
    return BMO_OK;
}
int32_t bmo_result_segments(bmo_result* r, double* pos, double* dir, double* n, double* t, double* nrm, int32_t* object, int32_t* part,
                            double* E0) {
    if (!r) return fail(BMO_EINVAL, "result NULL");
    if (!r->keep) return fail(BMO_ESTATE, "bmo_result_segments: trace was run without BMO_KEEP_SEGMENTS");
    BMO_CUDA(cudaSetDevice(r->ctx->device));
    cudaStream_t st = r->ctx->stream;
    const size_t rows = (size_t)r->seg_rows;
    if (rows == 0) return BMO_OK;
    // the device table holds one record of nsd doubles per row; the ABI hands out one array per quantity -> stage through a host buffer
    const size_t nsd = (size_t)r->nsd;
    std::vector<double> h(nsd * rows);
    std::vector<int32_t> hp(rows);
    BMO_CUDA(cudaMemcpyAsync(h.data(), r->seg_d, h.size() * sizeof(double), cudaMemcpyDeviceToHost, st));
    BMO_CUDA(cudaMemcpyAsync(hp.data(), r->seg_part, rows * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    BMO_CUDA(cudaStreamSynchronize(st));
    const std::vector<int32_t>& part_object = r->part_object;
    for (size_t i = 0; i < rows; i++) {
        const double* q = h.data() + i * nsd;
        if (pos) { pos[3 * i] = q[S_PX]; pos[3 * i + 1] = q[S_PY]; pos[3 * i + 2] = q[S_PZ]; }
        if (dir) { dir[3 * i] = q[S_DX]; dir[3 * i + 1] = q[S_DY]; dir[3 * i + 2] = q[S_DZ]; }
        if (n) n[i] = q[S_N];
        if (t) t[i] = q[S_T];
        if (nrm) { nrm[3 * i] = q[S_NX]; nrm[3 * i + 1] = q[S_NY]; nrm[3 * i + 2] = q[S_NZ]; }
        if (part) part[i] = hp[i];
        if (object) object[i] = hp[i] >= 0 ? part_object[hp[i]] : -1;
        if (E0 && r->mode == 1) for (int k = 0; k < 6; k++) E0[6 * i + k] = q[S_E0 + k];
    }
    return BMO_OK;
}
int32_t bmo_result_spots(bmo_result* r, int32_t* det_object, double* xz) {
    if (!r) return fail(BMO_EINVAL, "result NULL");
    BMO_CUDA(cudaSetDevice(r->ctx->device));
    cudaStream_t st = r->ctx->stream;
    const size_t nr = (size_t)r->n_beams * r->R;
    int32_t rc;
    if ((rc = d2h(det_object, r->spot_obj, nr, st))) return rc;
    if ((rc = d2h(xz, r->spot_xz, 2 * nr, st))) return rc;
    BMO_CUDA(cudaStreamSynchronize(st));
    return BMO_OK;
}
int32_t bmo_result_spots_device(bmo_result* r, const int32_t** det_object, const double** xz) {
    if (!r) return fail(BMO_EINVAL, "result NULL");
    if (det_object) *det_object = r->spot_obj;
    if (xz) *xz = r->spot_xz;
    return BMO_OK;
}
int32_t bmo_result_free(bmo_result* r) {
    if (!r) return BMO_OK;
    cudaSetDevice(r->ctx->device);
    cudaStream_t st = r->ctx->stream;
    if (r->beam_slab) dev_free(r->beam_slab, st);
    else {
        dev_free(r->parent, st); dev_free(r->slot, st); dev_free(r->nseg, st); dev_free(r->status, st); dev_free(r->lam, st); dev_free(r->pose, st);
        dev_free(r->w0, st); dev_free(r->e0, st); dev_free(r->plen, st); dev_free(r->popl, st);
        dev_free(r->spot_obj, st); dev_free(r->spot_xz, st);
    }
    dev_free(r->first_seg, st);
    dev_free(r->seg_d, st); dev_free(r->seg_part, st);
    for (auto& wb : r->wavebufs) free_wavebuf(wb, st);
    delete r;
    return BMO_OK;
}

// ---- FP64 peak probe (roofline denominator for the FP64-bound kernels) -------------------------------
__global__ void dfma_probe(double* out, int iters) {
    double a0 = threadIdx.x * 1e-9, a1 = a0 + 1, a2 = a0 + 2, a3 = a0 + 3, a4 = a0 + 4, a5 = a0 + 5, a6 = a0 + 6, a7 = a0 + 7;
    const double b = 1.0000001, c = 1e-9;
    for (int i = 0; i < iters; i++) {
        a0 = __fma_rn(a0, b, c); a1 = __fma_rn(a1, b, c); a2 = __fma_rn(a2, b, c); a3 = __fma_rn(a3, b, c);
        a4 = __fma_rn(a4, b, c); a5 = __fma_rn(a5, b, c); a6 = __fma_rn(a6, b, c); a7 = __fma_rn(a7, b, c);
    }
    out[(size_t)blockIdx.x * blockDim.x + threadIdx.x] = a0 + a1 + a2 + a3 + a4 + a5 + a6 + a7;
}
int32_t bmo_measure_fp64_peak(bmo_ctx* ctx, double* tflops) {
    if (!ctx || !tflops) return fail(BMO_EINVAL, "NULL");
    BMO_CUDA(cudaSetDevice(ctx->device));
    const int blocks = ctx->sm_count * 8, threads = 256, iters = 1 << 16;
    DevBuf<double> d;
    BMO_CUDA(d.alloc((size_t)blocks * threads, ctx->stream));
    float best = 1e30f;
    for (int rep = 0; rep < 5; rep++) {
        BMO_CUDA(cudaEventRecord(ctx->ev0, ctx->stream));
        dfma_probe<<<blocks, threads, 0, ctx->stream>>>(d.get(), iters);
        BMO_LAUNCH(ctx, "dfma_probe");
        BMO_CUDA(cudaEventRecord(ctx->ev1, ctx->stream));
        BMO_CUDA(cudaStreamSynchronize(ctx->stream));
        float ms;
        BMO_CUDA(cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1));
        if (rep > 0 && ms < best) best = ms;
    }
    *tflops = 2.0 * 8 * iters * (double)blocks * threads / (best * 1e-3) / 1e12;
    return BMO_OK;
}

// ---- self-check of the normal evaluations --------------------------------------------------------------
// normal3d (AbstractSDF.jl:79-95) of member prim_idx[i] at points[i], evaluated twice: with the written-out gradients of the
// unrotated lens primitives (identity_gradient, bmo_geom.cuh) where they apply, and with the generic dual-number evaluation.
// The two must agree bit for bit (tests/test_gpu_normals.py).
__global__ void debug_normals_kernel(const SysView S, int64_t n, const double* pts, const int32_t* prim, double* out_fast, double* out_gen) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const V3 p = mk3(pts[3 * i], pts[3 * i + 1], pts[3 * i + 2]);
    Stats st; st.sdf = 0; st.tri = 0;
    const V3 a = member_normal<true, true>(S.prims, prim[i], p, S.zr, st);
    const V3 b = member_normal<true, false>(S.prims, prim[i], p, S.zr, st);
    out_fast[3 * i] = a.x; out_fast[3 * i + 1] = a.y; out_fast[3 * i + 2] = a.z;
    out_gen[3 * i] = b.x; out_gen[3 * i + 1] = b.y; out_gen[3 * i + 2] = b.z;
}
int32_t bmo_debug_normals(bmo_sys* sys, int64_t n, const double* points, const int32_t* prim_idx, double* out_fast, double* out_generic) {
    if (!sys || !points || !prim_idx || !out_fast || !out_generic || n < 0) return fail(BMO_EINVAL, "bmo_debug_normals: bad argument");
    for (int64_t i = 0; i < n; i++)
        if (prim_idx[i] < 0 || prim_idx[i] >= sys->view.n_prims) return fail(BMO_EINVAL, "bmo_debug_normals: prim index out of range");
    if (n == 0) return BMO_OK;
    bmo_ctx* ctx = sys->ctx;
    BMO_CUDA(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    DevBuf<double> d_pts, d_a, d_b;
    DevBuf<int32_t> d_idx;
    BMO_CUDA(d_pts.alloc((size_t)3 * n, st)); BMO_CUDA(d_a.alloc((size_t)3 * n, st)); BMO_CUDA(d_b.alloc((size_t)3 * n, st));
    BMO_CUDA(d_idx.alloc((size_t)n, st));
    BMO_CUDA(cudaMemcpyAsync(d_pts.get(), points, (size_t)3 * n * sizeof(double), cudaMemcpyHostToDevice, st));
    BMO_CUDA(cudaMemcpyAsync(d_idx.get(), prim_idx, (size_t)n * sizeof(int32_t), cudaMemcpyHostToDevice, st));
    debug_normals_kernel<<<(unsigned)((n + 127) / 128), 128, 0, st>>>(sys->view, n, d_pts.get(), d_idx.get(), d_a.get(), d_b.get());
    BMO_LAUNCH(ctx, "debug_normals_kernel");
    BMO_CUDA(cudaMemcpyAsync(out_fast, d_a.get(), (size_t)3 * n * sizeof(double), cudaMemcpyDeviceToHost, st));
    BMO_CUDA(cudaMemcpyAsync(out_generic, d_b.get(), (size_t)3 * n * sizeof(double), cudaMemcpyDeviceToHost, st));
    BMO_CUDA(cudaStreamSynchronize(st));
    return BMO_OK;
}


