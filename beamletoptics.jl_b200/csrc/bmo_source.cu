// bmo_source.cu -- ray sources expanded on the device and the spot-diagram reduction.
//
// Sources (bmo_source_create): the host hands over a descriptor -- basis, ring table, rotate3d matrices, every
// transcendental of the host constructors (BeamGroups.jl:51-100, 152-195, 222-245) -- and the device writes the rays the
// trace reads with BMO_INPUT_DEVICE, instead of 24-48 B per ray crossing the bus.
//   source_rings  one thread per ring (thread 0: ray 0).  Ray j of a ring comes from the serial recurrence v <- rot v in
//                 linalg.matvec's order ((a0 v0 + a1 v1) + a2 v2): bit-identical to the host loop.  A closed form
//                 rotate3d(d, j * delta) v would round differently.
//   source_disc   one thread per ray (Fibonacci disc); sin / cos are CUDA's, within a few ulp of the host's.
// Pose-tiled sources (bmo_source_create_poses): n_poses copies of the rays, pose-major, with pose_id[i] = i / n_rays.  A
// disc thread computes ray i mod n_rays with the untiled arithmetic (rho over n_rays), ring sources run the recurrence
// once and source_tile replicates tile 0, so every tile is bit-identical to the untiled source.
// Spot statistics (bmo_spot_stats): two passes over a fixed partition of the spot entries (spot_sums: counts, sums,
// extrema and the histogram; spot_spread: the squared distances to the centroid).  Each block reduces its slice in a
// fixed order and the last block to finish combines the per-block partials in block order, so the result does not depend
// on which blocks ran when.
// Per-pose statistics (bmo_spot_stats_poses): the same two kernels over every pose at once.  The beams are ordered stably
// by pose (cub radix sort on the pose id, skipped when the result is already pose-major), each pose's entry list is cut
// with bmo_spot_stats's slice formula applied to that pose's entry count, and each pose has its own completion counters:
// a pose reduces the same values in the same order as a one-pose result that lists its entries in the same order.
// Compiled with -fmad=false; the arithmetic that must match the host bit for bit is spelled with __dmul_rn / __dadd_rn.
#include <cmath>
#include <cub/device/device_radix_sort.cuh>
#include "bmo_host.cuh"

namespace bmo {

struct SrcParams {
    int64_t n, n_rings;             // rays of one tile, rings
    int64_t total;                  // n * n_poses
    int32_t kind;
    double p[3], d[3], e1[3], e2[3], radius, phi0;
    const bmo_source_ring* rings;
    double *pos, *dir;              // dir: [total][3], or [3] for a uniform direction
    int32_t* pose_id;               // [total], NULL for one pose
};

// RayBundle's renormalisation: d * (1 / sqrt(dx dx + dy dy + dz dz))
BMO_D void renormalise(const double v[3], double* out) {
    const double s = __dadd_rn(__dadd_rn(__dmul_rn(v[0], v[0]), __dmul_rn(v[1], v[1])), __dmul_rn(v[2], v[2]));
    const double inv = __ddiv_rn(1.0, __dsqrt_rn(s));
    for (int i = 0; i < 3; i++) out[i] = __dmul_rn(v[i], inv);
}

__global__ void source_rings(SrcParams P) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t > P.n_rings) return;
    const bool point = P.kind == BMO_SRC_POINT;
    if (t == 0) {   // ray 0: the centre (collimated) or the axis (point); a collimated direction is stored once
        for (int i = 0; i < 3; i++) { P.pos[i] = P.p[i]; P.dir[i] = P.d[i]; }
        return;
    }
    const bmo_source_ring g = P.rings[t - 1];
    double v[3] = {g.start[0], g.start[1], g.start[2]};
    const double* a = g.rot;
    for (int64_t j = 0; j < g.count; j++) {
        double* q = P.pos + 3 * (g.first + j);
        if (point) {
            q[0] = P.p[0]; q[1] = P.p[1]; q[2] = P.p[2];
            renormalise(v, P.dir + 3 * (g.first + j));
        } else {
            for (int i = 0; i < 3; i++) q[i] = __dadd_rn(P.p[i], v[i]);
        }
        double w[3];
        for (int i = 0; i < 3; i++)
            w[i] = __dadd_rn(__dadd_rn(__dmul_rn(a[3 * i], v[0]), __dmul_rn(a[3 * i + 1], v[1])), __dmul_rn(a[3 * i + 2], v[2]));
        v[0] = w[0]; v[1] = w[1]; v[2] = w[2];
    }
}

// one thread per tiled ray t: ray k = t mod n of the descriptor (rho over the n rays of one tile)
__global__ void source_disc(SrcParams P) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= P.total) return;
    if (t == 0) for (int i = 0; i < 3; i++) P.dir[i] = P.d[i];
    const int64_t k = t % P.n;
    if (P.pose_id) P.pose_id[t] = (int32_t)(t / P.n);
    const double kd = (double)k;
    const double rho = __dsqrt_rn(__ddiv_rn(__dadd_rn(kd, 0.5), (double)P.n));
    const double phi = __dmul_rn(kd, P.phi0);
    const double r = __dmul_rn(P.radius, rho);
    double s, c;
    sincos(phi, &s, &c);
    const double rc = __dmul_rn(r, c), rs = __dmul_rn(r, s);
    for (int i = 0; i < 3; i++) P.pos[3 * t + i] = __dadd_rn(P.p[i], __dadd_rn(__dmul_rn(rc, P.e1[i]), __dmul_rn(rs, P.e2[i])));
}

// ring sources with several poses: replicate tile 0 (written by source_rings) and write the pose ids; one thread per ray
__global__ void source_tile(SrcParams P, int uniform) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= P.total) return;
    P.pose_id[t] = (int32_t)(t / P.n);
    if (t < P.n) return;
    const int64_t k = t % P.n;
    for (int i = 0; i < 3; i++) P.pos[3 * t + i] = P.pos[3 * k + i];
    if (!uniform)
        for (int i = 0; i < 3; i++) P.dir[3 * t + i] = P.dir[3 * k + i];
}

// ---- spot statistics ------------------------------------------------------------------------------------------
constexpr int SPOT_BLOCK = 256;
constexpr int64_t SPOT_SLICE = 4096;     // entries per block (times a factor that keeps the grid at <= 1024 blocks)

struct SpotPartial { unsigned long long hits, outside; double sx, sz, maxr, lo[2], hi[2], ssq; };

struct SpotParams {
    const int32_t* obj; const double* xz;
    int64_t n, per;                 // one pose (pstart == NULL): entries, entries per block
    int32_t det, has_window, nx, nz;
    double win[4];
    int32_t R;                      // entries per beam
    int32_t n_poses;
    const int32_t* order;           // NULL: entries in index order; else beam ids stably sorted by pose ([n_beams])
    const int64_t* pstart;          // NULL: one pose; else [n_poses + 1]: first position of each pose in the ordered entries
    const int64_t* pper;            // [n_poses]: entries per block of each pose
    const int32_t* pblk;            // [n_poses + 1]: first block of each pose
    unsigned long long* counts;     // NULL: no histogram; else [n_poses][nz][nx]
    SpotPartial* part;              // [gridDim.x]
    unsigned int* done;             // [n_poses][2] blocks of the pose finished with spot_sums / spot_spread
    bmo_spot_info* out;             // device, [n_poses]
};

// the pose of this block, the pose's blocks [first, first + nblk) and this block's slice [b0, b1) of the ordered entries
struct SpotSlice { int32_t pose, first, nblk; int64_t b0, b1; };
__device__ SpotSlice spot_slice(const SpotParams& P) {
    SpotSlice s;
    const int32_t b = (int32_t)blockIdx.x;
    if (!P.pstart) {
        s.pose = 0; s.first = 0; s.nblk = (int32_t)gridDim.x;
        s.b0 = (int64_t)b * P.per; s.b1 = min(P.n, s.b0 + P.per);
        return s;
    }
    int32_t lo = 0, hi = P.n_poses;   // last pose whose first block is <= b (every pose has at least one block)
    while (hi - lo > 1) {
        const int32_t mid = (lo + hi) / 2;
        if (P.pblk[mid] <= b) lo = mid; else hi = mid;
    }
    s.pose = lo; s.first = P.pblk[lo]; s.nblk = P.pblk[lo + 1] - s.first;
    s.b0 = P.pstart[lo] + (int64_t)(b - s.first) * P.pper[lo];
    s.b1 = min(P.pstart[lo + 1], s.b0 + P.pper[lo]);
    return s;
}
// entry index at position q of the ordered entry list (the R entries of a beam stay together, in entry order)
__device__ __forceinline__ int64_t spot_entry(const SpotParams& P, int64_t q) {
    return P.order ? (int64_t)P.order[q / P.R] * P.R + q % P.R : q;
}

// fixed-shape tree over the block's threads
template <class T, class Op> __device__ T block_reduce(T v, T* sh, Op op) {
    sh[threadIdx.x] = v;
    __syncthreads();
    for (int s = SPOT_BLOCK / 2; s > 0; s >>= 1) {
        if ((int)threadIdx.x < s) sh[threadIdx.x] = op(sh[threadIdx.x], sh[threadIdx.x + s]);
        __syncthreads();
    }
    T r = sh[0];
    __syncthreads();
    return r;
}
struct AddD { __device__ double operator()(double a, double b) const { return __dadd_rn(a, b); } };
struct AddU { __device__ unsigned long long operator()(unsigned long long a, unsigned long long b) const { return a + b; } };
struct MaxD { __device__ double operator()(double a, double b) const { return fmax(a, b); } };
struct MinD { __device__ double operator()(double a, double b) const { return fmin(a, b); } };

// true in every thread of the block that finishes last of `nblk` (its partial and those of the other blocks are visible)
__device__ bool last_block(unsigned int* done, int32_t nblk) {
    __shared__ bool last;
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) last = atomicAdd(done, 1u) == (unsigned)nblk - 1;
    __syncthreads();
    if (last) __threadfence();
    return last;
}

__global__ void __launch_bounds__(SPOT_BLOCK) spot_sums(SpotParams P) {
    __shared__ double shd[SPOT_BLOCK];
    __shared__ unsigned long long shu[SPOT_BLOCK];
    const SpotSlice sl = spot_slice(P);
    unsigned long long* counts = P.counts ? P.counts + (size_t)sl.pose * P.nx * P.nz : nullptr;
    unsigned long long hits = 0, outside = 0;
    double sx = 0, sz = 0, maxr = -INFINITY, lox = INFINITY, loz = INFINITY, hix = -INFINITY, hiz = -INFINITY;
    for (int64_t q = sl.b0 + threadIdx.x; q < sl.b1; q += SPOT_BLOCK) {
        const int64_t k = spot_entry(P, q);
        if (P.obj[k] != P.det) continue;
        const double x = P.xz[2 * k], z = P.xz[2 * k + 1];
        hits++;
        sx = __dadd_rn(sx, x); sz = __dadd_rn(sz, z);
        maxr = fmax(maxr, __dsqrt_rn(__dadd_rn(__dmul_rn(x, x), __dmul_rn(z, z))));
        lox = fmin(lox, x); hix = fmax(hix, x); loz = fmin(loz, z); hiz = fmax(hiz, z);
        if (P.has_window) {
            if (!(x >= P.win[0] && x <= P.win[1] && z >= P.win[2] && z <= P.win[3])) { outside++; continue; }
            if (counts) {
                const double fi = floor(__dmul_rn(__ddiv_rn(__dsub_rn(x, P.win[0]), __dsub_rn(P.win[1], P.win[0])), (double)P.nx));
                const double fj = floor(__dmul_rn(__ddiv_rn(__dsub_rn(z, P.win[2]), __dsub_rn(P.win[3], P.win[2])), (double)P.nz));
                const int64_t i = min((int64_t)fi, (int64_t)P.nx - 1), j = min((int64_t)fj, (int64_t)P.nz - 1);
                atomicAdd(counts + j * P.nx + i, 1ull);
            }
        }
    }
    SpotPartial r;
    r.hits = block_reduce(hits, shu, AddU());
    r.outside = block_reduce(outside, shu, AddU());
    r.sx = block_reduce(sx, shd, AddD());
    r.sz = block_reduce(sz, shd, AddD());
    r.maxr = block_reduce(maxr, shd, MaxD());
    r.lo[0] = block_reduce(lox, shd, MinD());
    r.lo[1] = block_reduce(loz, shd, MinD());
    r.hi[0] = block_reduce(hix, shd, MaxD());
    r.hi[1] = block_reduce(hiz, shd, MaxD());
    r.ssq = 0;
    if (threadIdx.x == 0) P.part[blockIdx.x] = r;
    if (!last_block(P.done + 2 * sl.pose, sl.nblk) || threadIdx.x != 0) return;
    // combine the pose's partials in block order
    const volatile SpotPartial* vp = P.part;
    unsigned long long H = 0, O = 0;
    double SX = 0, SZ = 0, M = -INFINITY, L0 = INFINITY, L1 = INFINITY, U0 = -INFINITY, U1 = -INFINITY;
    for (int32_t b = sl.first; b < sl.first + sl.nblk; b++) {
        H += vp[b].hits; O += vp[b].outside;
        SX = __dadd_rn(SX, vp[b].sx); SZ = __dadd_rn(SZ, vp[b].sz);
        M = fmax(M, vp[b].maxr);
        L0 = fmin(L0, vp[b].lo[0]); L1 = fmin(L1, vp[b].lo[1]); U0 = fmax(U0, vp[b].hi[0]); U1 = fmax(U1, vp[b].hi[1]);
    }
    bmo_spot_info o;
    o.hits = (int64_t)H; o.outside = (int64_t)O;
    const double nan = __longlong_as_double(0x7ff8000000000000ll);
    if (H == 0) {
        o.centroid[0] = o.centroid[1] = o.rms = o.max_r = o.lo[0] = o.lo[1] = o.hi[0] = o.hi[1] = nan;
    } else {
        o.centroid[0] = __ddiv_rn(SX, (double)H); o.centroid[1] = __ddiv_rn(SZ, (double)H);
        o.rms = nan; o.max_r = M; o.lo[0] = L0; o.lo[1] = L1; o.hi[0] = U0; o.hi[1] = U1;
    }
    P.out[sl.pose] = o;
}

__global__ void __launch_bounds__(SPOT_BLOCK) spot_spread(SpotParams P) {
    __shared__ double shd[SPOT_BLOCK];
    const SpotSlice sl = spot_slice(P);
    bmo_spot_info* out = P.out + sl.pose;
    if (out->hits == 0) return;   // every block of the pose sees the same count: nothing to do, rms stays NaN
    const double cx = out->centroid[0], cz = out->centroid[1];
    double s = 0;
    for (int64_t q = sl.b0 + threadIdx.x; q < sl.b1; q += SPOT_BLOCK) {
        const int64_t k = spot_entry(P, q);
        if (P.obj[k] != P.det) continue;
        const double dx = __dsub_rn(P.xz[2 * k], cx), dz = __dsub_rn(P.xz[2 * k + 1], cz);
        s = __dadd_rn(s, __dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dz, dz)));
    }
    s = block_reduce(s, shd, AddD());
    if (threadIdx.x == 0) P.part[blockIdx.x].ssq = s;
    if (!last_block(P.done + 2 * sl.pose + 1, sl.nblk) || threadIdx.x != 0) return;
    const volatile SpotPartial* vp = P.part;
    double S = 0;
    for (int32_t b = sl.first; b < sl.first + sl.nblk; b++) S = __dadd_rn(S, vp[b].ssq);
    out->rms = __dsqrt_rn(__ddiv_rn(S, (double)out->hits));
}

// per-pose beam counts of a result; bit 0 of *flags: the poses are not in non-decreasing beam order, bit 1: a pose id
// outside [0, n_poses).  Each thread counts a run of POSE_RUN consecutive beams and adds a count when the pose changes, and
// the lanes of a warp that flush the same pose add once: a pose-major result takes about one atomic per warp, not per beam.
constexpr int64_t POSE_RUN = 64;
__device__ __forceinline__ void add_pose_count(unsigned long long* cnt, int32_t p, unsigned long long c, bool act) {
    const unsigned live = __ballot_sync(0xffffffffu, act);
    if (!act) return;
    const unsigned same = __match_any_sync(live, p);
    unsigned long long sum = 0;
    for (unsigned m = same; m; m &= m - 1) sum += __shfl_sync(same, c, __ffs(m) - 1);
    if ((int)(threadIdx.x & 31) == __ffs(same) - 1) atomicAdd(cnt + p, sum);
}
__global__ void spot_pose_count(const int32_t* pose, int64_t nb, int32_t n_poses, unsigned long long* cnt, unsigned int* flags) {
    const int64_t b0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) * POSE_RUN, b1 = min(nb, b0 + POSE_RUN);
    int32_t cur = -1;
    unsigned long long c = 0;
    bool bad = false, unsorted = b0 > 0 && b0 < nb && pose[b0 - 1] > pose[b0];
    for (int64_t b = b0; b < b1; b++) {
        const int32_t p = pose[b];
        if ((unsigned)p >= (unsigned)n_poses) { bad = true; continue; }
        if (p != cur && c) { atomicAdd(cnt + cur, c); c = 0; }
        unsorted |= cur > p;
        cur = p; c++;
    }
    add_pose_count(cnt, cur, c, c > 0);
    if (bad) atomicOr(flags, 2u);
    if (unsorted) atomicOr(flags, 1u);
}

__global__ void iota32(int32_t* v, int64_t n) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) v[i] = (int32_t)i;
}

}  // namespace bmo

using namespace bmo;

struct bmo_source {
    bmo_ctx* ctx = nullptr;
    int64_t n = 0;              // rays of all tiles: n_rays * n_poses
    int64_t n_rays = 0;
    int32_t n_poses = 1;
    bool uniform = false;
    double* pos = nullptr;      // [n][3]
    double* dir = nullptr;      // [n][3], or [3] when uniform
    int32_t* pose_id = nullptr; // [n], NULL for one pose
};

static int32_t launched(bmo_ctx* ctx, const char* what) {
    ctx->launches++;
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail(BMO_ECUDA, std::string(what) + ": " + cudaGetErrorString(e));
    return BMO_OK;
}

static bool finite3(const double* v) { return std::isfinite(v[0]) && std::isfinite(v[1]) && std::isfinite(v[2]); }

static int32_t check_desc(const bmo_source_desc* d) {
    if (d->kind != BMO_SRC_DISC && d->kind != BMO_SRC_COLLIMATED && d->kind != BMO_SRC_POINT)
        return fail(BMO_EINVAL, "bmo_source_create: unknown source kind " + std::to_string(d->kind));
    if (d->n_rays < 1) return fail(BMO_EINVAL, "bmo_source_create: n_rays must be >= 1");
    if (!finite3(d->pos) || !finite3(d->dir)) return fail(BMO_EINVAL, "bmo_source_create: pos / dir not finite");
    if (d->kind == BMO_SRC_DISC) {
        if (d->n_rings != 0) return fail(BMO_EINVAL, "bmo_source_create: a disc source has no rings");
        if (!finite3(d->e1) || !finite3(d->e2) || !std::isfinite(d->radius) || !std::isfinite(d->phi0))
            return fail(BMO_EINVAL, "bmo_source_create: disc basis / radius / phi0 not finite");
        return BMO_OK;
    }
    if (d->n_rings < 0 || (d->n_rings > 0 && !d->rings)) return fail(BMO_EINVAL, "bmo_source_create: bad ring table");
    int64_t next = 1;
    for (int64_t i = 0; i < d->n_rings; i++) {
        const bmo_source_ring& g = d->rings[i];
        if (g.first != next || g.count < 0 || g.count > d->n_rays - next)
            return fail(BMO_EINVAL, "bmo_source_create: ring " + std::to_string(i) + " does not continue the rays at " + std::to_string(next));
        if (!finite3(g.start) || !finite3(g.rot) || !finite3(g.rot + 3) || !finite3(g.rot + 6))
            return fail(BMO_EINVAL, "bmo_source_create: ring " + std::to_string(i) + " not finite");
        next += g.count;
    }
    if (next != d->n_rays) return fail(BMO_EINVAL, "bmo_source_create: the rings hold " + std::to_string(next - 1) + " rays, n_rays - 1 = " + std::to_string(d->n_rays - 1));
    return BMO_OK;
}

int32_t bmo_source_free(bmo_source* s) {
    if (!s) return BMO_OK;
    cudaSetDevice(s->ctx->device);
    dev_free(s->pos, s->ctx->stream);
    dev_free(s->dir, s->ctx->stream);
    dev_free(s->pose_id, s->ctx->stream);
    delete s;
    return BMO_OK;
}

int32_t bmo_source_create_poses(bmo_ctx* ctx, const bmo_source_desc* desc, int32_t n_poses, bmo_source** out) {
    NvtxRange nvtx_("bmo_source_create");
    if (!ctx || !desc || !out) return fail(BMO_EINVAL, "bmo_source_create: NULL argument");
    if (n_poses < 1) return fail(BMO_EINVAL, "bmo_source_create_poses: n_poses must be >= 1");
    int32_t rc;
    if ((rc = check_desc(desc))) return rc;
    if (desc->n_rays > INT64_MAX / n_poses) return fail(BMO_EINVAL, "bmo_source_create_poses: n_rays * n_poses overflows int64");
    BMO_CUDA(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    bmo_source* s = new bmo_source();
    s->ctx = ctx; s->n_rays = desc->n_rays; s->n_poses = n_poses; s->n = desc->n_rays * n_poses; s->uniform = desc->kind != BMO_SRC_POINT;
    const int64_t n = s->n;
    SrcParams P{};
    P.n = desc->n_rays; P.total = n; P.n_rings = desc->n_rings; P.kind = desc->kind;
    for (int i = 0; i < 3; i++) { P.p[i] = desc->pos[i]; P.d[i] = desc->dir[i]; P.e1[i] = desc->e1[i]; P.e2[i] = desc->e2[i]; }
    P.radius = desc->radius; P.phi0 = desc->phi0;
    bmo_source_ring* d_rings = nullptr;
    cudaError_t e = dev_alloc(&s->pos, (size_t)n * 3, st);
    if (e == cudaSuccess) e = dev_alloc(&s->dir, s->uniform ? (size_t)3 : (size_t)n * 3, st);
    if (e == cudaSuccess && n_poses > 1) e = dev_alloc(&s->pose_id, (size_t)n, st);
    if (e == cudaSuccess && desc->kind != BMO_SRC_DISC && desc->n_rings > 0) {
        e = dev_alloc(&d_rings, (size_t)desc->n_rings, st);
        if (e == cudaSuccess) e = cudaMemcpyAsync(d_rings, desc->rings, (size_t)desc->n_rings * sizeof(bmo_source_ring), cudaMemcpyHostToDevice, st);
    }
    if (e != cudaSuccess) {
        dev_free(d_rings, st);
        bmo_source_free(s);
        return fail(BMO_ECUDA, std::string("bmo_source_create: ") + cudaGetErrorString(e));
    }
    P.rings = d_rings; P.pos = s->pos; P.dir = s->dir; P.pose_id = s->pose_id;
    if (desc->kind == BMO_SRC_DISC) {
        source_disc<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(P);
        rc = launched(ctx, "source_disc");
    } else {
        // the serial recurrence runs once (tile 0); further poses are copies of it
        source_rings<<<(unsigned)((desc->n_rings + 1 + 63) / 64), 64, 0, st>>>(P);
        rc = launched(ctx, "source_rings");
        if (!rc && n_poses > 1) {
            source_tile<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(P, s->uniform ? 1 : 0);
            rc = launched(ctx, "source_tile");
        }
    }
    dev_free(d_rings, st);
    if (rc) { bmo_source_free(s); return rc; }
    *out = s;
    return BMO_OK;
}

int32_t bmo_source_create(bmo_ctx* ctx, const bmo_source_desc* desc, bmo_source** out) {
    return bmo_source_create_poses(ctx, desc, 1, out);
}

int32_t bmo_source_pose_ids(bmo_source* s, int32_t* n_poses, const int32_t** pose_id) {
    if (!s) return fail(BMO_EINVAL, "bmo_source_pose_ids: source NULL");
    if (n_poses) *n_poses = s->n_poses;
    if (pose_id) *pose_id = s->pose_id;
    return BMO_OK;
}

int32_t bmo_source_device(bmo_source* s, int64_t* n, const double** pos, const double** dir, int32_t* uniform_dir) {
    if (!s) return fail(BMO_EINVAL, "bmo_source_device: source NULL");
    if (n) *n = s->n;
    if (pos) *pos = s->pos;
    if (dir) *dir = s->dir;
    if (uniform_dir) *uniform_dir = s->uniform ? 1 : 0;
    return BMO_OK;
}

int32_t bmo_source_rays(bmo_source* s, double* pos, double* dir) {
    if (!s) return fail(BMO_EINVAL, "bmo_source_rays: source NULL");
    BMO_CUDA(cudaSetDevice(s->ctx->device));
    cudaStream_t st = s->ctx->stream;
    const size_t n = (size_t)s->n;
    if (pos) BMO_CUDA(cudaMemcpyAsync(pos, s->pos, n * 3 * sizeof(double), cudaMemcpyDeviceToHost, st));
    if (dir) BMO_CUDA(cudaMemcpyAsync(dir, s->dir, (s->uniform ? 3 : n * 3) * sizeof(double), cudaMemcpyDeviceToHost, st));
    BMO_CUDA(cudaStreamSynchronize(st));
    if (dir && s->uniform)
        for (size_t i = 1; i < n; i++) { dir[3 * i] = dir[0]; dir[3 * i + 1] = dir[1]; dir[3 * i + 2] = dir[2]; }
    return BMO_OK;
}

// bmo_spot_stats (n_poses = 1: every entry, index order) and bmo_spot_stats_poses (n_poses = the result's pose count)
static int32_t spot_stats(const char* what, bmo_result* r, int32_t det_object, int32_t n_poses, const double* window, int32_t nx,
                          int32_t nz, bmo_spot_info* out, int64_t* counts, uint32_t flags) {
    const std::string fn(what);
    if (!r || !out) return fail(BMO_EINVAL, fn + ": NULL argument");
    if (det_object < 0 || det_object >= (int32_t)r->object_kind.size() || r->object_kind[det_object] != BMO_OBJ_SPOTDETECTOR)
        return fail(BMO_EINVAL, fn + ": object " + std::to_string(det_object) + " is not a Spotdetector of the result's system");
    if (window) {
        for (int i = 0; i < 4; i++)
            if (!std::isfinite(window[i])) return fail(BMO_EINVAL, fn + ": window not finite");
        if (!(window[1] > window[0]) || !(window[3] > window[2])) return fail(BMO_EINVAL, fn + ": window needs x_hi > x_lo and z_hi > z_lo");
    }
    if (counts) {
        if (!window) return fail(BMO_EINVAL, fn + ": a histogram needs a window");
        if (nx < 1 || nz < 1) return fail(BMO_EINVAL, fn + ": nx and nz must be >= 1");
    }
    bmo_ctx* ctx = r->ctx;
    BMO_CUDA(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    const int64_t n = r->n_beams * r->R;
    const auto slice = [](int64_t m) { return SPOT_SLICE * std::max<int64_t>(1, (m + SPOT_SLICE * 1024 - 1) / (SPOT_SLICE * 1024)); };
    const size_t np = (size_t)n_poses;
    const size_t bins = counts ? (size_t)nx * (size_t)nz : 0;
    const bool dev_counts = counts && (flags & BMO_INPUT_DEVICE);
    SpotParams P{};
    P.obj = r->spot_obj; P.xz = r->spot_xz; P.n = n; P.det = det_object; P.R = r->R; P.n_poses = n_poses;
    P.has_window = window != nullptr; P.nx = nx; P.nz = nz;
    if (window) for (int i = 0; i < 4; i++) P.win[i] = window[i];
    // Several poses: order the beams stably by pose and cut every pose's entries with the one-pose slice formula.  The host
    // needs the per-pose counts to size the grid: one read-back of n_poses + 1 words.
    std::vector<int64_t> tab;   // pstart [n_poses + 1], pper [n_poses], then pblk [n_poses + 1] as int32 pairs
    int64_t nblk = 0;
    int32_t* order = nullptr;
    cudaError_t e = cudaSuccess;
    int32_t rc = BMO_OK;
    if (n_poses == 1) {
        P.per = slice(n);
        nblk = std::max<int64_t>(1, (n + P.per - 1) / P.per);
    } else {
        const int64_t nb = r->n_beams;
        if (nb > INT32_MAX) return fail(BMO_EINVAL, fn + ": more beams than a 32-bit beam id can number");
        unsigned long long* cnt = nullptr;   // [n_poses] counts, then the flags word
        BMO_CUDA(dev_alloc(&cnt, np + 1, st));
        std::vector<unsigned long long> h(np + 1);
        e = cudaMemsetAsync(cnt, 0, (np + 1) * sizeof(unsigned long long), st);
        if (e == cudaSuccess && nb > 0) {
            const int64_t runs = (nb + POSE_RUN - 1) / POSE_RUN;
            spot_pose_count<<<(unsigned)((runs + 255) / 256), 256, 0, st>>>(r->pose, nb, n_poses, cnt, (unsigned int*)(cnt + np));
            rc = launched(ctx, "spot_pose_count");
        }
        if (!rc && e == cudaSuccess) e = cudaMemcpyAsync(h.data(), cnt, (np + 1) * sizeof(unsigned long long), cudaMemcpyDeviceToHost, st);
        if (!rc && e == cudaSuccess) e = cudaStreamSynchronize(st);
        dev_free(cnt, st);
        if (rc) return rc;
        if (e != cudaSuccess) return fail(BMO_ECUDA, fn + ": " + cudaGetErrorString(e));
        if (h[np] & 2u) return fail(BMO_EINVAL, fn + ": a beam of the result carries a pose id outside [0, n_poses)");
        if (h[np] & 1u) {   // not pose-major (beamsplitter children, or pose ids in any order): stable radix sort on the pose id
            int32_t *keys = nullptr, *iota = nullptr;
            void* tmp = nullptr;
            size_t tmp_bytes = 0;
            const int end_bit = 32 - __builtin_clz((unsigned)(n_poses - 1));
            e = cub::DeviceRadixSort::SortPairs(nullptr, tmp_bytes, (const int32_t*)r->pose, keys, (const int32_t*)iota, order, (int)nb, 0, end_bit, st);
            if (e == cudaSuccess) e = dev_alloc(&order, (size_t)nb, st);
            if (e == cudaSuccess) e = dev_alloc(&keys, (size_t)nb, st);
            if (e == cudaSuccess) e = dev_alloc(&iota, (size_t)nb, st);
            if (e == cudaSuccess) e = dev_alloc((char**)&tmp, tmp_bytes, st);
            if (e == cudaSuccess) {
                iota32<<<(unsigned)((nb + 255) / 256), 256, 0, st>>>(iota, nb);
                rc = launched(ctx, "iota32");
            }
            if (!rc && e == cudaSuccess) {
                e = cub::DeviceRadixSort::SortPairs(tmp, tmp_bytes, (const int32_t*)r->pose, keys, (const int32_t*)iota, order, (int)nb, 0, end_bit, st);
                if (e == cudaSuccess) rc = launched(ctx, "radix sort by pose");
            }
            dev_free(keys, st); dev_free(iota, st); dev_free(tmp, st);
            if (rc || e != cudaSuccess) {
                dev_free(order, st);
                if (rc) return rc;
                return fail(BMO_ECUDA, fn + ": " + cudaGetErrorString(e));
            }
        }
        tab.assign(2 * np + 1 + (np + 2) / 2, 0);
        int32_t* pblk = (int32_t*)(tab.data() + 2 * np + 1);
        for (size_t p = 0; p < np; p++) {
            const int64_t m = (int64_t)h[p] * r->R;
            const int64_t per = slice(m);
            tab[p + 1] = tab[p] + m;
            tab[np + 1 + p] = per;
            pblk[p] = (int32_t)nblk;
            nblk += std::max<int64_t>(1, (m + per - 1) / per);
        }
        pblk[np] = (int32_t)nblk;
        if (nblk > INT32_MAX) { dev_free(order, st); return fail(BMO_EINVAL, fn + ": too many blocks"); }
    }
    // one scratch block: partials, two completion counters per pose, the statistics, the histogram of a host `counts`, the
    // per-pose slice table
    const size_t off_done = (size_t)nblk * sizeof(SpotPartial), done_bytes = (8 * np + 15) / 16 * 16;
    const size_t off_out = off_done + done_bytes, off_hist = off_out + np * sizeof(bmo_spot_info);
    const size_t off_tab = off_hist + (counts && !dev_counts ? np * bins * sizeof(int64_t) : 0);
    const size_t bytes = off_tab + tab.size() * sizeof(int64_t);
    char* scr = nullptr;
    e = dev_alloc(&scr, bytes, st);
    if (e != cudaSuccess) { dev_free(order, st); return fail(BMO_ECUDA, fn + ": " + cudaGetErrorString(e)); }
    P.part = (SpotPartial*)scr; P.done = (unsigned int*)(scr + off_done); P.out = (bmo_spot_info*)(scr + off_out);
    P.counts = counts ? (dev_counts ? (unsigned long long*)counts : (unsigned long long*)(scr + off_hist)) : nullptr;
    P.order = order;
    if (!tab.empty()) {
        P.pstart = (const int64_t*)(scr + off_tab); P.pper = P.pstart + np + 1; P.pblk = (const int32_t*)(P.pper + np);
        e = cudaMemcpyAsync(scr + off_tab, tab.data(), tab.size() * sizeof(int64_t), cudaMemcpyHostToDevice, st);
    }
    if (e == cudaSuccess) e = cudaMemsetAsync(P.done, 0, done_bytes, st);
    if (e == cudaSuccess && P.counts) e = cudaMemsetAsync(P.counts, 0, np * bins * sizeof(int64_t), st);
    if (e == cudaSuccess) {
        spot_sums<<<(unsigned)nblk, SPOT_BLOCK, 0, st>>>(P);
        rc = launched(ctx, "spot_sums");
        if (!rc) {
            spot_spread<<<(unsigned)nblk, SPOT_BLOCK, 0, st>>>(P);
            rc = launched(ctx, "spot_spread");
        }
        if (!rc) e = cudaMemcpyAsync(out, P.out, np * sizeof(bmo_spot_info), cudaMemcpyDeviceToHost, st);
        if (!rc && e == cudaSuccess && counts && !dev_counts) e = cudaMemcpyAsync(counts, P.counts, np * bins * sizeof(int64_t), cudaMemcpyDeviceToHost, st);
        if (!rc && e == cudaSuccess) e = cudaStreamSynchronize(st);
    }
    dev_free(scr, st);
    dev_free(order, st);
    if (rc) return rc;
    if (e != cudaSuccess) return fail(BMO_ECUDA, fn + ": " + cudaGetErrorString(e));
    return BMO_OK;
}

int32_t bmo_spot_stats(bmo_result* r, int32_t det_object, const double* window, int32_t nx, int32_t nz, bmo_spot_info* out,
                       int64_t* counts, uint32_t flags) {
    NvtxRange nvtx_("bmo_spot_stats");
    return spot_stats("bmo_spot_stats", r, det_object, 1, window, nx, nz, out, counts, flags);
}

int32_t bmo_spot_stats_poses(bmo_result* r, int32_t det_object, int32_t n_poses, const double* window, int32_t nx, int32_t nz,
                             bmo_spot_info* out, int64_t* counts, uint32_t flags) {
    NvtxRange nvtx_("bmo_spot_stats_poses");
    if (r && n_poses != r->n_poses)
        return fail(BMO_EINVAL, "bmo_spot_stats_poses: n_poses " + std::to_string(n_poses) + " differs from the " +
                                    std::to_string(r->n_poses) + " poses the result was traced with");
    return spot_stats("bmo_spot_stats_poses", r, det_object, n_poses, window, nx, nz, out, counts, flags);
}
