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
// Source slices (bmo_source_create_slice): rays [first, first + count) of the one-pose source.  A disc thread computes ray
// first + i; a ring that overlaps the slice runs its recurrence from its own start and writes the rays inside the slice.
// Beamlet sources (bmo_source_create_beamlets): the kernels above write the chief positions of one tile (or slice) into a
// temporary, and source_beamlets writes every tile's [18] rays, w0, E0 and pose id from them and the host's constants, one
// thread per beamlet, with from_params' additions and products.
// Spot statistics (bmo_spot_stats): two passes over a fixed partition of the spot entries (spot_sums: counts, sums,
// extrema and the histogram; spot_spread: the squared distances to the centroid).  Each block reduces its slice in a
// fixed order and the last block to finish combines the per-block partials in block order, so the result does not depend
// on which blocks ran when.
// Per-pose statistics (bmo_spot_stats_poses): the same two kernels over every pose at once.  The beams are ordered stably
// by pose (cub radix sort on the pose id, skipped when the result is already pose-major), each pose's entry list is cut
// with bmo_spot_stats's slice formula applied to that pose's entry count, and each pose has its own completion counters:
// a pose reduces the same values in the same order as a one-pose result that lists its entries in the same order.
// Several results (bmo_spot_stats_results): the same two kernels over the concatenation of the results' entries, cut by
// the slice formula on the total; a table of (spot arrays, first concatenated entry) per result tells each thread where
// an entry lives, so a block may straddle two results and still reduce what one result listing the same entries gives.
// Several ranks (bmo_spot_stats_sharded, collective steps in bmo_comm.cu): each rank runs both passes over its own entries
// without the last-block combine; the partials of all ranks are all-gathered and spot_combine runs the same combine loop
// over them in global block order on every rank.
// Compiled with -fmad=false; the arithmetic that must match the host bit for bit is spelled with __dmul_rn / __dadd_rn.
#include <cmath>
#include <cub/device/device_radix_sort.cuh>
#include "bmo_host.cuh"

namespace bmo {

struct SrcParams {
    int64_t n, n_rings;             // rays of the descriptor, rings
    int64_t first, count;           // the rays [first, first + count) of the descriptor that one tile holds
    int64_t total;                  // count * n_poses
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
        if (!point) for (int i = 0; i < 3; i++) P.dir[i] = P.d[i];
        if (P.first == 0) for (int i = 0; i < 3; i++) { P.pos[i] = P.p[i]; P.dir[i] = P.d[i]; }
        return;
    }
    // ray k of the descriptor is stored at k - first; the recurrence starts at the ring's first ray whatever the slice
    const bmo_source_ring g = P.rings[t - 1];
    const int64_t stop = min(g.first + g.count, P.first + P.count);
    if (stop <= P.first) return;
    double v[3] = {g.start[0], g.start[1], g.start[2]};
    const double* a = g.rot;
    for (int64_t k = g.first; k < stop; k++) {
        if (k >= P.first) {
            double* q = P.pos + 3 * (k - P.first);
            if (point) {
                q[0] = P.p[0]; q[1] = P.p[1]; q[2] = P.p[2];
                renormalise(v, P.dir + 3 * (k - P.first));
            } else {
                for (int i = 0; i < 3; i++) q[i] = __dadd_rn(P.p[i], v[i]);
            }
        }
        double w[3];
        for (int i = 0; i < 3; i++)
            w[i] = __dadd_rn(__dadd_rn(__dmul_rn(a[3 * i], v[0]), __dmul_rn(a[3 * i + 1], v[1])), __dmul_rn(a[3 * i + 2], v[2]));
        v[0] = w[0]; v[1] = w[1]; v[2] = w[2];
    }
}

// one thread per stored ray t: ray k = first + t mod count of the descriptor (rho over its n rays)
__global__ void source_disc(SrcParams P) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= P.total) return;
    if (t == 0) for (int i = 0; i < 3; i++) P.dir[i] = P.d[i];
    const int64_t k = P.first + t % P.count;
    if (P.pose_id) P.pose_id[t] = (int32_t)(t / P.count);
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

struct BeamletParams {
    const double* pos;              // [count][3]: the chief positions of one tile
    int64_t count, total;           // beamlets of a tile, of all tiles
    double dv[3], dd[3], s[3], w0, div_offset, e0[2];
    double *rays, *w0_out, *e0_out; // [total][18], [total], [total][2]
    int32_t* pose_id;               // [total], NULL for one pose
};

// one thread per stored beamlet t: tile t / count, beamlet t mod count of the tile; from_params' rows and operation order
__global__ void source_beamlets(BeamletParams B) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= B.total) return;
    const int64_t k = t % B.count;
    const double p[3] = {B.pos[3 * k], B.pos[3 * k + 1], B.pos[3 * k + 2]};
    double* r = B.rays + 18 * t;
    for (int i = 0; i < 3; i++) {
        r[i] = p[i];
        r[3 + i] = B.dv[i];
        r[6 + i] = __dadd_rn(p[i], __dmul_rn(B.s[i], B.w0));
        r[9 + i] = B.dv[i];
        r[12 + i] = __dadd_rn(p[i], __dmul_rn(B.s[i], B.div_offset));
        r[15 + i] = B.dd[i];
    }
    B.w0_out[t] = B.w0;
    B.e0_out[2 * t] = B.e0[0];
    B.e0_out[2 * t + 1] = B.e0[1];
    if (B.pose_id) B.pose_id[t] = (int32_t)(t / B.count);
}

// ---- spot statistics ------------------------------------------------------------------------------------------
constexpr int SPOT_BLOCK = 256;

struct SpotPartial { unsigned long long hits, outside; double sx, sz, maxr, lo[2], hi[2], ssq; };

// one result of a reduction over several: its spot arrays and the position of its entry 0 in the concatenated entries
struct SpotRes { const int32_t* obj; const double* xz; int64_t first; };

struct SpotParams {
    const int32_t* obj; const double* xz;   // the one result (res == NULL)
    const SpotRes* res;             // NULL, or [n_res + 1]: several results in list order; res[n_res].first = n
    int32_t n_res;
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
    unsigned int* done;             // [n_poses][2] blocks of the pose finished with spot_sums / spot_spread; NULL: no
                                    // combine (bmo_spot_stats_sharded combines the partials of every rank in spot_combine)
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
// several results: the one that holds position q of the concatenated entries (the last r with res[r].first <= q)
__device__ int32_t spot_res_of(const SpotParams& P, int64_t q) {
    int32_t lo = 0, hi = P.n_res;
    while (hi - lo > 1) {
        const int32_t mid = (lo + hi) / 2;
        if (P.res[mid].first <= q) lo = mid; else hi = mid;
    }
    return lo;
}
// the entry at position q: true with its (x, z) if it lies on the detector.  r is the thread's result cursor (several
// results): a thread visits increasing q, so the cursor only moves forward.
__device__ __forceinline__ bool spot_at(const SpotParams& P, int64_t q, int32_t& r, double& x, double& z) {
    const int32_t* obj = P.obj;
    const double* xz = P.xz;
    int64_t k;
    if (P.res) {
        while (q >= P.res[r + 1].first) r++;
        obj = P.res[r].obj; xz = P.res[r].xz; k = q - P.res[r].first;
    } else {
        k = spot_entry(P, q);
    }
    if (obj[k] != P.det) return false;
    x = xz[2 * k]; z = xz[2 * k + 1];
    return true;
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

// the partials combined in block order: the loop the last block of spot_sums runs, and spot_combine over every rank's
struct SpotAcc {
    unsigned long long H = 0, O = 0;
    double SX = 0, SZ = 0, M = -INFINITY, L0 = INFINITY, L1 = INFINITY, U0 = -INFINITY, U1 = -INFINITY;
    template <class Part> __device__ void add(Part& p) {   // volatile in the last block, plain in spot_combine
        H += p.hits; O += p.outside;
        SX = __dadd_rn(SX, p.sx); SZ = __dadd_rn(SZ, p.sz);
        M = fmax(M, p.maxr);
        L0 = fmin(L0, p.lo[0]); L1 = fmin(L1, p.lo[1]); U0 = fmax(U0, p.hi[0]); U1 = fmax(U1, p.hi[1]);
    }
    __device__ bmo_spot_info info() const {
        bmo_spot_info o;
        o.hits = (int64_t)H; o.outside = (int64_t)O;
        const double nan = __longlong_as_double(0x7ff8000000000000ll);
        if (H == 0) {
            o.centroid[0] = o.centroid[1] = o.rms = o.max_r = o.lo[0] = o.lo[1] = o.hi[0] = o.hi[1] = nan;
        } else {
            o.centroid[0] = __ddiv_rn(SX, (double)H); o.centroid[1] = __ddiv_rn(SZ, (double)H);
            o.rms = nan; o.max_r = M; o.lo[0] = L0; o.lo[1] = L1; o.hi[0] = U0; o.hi[1] = U1;
        }
        return o;
    }
};

__global__ void __launch_bounds__(SPOT_BLOCK) spot_sums(SpotParams P) {
    __shared__ double shd[SPOT_BLOCK];
    __shared__ unsigned long long shu[SPOT_BLOCK];
    const SpotSlice sl = spot_slice(P);
    unsigned long long* counts = P.counts ? P.counts + (size_t)sl.pose * P.nx * P.nz : nullptr;
    unsigned long long hits = 0, outside = 0;
    double sx = 0, sz = 0, maxr = -INFINITY, lox = INFINITY, loz = INFINITY, hix = -INFINITY, hiz = -INFINITY;
    int32_t cur = P.res ? spot_res_of(P, sl.b0 + threadIdx.x) : 0;
    for (int64_t q = sl.b0 + threadIdx.x; q < sl.b1; q += SPOT_BLOCK) {
        double x, z;
        if (!spot_at(P, q, cur, x, z)) continue;
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
    if (!P.done || !last_block(P.done + 2 * sl.pose, sl.nblk) || threadIdx.x != 0) return;
    // combine the pose's partials in block order
    const volatile SpotPartial* vp = P.part;
    SpotAcc a;
    for (int32_t b = sl.first; b < sl.first + sl.nblk; b++) a.add(vp[b]);
    P.out[sl.pose] = a.info();
}

__global__ void __launch_bounds__(SPOT_BLOCK) spot_spread(SpotParams P) {
    __shared__ double shd[SPOT_BLOCK];
    const SpotSlice sl = spot_slice(P);
    bmo_spot_info* out = P.out + sl.pose;
    if (out->hits == 0) return;   // every block of the pose sees the same count: nothing to do, rms stays NaN
    const double cx = out->centroid[0], cz = out->centroid[1];
    double s = 0;
    int32_t cur = P.res ? spot_res_of(P, sl.b0 + threadIdx.x) : 0;
    for (int64_t q = sl.b0 + threadIdx.x; q < sl.b1; q += SPOT_BLOCK) {
        double x, z;
        if (!spot_at(P, q, cur, x, z)) continue;
        const double dx = __dsub_rn(x, cx), dz = __dsub_rn(z, cz);
        s = __dadd_rn(s, __dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dz, dz)));
    }
    s = block_reduce(s, shd, AddD());
    if (threadIdx.x == 0) P.part[blockIdx.x].ssq = s;
    if (!P.done || !last_block(P.done + 2 * sl.pose + 1, sl.nblk) || threadIdx.x != 0) return;
    const volatile SpotPartial* vp = P.part;
    double S = 0;
    for (int32_t b = sl.first; b < sl.first + sl.nblk; b++) S = __dadd_rn(S, vp[b].ssq);
    out->rms = __dsqrt_rn(__ddiv_rn(S, (double)out->hits));
}

// bmo_spot_stats_sharded: the all-gathered partials of every rank, all[k * stride + b] for rank k's blocks b < ceil(entries[k] /
// per), combined in global block order -- the combine loop of spot_sums (pass 0) or spot_spread (pass 1), on one thread
// (a kernel of its own after the all-gather: plain loads, which the compiler may issue ahead of the serial sums)
__global__ void spot_combine(const SpotPartial* __restrict__ all, int32_t n_ranks, int32_t stride, const int64_t* entries, int64_t per,
                             int32_t pass, bmo_spot_info* out) {
    if (pass == 0) {
        SpotAcc a;
        for (int32_t k = 0; k < n_ranks; k++) {
            const SpotPartial* p = all + (int64_t)k * stride;
            const int64_t nb = (entries[k] + per - 1) / per;
#pragma unroll 8
            for (int64_t b = 0; b < nb; b++) a.add(p[b]);
        }
        *out = a.info();
        return;
    }
    if (out->hits == 0) return;
    double S = 0;
    for (int32_t k = 0; k < n_ranks; k++) {
        const SpotPartial* p = all + (int64_t)k * stride;
        const int64_t nb = (entries[k] + per - 1) / per;
#pragma unroll 8
        for (int64_t b = 0; b < nb; b++) S = __dadd_rn(S, p[b].ssq);
    }
    out->rms = __dsqrt_rn(__ddiv_rn(S, (double)out->hits));
}

// per-pose beam counts of a result; bit 0 of *flags: the poses are not in non-decreasing beam order, bit 1: a pose id
// outside [0, n_poses).  Counted in runs of POSE_RUN beams (add_pose_count, bmo_host.cuh).
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
    bool beamlets = false;      // bmo_source_create_beamlets: rays / w0 / e0 instead of pos / dir
    double* rays = nullptr;     // [n][18]
    double* w0 = nullptr;       // [n]
    double* e0 = nullptr;       // [n][2]
};

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
    dev_free(s->rays, s->ctx->stream);
    dev_free(s->w0, s->ctx->stream);
    dev_free(s->e0, s->ctx->stream);
    delete s;
    return BMO_OK;
}

// n_poses copies of the rays [first, first + count) of the descriptor into pos [count * n_poses][3], dir ([3] for a uniform
// direction) and pose_id (NULL for one pose); n_poses > 1 only for the whole source
static int32_t expand_rays(bmo_ctx* ctx, const bmo_source_desc* desc, int32_t n_poses, int64_t first, int64_t count, double* pos,
                           double* dir, int32_t* pose_id) {
    cudaStream_t st = ctx->stream;
    const int64_t n = count * n_poses;
    SrcParams P{};
    P.n = desc->n_rays; P.first = first; P.count = count; P.total = n; P.n_rings = desc->n_rings; P.kind = desc->kind;
    for (int i = 0; i < 3; i++) { P.p[i] = desc->pos[i]; P.d[i] = desc->dir[i]; P.e1[i] = desc->e1[i]; P.e2[i] = desc->e2[i]; }
    P.radius = desc->radius; P.phi0 = desc->phi0;
    DevBuf<bmo_source_ring> d_rings;
    if (desc->kind != BMO_SRC_DISC && desc->n_rings > 0) {
        BMO_CUDA(d_rings.alloc((size_t)desc->n_rings, st));
        BMO_CUDA(cudaMemcpyAsync(d_rings.get(), desc->rings, (size_t)desc->n_rings * sizeof(bmo_source_ring), cudaMemcpyHostToDevice, st));
    }
    P.rings = d_rings.get(); P.pos = pos; P.dir = dir; P.pose_id = pose_id;
    if (desc->kind == BMO_SRC_DISC) {
        source_disc<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(P);
        BMO_LAUNCH(ctx, "source_disc");
    } else {
        // the serial recurrence runs once (tile 0); further poses are copies of it
        source_rings<<<(unsigned)((desc->n_rings + 1 + 63) / 64), 64, 0, st>>>(P);
        BMO_LAUNCH(ctx, "source_rings");
        if (n_poses > 1) {
            source_tile<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(P, desc->kind != BMO_SRC_POINT ? 1 : 0);
            BMO_LAUNCH(ctx, "source_tile");
        }
    }
    return BMO_OK;
}

static int32_t source_create(bmo_ctx* ctx, const bmo_source_desc* desc, int32_t n_poses, int64_t first, int64_t count, bmo_source** out) {
    BMO_CUDA(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    std::unique_ptr<bmo_source, FreeWith<bmo_source_free>> s(new bmo_source());
    s->ctx = ctx; s->n_rays = desc->n_rays; s->n_poses = n_poses; s->n = count * n_poses; s->uniform = desc->kind != BMO_SRC_POINT;
    const int64_t n = s->n;
    BMO_CUDA(dev_alloc(&s->pos, (size_t)n * 3, st));
    BMO_CUDA(dev_alloc(&s->dir, s->uniform ? (size_t)3 : (size_t)n * 3, st));
    if (n_poses > 1) BMO_CUDA(dev_alloc(&s->pose_id, (size_t)n, st));
    int32_t rc;
    if ((rc = expand_rays(ctx, desc, n_poses, first, count, s->pos, s->dir, s->pose_id))) return rc;
    *out = s.release();
    return BMO_OK;
}

int32_t bmo_source_create_poses(bmo_ctx* ctx, const bmo_source_desc* desc, int32_t n_poses, bmo_source** out) {
    NvtxRange nvtx_("bmo_source_create");
    if (!ctx || !desc || !out) return fail(BMO_EINVAL, "bmo_source_create: NULL argument");
    if (n_poses < 1) return fail(BMO_EINVAL, "bmo_source_create_poses: n_poses must be >= 1");
    int32_t rc;
    if ((rc = check_desc(desc))) return rc;
    if (desc->n_rays > INT64_MAX / n_poses) return fail(BMO_EINVAL, "bmo_source_create_poses: n_rays * n_poses overflows int64");
    return source_create(ctx, desc, n_poses, 0, desc->n_rays, out);
}

int32_t bmo_source_create(bmo_ctx* ctx, const bmo_source_desc* desc, bmo_source** out) {
    return bmo_source_create_poses(ctx, desc, 1, out);
}

int32_t bmo_source_create_slice(bmo_ctx* ctx, const bmo_source_desc* desc, int64_t first, int64_t count, bmo_source** out) {
    NvtxRange nvtx_("bmo_source_create_slice");
    if (!ctx || !desc || !out) return fail(BMO_EINVAL, "bmo_source_create_slice: NULL argument");
    int32_t rc;
    if ((rc = check_desc(desc))) return rc;
    if (first < 0 || count < 1 || first > desc->n_rays - count)
        return fail(BMO_EINVAL, "bmo_source_create_slice: rays [" + std::to_string(first) + ", " + std::to_string(first) + " + " +
                                    std::to_string(count) + ") are not a non-empty part of the source's " + std::to_string(desc->n_rays));
    return source_create(ctx, desc, 1, first, count, out);
}

static bool finite_n(const double* v, int n) {
    for (int i = 0; i < n; i++)
        if (!std::isfinite(v[i])) return false;
    return true;
}

int32_t bmo_source_create_beamlets(bmo_ctx* ctx, const bmo_source_desc* desc, const bmo_beamlet_desc* bd, int32_t n_poses, int64_t first,
                                   int64_t count, bmo_source** out) {
    NvtxRange nvtx_("bmo_source_create_beamlets");
    const std::string fn = "bmo_source_create_beamlets";
    if (!ctx || !desc || !bd || !out) return fail(BMO_EINVAL, fn + ": NULL argument");
    int32_t rc;
    if ((rc = check_desc(desc))) return rc;
    if (desc->kind == BMO_SRC_POINT) return fail(BMO_EINVAL, fn + ": a point source's rays have no common direction for its beamlets");
    if (!finite_n(bd->dv, 3) || !finite_n(bd->dd, 3) || !finite_n(bd->s, 3) || !std::isfinite(bd->w0) || !std::isfinite(bd->div_offset) ||
        !finite_n(bd->E0, 2))
        return fail(BMO_EINVAL, fn + ": beamlet constants not finite");
    if (!(bd->w0 > 0)) return fail(BMO_EINVAL, fn + ": w0 must be > 0");
    if (n_poses < 1) return fail(BMO_EINVAL, fn + ": n_poses must be >= 1");
    if (first < 0 || count < 1 || first > desc->n_rays - count)
        return fail(BMO_EINVAL, fn + ": beamlets [" + std::to_string(first) + ", " + std::to_string(first) + " + " + std::to_string(count) +
                                    ") are not a non-empty part of the source's " + std::to_string(desc->n_rays));
    if (n_poses > 1 && (first != 0 || count != desc->n_rays)) return fail(BMO_EINVAL, fn + ": a slice of a source is made with one pose");
    if (count > INT64_MAX / n_poses) return fail(BMO_EINVAL, fn + ": count * n_poses overflows int64");
    BMO_CUDA(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    std::unique_ptr<bmo_source, FreeWith<bmo_source_free>> s(new bmo_source());
    s->ctx = ctx; s->n_rays = desc->n_rays; s->n_poses = n_poses; s->n = count * n_poses; s->beamlets = true;
    const int64_t n = s->n;
    // the chief positions of one tile, by the ray source's own kernels
    DevBuf<double> pos, dir;
    BMO_CUDA(pos.alloc((size_t)count * 3, st));
    BMO_CUDA(dir.alloc(3, st));
    if ((rc = expand_rays(ctx, desc, 1, first, count, pos.get(), dir.get(), nullptr))) return rc;
    BMO_CUDA(dev_alloc(&s->rays, (size_t)n * 18, st));
    BMO_CUDA(dev_alloc(&s->w0, (size_t)n, st));
    BMO_CUDA(dev_alloc(&s->e0, (size_t)n * 2, st));
    if (n_poses > 1) BMO_CUDA(dev_alloc(&s->pose_id, (size_t)n, st));
    BeamletParams B{};
    B.pos = pos.get(); B.count = count; B.total = n;
    for (int i = 0; i < 3; i++) { B.dv[i] = bd->dv[i]; B.dd[i] = bd->dd[i]; B.s[i] = bd->s[i]; }
    B.w0 = bd->w0; B.div_offset = bd->div_offset; B.e0[0] = bd->E0[0]; B.e0[1] = bd->E0[1];
    B.rays = s->rays; B.w0_out = s->w0; B.e0_out = s->e0; B.pose_id = s->pose_id;
    source_beamlets<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(B);
    BMO_LAUNCH(ctx, "source_beamlets");
    *out = s.release();
    return BMO_OK;
}

int32_t bmo_source_beamlets_device(bmo_source* s, int64_t* n, const double** rays, const double** w0, const double** E0) {
    if (!s) return fail(BMO_EINVAL, "bmo_source_beamlets_device: source NULL");
    if (!s->beamlets) return fail(BMO_EINVAL, "bmo_source_beamlets_device: a ray source holds no beamlets (bmo_source_device)");
    if (n) *n = s->n;
    if (rays) *rays = s->rays;
    if (w0) *w0 = s->w0;
    if (E0) *E0 = s->e0;
    return BMO_OK;
}

int32_t bmo_source_beamlets(bmo_source* s, double* rays, double* w0, double* E0) {
    if (!s) return fail(BMO_EINVAL, "bmo_source_beamlets: source NULL");
    if (!s->beamlets) return fail(BMO_EINVAL, "bmo_source_beamlets: a ray source holds no beamlets (bmo_source_rays)");
    BMO_CUDA(cudaSetDevice(s->ctx->device));
    cudaStream_t st = s->ctx->stream;
    const size_t n = (size_t)s->n;
    if (rays) BMO_CUDA(cudaMemcpyAsync(rays, s->rays, n * 18 * sizeof(double), cudaMemcpyDeviceToHost, st));
    if (w0) BMO_CUDA(cudaMemcpyAsync(w0, s->w0, n * sizeof(double), cudaMemcpyDeviceToHost, st));
    if (E0) BMO_CUDA(cudaMemcpyAsync(E0, s->e0, n * 2 * sizeof(double), cudaMemcpyDeviceToHost, st));
    BMO_CUDA(cudaStreamSynchronize(st));
    return BMO_OK;
}

int32_t bmo_source_pose_ids(bmo_source* s, int32_t* n_poses, const int32_t** pose_id) {
    if (!s) return fail(BMO_EINVAL, "bmo_source_pose_ids: source NULL");
    if (n_poses) *n_poses = s->n_poses;
    if (pose_id) *pose_id = s->pose_id;
    return BMO_OK;
}

int32_t bmo_source_device(bmo_source* s, int64_t* n, const double** pos, const double** dir, int32_t* uniform_dir) {
    if (!s) return fail(BMO_EINVAL, "bmo_source_device: source NULL");
    if (s->beamlets) return fail(BMO_EINVAL, "bmo_source_device: a beamlet source holds no rays (bmo_source_beamlets_device)");
    if (n) *n = s->n;
    if (pos) *pos = s->pos;
    if (dir) *dir = s->dir;
    if (uniform_dir) *uniform_dir = s->uniform ? 1 : 0;
    return BMO_OK;
}

int32_t bmo_source_rays(bmo_source* s, double* pos, double* dir) {
    if (!s) return fail(BMO_EINVAL, "bmo_source_rays: source NULL");
    if (s->beamlets) return fail(BMO_EINVAL, "bmo_source_rays: a beamlet source holds no rays (bmo_source_beamlets)");
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

int32_t bmo::spot_check_result(const std::string& fn, const bmo_result* r, int32_t det_object) {
    if (!r) return fail(BMO_EINVAL, fn + ": NULL argument");
    if (det_object < 0 || det_object >= (int32_t)r->object_kind.size() || r->object_kind[det_object] != BMO_OBJ_SPOTDETECTOR)
        return fail(BMO_EINVAL, fn + ": object " + std::to_string(det_object) + " is not a Spotdetector of the result's system");
    return BMO_OK;
}

int32_t bmo::spot_check_args(const std::string& fn, const double* window, int32_t nx, int32_t nz, const void* counts) {
    if (window) {
        for (int i = 0; i < 4; i++)
            if (!std::isfinite(window[i])) return fail(BMO_EINVAL, fn + ": window not finite");
        if (!(window[1] > window[0]) || !(window[3] > window[2])) return fail(BMO_EINVAL, fn + ": window needs x_hi > x_lo and z_hi > z_lo");
    }
    if (counts) {
        if (!window) return fail(BMO_EINVAL, fn + ": a histogram needs a window");
        if (nx < 1 || nz < 1) return fail(BMO_EINVAL, fn + ": nx and nz must be >= 1");
    }
    return BMO_OK;
}

// bmo_spot_stats (one result, n_poses = 1: every entry, index order), bmo_spot_stats_poses (one result, n_poses = its pose
// count) and bmo_spot_stats_results (several results, n_poses = 1: their entries concatenated in list order)
int32_t bmo::spot_stats(const char* what, int32_t n_res, bmo_result* const* rs, int32_t det_object, int32_t n_poses, const double* window,
                        int32_t nx, int32_t nz, bmo_spot_info* out, int64_t* counts, uint32_t flags) {
    const std::string fn(what);
    if (!out) return fail(BMO_EINVAL, fn + ": NULL argument");
    int32_t rc;
    for (int32_t k = 0; k < n_res; k++) {
        if ((rc = spot_check_result(fn, rs[k], det_object))) return rc;
        if (rs[k]->ctx != rs[0]->ctx) return fail(BMO_EINVAL, fn + ": result " + std::to_string(k) + " belongs to another context than result 0");
    }
    if ((rc = spot_check_args(fn, window, nx, nz, counts))) return rc;
    bmo_result* r = rs[0];
    bmo_ctx* ctx = r->ctx;
    BMO_CUDA(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    // several results: the table of their spot arrays and first concatenated entries, closed by the total
    std::vector<SpotRes> rtab;
    int64_t n = 0;
    for (int32_t k = 0; k < n_res; k++) {
        if (n_res > 1) rtab.push_back({rs[k]->spot_obj, rs[k]->spot_xz, n});
        n += rs[k]->n_beams * rs[k]->R;
    }
    if (n_res > 1) rtab.push_back({nullptr, nullptr, n});
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
    DevBuf<int32_t> order;
    if (n_poses == 1) {
        P.per = spot_per(n);
        nblk = std::max<int64_t>(1, (n + P.per - 1) / P.per);
    } else {
        const int64_t nb = r->n_beams;
        if (nb > INT32_MAX) return fail(BMO_EINVAL, fn + ": more beams than a 32-bit beam id can number");
        DevBuf<unsigned long long> cnt;   // [n_poses] counts, then the flags word
        BMO_CUDA(cnt.alloc(np + 1, st));
        std::vector<unsigned long long> h(np + 1);
        BMO_CUDA(cudaMemsetAsync(cnt.get(), 0, (np + 1) * sizeof(unsigned long long), st));
        if (nb > 0) {
            const int64_t runs = (nb + POSE_RUN - 1) / POSE_RUN;
            spot_pose_count<<<(unsigned)((runs + 255) / 256), 256, 0, st>>>(r->pose, nb, n_poses, cnt.get(), (unsigned int*)(cnt.get() + np));
            BMO_LAUNCH(ctx, "spot_pose_count");
        }
        BMO_CUDA(cudaMemcpyAsync(h.data(), cnt.get(), (np + 1) * sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
        BMO_CUDA(cudaStreamSynchronize(st));
        cnt.reset();
        if (h[np] & 2u) return fail(BMO_EINVAL, fn + ": a beam of the result carries a pose id outside [0, n_poses)");
        if (h[np] & 1u) {   // not pose-major (beamsplitter children, or pose ids in any order): stable radix sort on the pose id
            DevBuf<int32_t> keys, iota;
            DevBuf<char> tmp;
            size_t tmp_bytes = 0;
            const int end_bit = 32 - __builtin_clz((unsigned)(n_poses - 1));
            BMO_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, tmp_bytes, (const int32_t*)r->pose, keys.get(), (const int32_t*)iota.get(), order.get(),
                                                     (int)nb, 0, end_bit, st));
            BMO_CUDA(order.alloc((size_t)nb, st));
            BMO_CUDA(keys.alloc((size_t)nb, st));
            BMO_CUDA(iota.alloc((size_t)nb, st));
            BMO_CUDA(tmp.alloc(tmp_bytes, st));
            iota32<<<(unsigned)((nb + 255) / 256), 256, 0, st>>>(iota.get(), nb);
            BMO_LAUNCH(ctx, "iota32");
            BMO_CUDA(cub::DeviceRadixSort::SortPairs(tmp.get(), tmp_bytes, (const int32_t*)r->pose, keys.get(), (const int32_t*)iota.get(), order.get(),
                                                     (int)nb, 0, end_bit, st));
            BMO_LAUNCH(ctx, "radix sort by pose");
        }
        tab.assign(2 * np + 1 + (np + 2) / 2, 0);
        int32_t* pblk = (int32_t*)(tab.data() + 2 * np + 1);
        for (size_t p = 0; p < np; p++) {
            const int64_t m = (int64_t)h[p] * r->R;
            const int64_t per = spot_per(m);
            tab[p + 1] = tab[p] + m;
            tab[np + 1 + p] = per;
            pblk[p] = (int32_t)nblk;
            nblk += std::max<int64_t>(1, (m + per - 1) / per);
        }
        pblk[np] = (int32_t)nblk;
        if (nblk > INT32_MAX) return fail(BMO_EINVAL, fn + ": too many blocks");
    }
    // one scratch block: partials, two completion counters per pose, the statistics, the histogram of a host `counts`, the
    // per-pose slice table, the result table
    const size_t off_done = (size_t)nblk * sizeof(SpotPartial), done_bytes = (8 * np + 15) / 16 * 16;
    const size_t off_out = off_done + done_bytes, off_hist = off_out + np * sizeof(bmo_spot_info);
    const size_t off_tab = off_hist + (counts && !dev_counts ? np * bins * sizeof(int64_t) : 0);
    const size_t off_res = off_tab + tab.size() * sizeof(int64_t);
    const size_t bytes = off_res + rtab.size() * sizeof(SpotRes);
    DevBuf<char> buf;
    BMO_CUDA(buf.alloc(bytes, st));
    char* scr = buf.get();
    P.part = (SpotPartial*)scr; P.done = (unsigned int*)(scr + off_done); P.out = (bmo_spot_info*)(scr + off_out);
    P.counts = counts ? (dev_counts ? (unsigned long long*)counts : (unsigned long long*)(scr + off_hist)) : nullptr;
    P.order = order.get();
    if (!tab.empty()) {
        P.pstart = (const int64_t*)(scr + off_tab); P.pper = P.pstart + np + 1; P.pblk = (const int32_t*)(P.pper + np);
        BMO_CUDA(cudaMemcpyAsync(scr + off_tab, tab.data(), tab.size() * sizeof(int64_t), cudaMemcpyHostToDevice, st));
    }
    if (!rtab.empty()) {
        P.res = (const SpotRes*)(scr + off_res); P.n_res = n_res;
        BMO_CUDA(cudaMemcpyAsync(scr + off_res, rtab.data(), rtab.size() * sizeof(SpotRes), cudaMemcpyHostToDevice, st));
    }
    BMO_CUDA(cudaMemsetAsync(P.done, 0, done_bytes, st));
    if (P.counts) BMO_CUDA(cudaMemsetAsync(P.counts, 0, np * bins * sizeof(int64_t), st));
    spot_sums<<<(unsigned)nblk, SPOT_BLOCK, 0, st>>>(P);
    BMO_LAUNCH(ctx, "spot_sums");
    spot_spread<<<(unsigned)nblk, SPOT_BLOCK, 0, st>>>(P);
    BMO_LAUNCH(ctx, "spot_spread");
    BMO_CUDA(cudaMemcpyAsync(out, P.out, np * sizeof(bmo_spot_info), cudaMemcpyDeviceToHost, st));
    if (counts && !dev_counts) BMO_CUDA(cudaMemcpyAsync(counts, P.counts, np * bins * sizeof(int64_t), cudaMemcpyDeviceToHost, st));
    BMO_CUDA(cudaStreamSynchronize(st));
    return BMO_OK;
}

int32_t bmo_spot_stats(bmo_result* r, int32_t det_object, const double* window, int32_t nx, int32_t nz, bmo_spot_info* out,
                       int64_t* counts, uint32_t flags) {
    NvtxRange nvtx_("bmo_spot_stats");
    return spot_stats("bmo_spot_stats", 1, &r, det_object, 1, window, nx, nz, out, counts, flags);
}

int32_t bmo_spot_stats_poses(bmo_result* r, int32_t det_object, int32_t n_poses, const double* window, int32_t nx, int32_t nz,
                             bmo_spot_info* out, int64_t* counts, uint32_t flags) {
    NvtxRange nvtx_("bmo_spot_stats_poses");
    if (r && n_poses != r->n_poses)
        return fail(BMO_EINVAL, "bmo_spot_stats_poses: n_poses " + std::to_string(n_poses) + " differs from the " +
                                    std::to_string(r->n_poses) + " poses the result was traced with");
    return spot_stats("bmo_spot_stats_poses", 1, &r, det_object, n_poses, window, nx, nz, out, counts, flags);
}

int32_t bmo_spot_stats_results(int32_t n_results, bmo_result* const* results, int32_t det_object, const double* window, int32_t nx,
                               int32_t nz, bmo_spot_info* out, int64_t* counts, uint32_t flags) {
    NvtxRange nvtx_("bmo_spot_stats_results");
    if (n_results < 1 || !results) return fail(BMO_EINVAL, "bmo_spot_stats_results: needs n_results >= 1 results");
    return spot_stats("bmo_spot_stats_results", n_results, results, det_object, 1, window, nx, nz, out, counts, flags);
}

int32_t bmo::spot_stats_shard(const std::string& fn, bmo_ctx* ctx, bmo_result* r, int32_t det_object, const double* window, int32_t nx,
                              int32_t nz, const std::vector<int64_t>& entries, int64_t per, SpotExchange& x, bmo_spot_info* out,
                              int64_t* counts, uint32_t flags) {
    BMO_CUDA(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    const int32_t W = (int32_t)entries.size();
    int64_t stride = 1;             // blocks of the largest rank: every rank's partials are padded to it for the all-gather
    for (int64_t m : entries) stride = std::max(stride, (m + per - 1) / per);
    const int64_t n = r ? r->n_beams * r->R : 0, nblk = (n + per - 1) / per;
    const size_t bins = counts ? (size_t)nx * (size_t)nz : 0;
    const bool dev_counts = counts && (flags & BMO_INPUT_DEVICE);
    // one scratch block: this rank's partials, every rank's, the entry counts, the statistics, the histogram of a host `counts`
    const size_t part_bytes = (size_t)stride * sizeof(SpotPartial);
    const size_t off_all = part_bytes, off_ent = off_all + (size_t)W * part_bytes, off_out = off_ent + (size_t)W * sizeof(int64_t);
    const size_t off_hist = off_out + sizeof(bmo_spot_info), bytes = off_hist + (counts && !dev_counts ? bins * sizeof(int64_t) : 0);
    DevBuf<char> buf;
    BMO_CUDA(buf.alloc(bytes, st));
    char* scr = buf.get();
    SpotParams P{};
    if (r) { P.obj = r->spot_obj; P.xz = r->spot_xz; P.R = r->R; }
    P.n = n; P.per = per; P.det = det_object; P.n_poses = 1;
    P.has_window = window != nullptr; P.nx = nx; P.nz = nz;
    if (window) for (int i = 0; i < 4; i++) P.win[i] = window[i];
    P.part = (SpotPartial*)scr; P.out = (bmo_spot_info*)(scr + off_out);
    P.counts = counts ? (dev_counts ? (unsigned long long*)counts : (unsigned long long*)(scr + off_hist)) : nullptr;
    const SpotPartial* all = (const SpotPartial*)(scr + off_all);
    const int64_t* ent = (const int64_t*)(scr + off_ent);
    int32_t rc;
    BMO_CUDA(cudaMemcpyAsync(scr + off_ent, entries.data(), (size_t)W * sizeof(int64_t), cudaMemcpyHostToDevice, st));
    if (P.counts) BMO_CUDA(cudaMemsetAsync(P.counts, 0, bins * sizeof(int64_t), st));
    // pass 1: this rank's sums; every rank combines all partials in global block order
    if (nblk) { spot_sums<<<(unsigned)nblk, SPOT_BLOCK, 0, st>>>(P); BMO_LAUNCH(ctx, "spot_sums"); }
    if ((rc = x.gather(P.part, scr + off_all, part_bytes))) return rc;
    spot_combine<<<1, 1, 0, st>>>(all, W, (int32_t)stride, ent, per, 0, P.out);
    BMO_LAUNCH(ctx, "spot_combine");
    // pass 2: the squared distances to the common centroid
    if (nblk) { spot_spread<<<(unsigned)nblk, SPOT_BLOCK, 0, st>>>(P); BMO_LAUNCH(ctx, "spot_spread"); }
    if ((rc = x.gather(P.part, scr + off_all, part_bytes))) return rc;
    spot_combine<<<1, 1, 0, st>>>(all, W, (int32_t)stride, ent, per, 1, P.out);
    BMO_LAUNCH(ctx, "spot_combine");
    // the histogram: integer counts, summed exactly
    if (P.counts && (rc = x.sum((int64_t*)P.counts, bins))) return rc;
    BMO_CUDA(cudaMemcpyAsync(out, P.out, sizeof(bmo_spot_info), cudaMemcpyDeviceToHost, st));
    if (counts && !dev_counts) BMO_CUDA(cudaMemcpyAsync(counts, P.counts, bins * sizeof(int64_t), cudaMemcpyDeviceToHost, st));
    BMO_CUDA(cudaStreamSynchronize(st));
    return BMO_OK;
}
