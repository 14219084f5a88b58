// bmo_source.cu -- ray sources expanded on the device and the spot-diagram reduction.
//
// Sources (bmo_source_create): the host hands over a descriptor -- basis, ring table, rotate3d matrices, every
// transcendental of the host constructors (BeamGroups.jl:51-100, 152-195, 222-245) -- and the device writes the rays the
// trace reads with BMO_INPUT_DEVICE, instead of 24-48 B per ray crossing the bus.
//   source_rings  one thread per ring (thread 0: ray 0).  Ray j of a ring comes from the serial recurrence v <- rot v in
//                 linalg.matvec's order ((a0 v0 + a1 v1) + a2 v2): bit-identical to the host loop.  A closed form
//                 rotate3d(d, j * delta) v would round differently.
//   source_disc   one thread per ray (Fibonacci disc); sin / cos are CUDA's, within a few ulp of the host's.
// Spot statistics (bmo_spot_stats): two passes over a fixed partition of the spot entries (spot_sums: counts, sums,
// extrema and the histogram; spot_spread: the squared distances to the centroid).  Each block reduces its slice in a
// fixed order and the last block to finish combines the per-block partials in block order, so the result does not depend
// on which blocks ran when.
// Compiled with -fmad=false; the arithmetic that must match the host bit for bit is spelled with __dmul_rn / __dadd_rn.
#include <cmath>
#include "bmo_host.cuh"

namespace bmo {

struct SrcParams {
    int64_t n, n_rings;
    int32_t kind;
    double p[3], d[3], e1[3], e2[3], radius, phi0;
    const bmo_source_ring* rings;
    double *pos, *dir;
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

__global__ void source_disc(SrcParams P) {
    const int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= P.n) return;
    if (k == 0) for (int i = 0; i < 3; i++) P.dir[i] = P.d[i];
    const double kd = (double)k;
    const double rho = __dsqrt_rn(__ddiv_rn(__dadd_rn(kd, 0.5), (double)P.n));
    const double phi = __dmul_rn(kd, P.phi0);
    const double r = __dmul_rn(P.radius, rho);
    double s, c;
    sincos(phi, &s, &c);
    const double rc = __dmul_rn(r, c), rs = __dmul_rn(r, s);
    for (int i = 0; i < 3; i++) P.pos[3 * k + i] = __dadd_rn(P.p[i], __dadd_rn(__dmul_rn(rc, P.e1[i]), __dmul_rn(rs, P.e2[i])));
}

// ---- spot statistics ------------------------------------------------------------------------------------------
constexpr int SPOT_BLOCK = 256;
constexpr int64_t SPOT_SLICE = 4096;     // entries per block (times a factor that keeps the grid at <= 1024 blocks)

struct SpotPartial { unsigned long long hits, outside; double sx, sz, maxr, lo[2], hi[2], ssq; };

struct SpotParams {
    const int32_t* obj; const double* xz;
    int64_t n, per;                 // entries, entries per block
    int32_t det, has_window, nx, nz;
    double win[4];
    unsigned long long* counts;     // NULL: no histogram
    SpotPartial* part;              // [gridDim.x]
    unsigned int* done;             // [2] blocks finished with spot_sums / spot_spread
    bmo_spot_info* out;             // device
};

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

// true in every thread of the block that finishes last (its partial and those of all other blocks are visible)
__device__ bool last_block(unsigned int* done) {
    __shared__ bool last;
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) last = atomicAdd(done, 1u) == gridDim.x - 1;
    __syncthreads();
    if (last) __threadfence();
    return last;
}

__global__ void __launch_bounds__(SPOT_BLOCK) spot_sums(SpotParams P) {
    __shared__ double shd[SPOT_BLOCK];
    __shared__ unsigned long long shu[SPOT_BLOCK];
    const int64_t b0 = (int64_t)blockIdx.x * P.per, b1 = min(P.n, b0 + P.per);
    unsigned long long hits = 0, outside = 0;
    double sx = 0, sz = 0, maxr = -INFINITY, lox = INFINITY, loz = INFINITY, hix = -INFINITY, hiz = -INFINITY;
    for (int64_t k = b0 + threadIdx.x; k < b1; k += SPOT_BLOCK) {
        if (P.obj[k] != P.det) continue;
        const double x = P.xz[2 * k], z = P.xz[2 * k + 1];
        hits++;
        sx = __dadd_rn(sx, x); sz = __dadd_rn(sz, z);
        maxr = fmax(maxr, __dsqrt_rn(__dadd_rn(__dmul_rn(x, x), __dmul_rn(z, z))));
        lox = fmin(lox, x); hix = fmax(hix, x); loz = fmin(loz, z); hiz = fmax(hiz, z);
        if (P.has_window) {
            if (!(x >= P.win[0] && x <= P.win[1] && z >= P.win[2] && z <= P.win[3])) { outside++; continue; }
            if (P.counts) {
                const double fi = floor(__dmul_rn(__ddiv_rn(__dsub_rn(x, P.win[0]), __dsub_rn(P.win[1], P.win[0])), (double)P.nx));
                const double fj = floor(__dmul_rn(__ddiv_rn(__dsub_rn(z, P.win[2]), __dsub_rn(P.win[3], P.win[2])), (double)P.nz));
                const int64_t i = min((int64_t)fi, (int64_t)P.nx - 1), j = min((int64_t)fj, (int64_t)P.nz - 1);
                atomicAdd(P.counts + j * P.nx + i, 1ull);
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
    if (!last_block(P.done) || threadIdx.x != 0) return;
    // combine in block order
    const volatile SpotPartial* vp = P.part;
    unsigned long long H = 0, O = 0;
    double SX = 0, SZ = 0, M = -INFINITY, L0 = INFINITY, L1 = INFINITY, U0 = -INFINITY, U1 = -INFINITY;
    for (unsigned b = 0; b < gridDim.x; b++) {
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
    *P.out = o;
}

__global__ void __launch_bounds__(SPOT_BLOCK) spot_spread(SpotParams P) {
    __shared__ double shd[SPOT_BLOCK];
    if (P.out->hits == 0) return;   // every block sees the same count: nothing to do, rms stays NaN
    const double cx = P.out->centroid[0], cz = P.out->centroid[1];
    const int64_t b0 = (int64_t)blockIdx.x * P.per, b1 = min(P.n, b0 + P.per);
    double s = 0;
    for (int64_t k = b0 + threadIdx.x; k < b1; k += SPOT_BLOCK) {
        if (P.obj[k] != P.det) continue;
        const double dx = __dsub_rn(P.xz[2 * k], cx), dz = __dsub_rn(P.xz[2 * k + 1], cz);
        s = __dadd_rn(s, __dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dz, dz)));
    }
    s = block_reduce(s, shd, AddD());
    if (threadIdx.x == 0) P.part[blockIdx.x].ssq = s;
    if (!last_block(P.done + 1) || threadIdx.x != 0) return;
    const volatile SpotPartial* vp = P.part;
    double S = 0;
    for (unsigned b = 0; b < gridDim.x; b++) S = __dadd_rn(S, vp[b].ssq);
    P.out->rms = __dsqrt_rn(__ddiv_rn(S, (double)P.out->hits));
}

}  // namespace bmo

using namespace bmo;

struct bmo_source {
    bmo_ctx* ctx = nullptr;
    int64_t n = 0;
    bool uniform = false;
    double* pos = nullptr;   // [n][3]
    double* dir = nullptr;   // [n][3], or [3] when uniform
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
    delete s;
    return BMO_OK;
}

int32_t bmo_source_create(bmo_ctx* ctx, const bmo_source_desc* desc, bmo_source** out) {
    NvtxRange nvtx_("bmo_source_create");
    if (!ctx || !desc || !out) return fail(BMO_EINVAL, "bmo_source_create: NULL argument");
    int32_t rc;
    if ((rc = check_desc(desc))) return rc;
    BMO_CUDA(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    bmo_source* s = new bmo_source();
    s->ctx = ctx; s->n = desc->n_rays; s->uniform = desc->kind != BMO_SRC_POINT;
    const int64_t n = s->n;
    SrcParams P{};
    P.n = n; P.n_rings = desc->n_rings; P.kind = desc->kind;
    for (int i = 0; i < 3; i++) { P.p[i] = desc->pos[i]; P.d[i] = desc->dir[i]; P.e1[i] = desc->e1[i]; P.e2[i] = desc->e2[i]; }
    P.radius = desc->radius; P.phi0 = desc->phi0;
    bmo_source_ring* d_rings = nullptr;
    cudaError_t e = dev_alloc(&s->pos, (size_t)n * 3, st);
    if (e == cudaSuccess) e = dev_alloc(&s->dir, s->uniform ? (size_t)3 : (size_t)n * 3, st);
    if (e == cudaSuccess && desc->kind != BMO_SRC_DISC && desc->n_rings > 0) {
        e = dev_alloc(&d_rings, (size_t)desc->n_rings, st);
        if (e == cudaSuccess) e = cudaMemcpyAsync(d_rings, desc->rings, (size_t)desc->n_rings * sizeof(bmo_source_ring), cudaMemcpyHostToDevice, st);
    }
    if (e != cudaSuccess) {
        dev_free(d_rings, st);
        bmo_source_free(s);
        return fail(BMO_ECUDA, std::string("bmo_source_create: ") + cudaGetErrorString(e));
    }
    P.rings = d_rings; P.pos = s->pos; P.dir = s->dir;
    if (desc->kind == BMO_SRC_DISC) {
        source_disc<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(P);
        rc = launched(ctx, "source_disc");
    } else {
        source_rings<<<(unsigned)((desc->n_rings + 1 + 63) / 64), 64, 0, st>>>(P);
        rc = launched(ctx, "source_rings");
    }
    dev_free(d_rings, st);
    if (rc) { bmo_source_free(s); return rc; }
    *out = s;
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

int32_t bmo_spot_stats(bmo_result* r, int32_t det_object, const double* window, int32_t nx, int32_t nz, bmo_spot_info* out,
                       int64_t* counts, uint32_t flags) {
    NvtxRange nvtx_("bmo_spot_stats");
    if (!r || !out) return fail(BMO_EINVAL, "bmo_spot_stats: NULL argument");
    if (det_object < 0 || det_object >= (int32_t)r->object_kind.size() || r->object_kind[det_object] != BMO_OBJ_SPOTDETECTOR)
        return fail(BMO_EINVAL, "bmo_spot_stats: object " + std::to_string(det_object) + " is not a Spotdetector of the result's system");
    if (window) {
        for (int i = 0; i < 4; i++)
            if (!std::isfinite(window[i])) return fail(BMO_EINVAL, "bmo_spot_stats: window not finite");
        if (!(window[1] > window[0]) || !(window[3] > window[2])) return fail(BMO_EINVAL, "bmo_spot_stats: window needs x_hi > x_lo and z_hi > z_lo");
    }
    if (counts) {
        if (!window) return fail(BMO_EINVAL, "bmo_spot_stats: a histogram needs a window");
        if (nx < 1 || nz < 1) return fail(BMO_EINVAL, "bmo_spot_stats: nx and nz must be >= 1");
    }
    bmo_ctx* ctx = r->ctx;
    BMO_CUDA(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    const int64_t n = r->n_beams * r->R;
    const int64_t per = SPOT_SLICE * std::max<int64_t>(1, (n + SPOT_SLICE * 1024 - 1) / (SPOT_SLICE * 1024));
    const int64_t nblk = std::max<int64_t>(1, (n + per - 1) / per);
    const size_t bins = counts ? (size_t)nx * (size_t)nz : 0;
    const bool dev_counts = counts && (flags & BMO_INPUT_DEVICE);
    // one scratch block: partials, two completion counters, the statistics, the histogram of a host `counts`
    const size_t off_done = (size_t)nblk * sizeof(SpotPartial), off_out = off_done + 16, off_hist = off_out + sizeof(bmo_spot_info);
    const size_t bytes = off_hist + (counts && !dev_counts ? bins * sizeof(int64_t) : 0);
    char* scr = nullptr;
    BMO_CUDA(dev_alloc(&scr, bytes, st));
    SpotParams P{};
    P.obj = r->spot_obj; P.xz = r->spot_xz; P.n = n; P.per = per; P.det = det_object;
    P.has_window = window != nullptr; P.nx = nx; P.nz = nz;
    if (window) for (int i = 0; i < 4; i++) P.win[i] = window[i];
    P.part = (SpotPartial*)scr; P.done = (unsigned int*)(scr + off_done); P.out = (bmo_spot_info*)(scr + off_out);
    P.counts = counts ? (dev_counts ? (unsigned long long*)counts : (unsigned long long*)(scr + off_hist)) : nullptr;
    cudaError_t e = cudaMemsetAsync(P.done, 0, 16, st);
    if (e == cudaSuccess && P.counts) e = cudaMemsetAsync(P.counts, 0, bins * sizeof(int64_t), st);
    int32_t rc = BMO_OK;
    if (e == cudaSuccess) {
        spot_sums<<<(unsigned)nblk, SPOT_BLOCK, 0, st>>>(P);
        rc = launched(ctx, "spot_sums");
        if (!rc) {
            spot_spread<<<(unsigned)nblk, SPOT_BLOCK, 0, st>>>(P);
            rc = launched(ctx, "spot_spread");
        }
        if (!rc) e = cudaMemcpyAsync(out, P.out, sizeof(bmo_spot_info), cudaMemcpyDeviceToHost, st);
        if (!rc && e == cudaSuccess && counts && !dev_counts) e = cudaMemcpyAsync(counts, P.counts, bins * sizeof(int64_t), cudaMemcpyDeviceToHost, st);
        if (!rc && e == cudaSuccess) e = cudaStreamSynchronize(st);
    }
    dev_free(scr, st);
    if (rc) return rc;
    if (e != cudaSuccess) return fail(BMO_ECUDA, std::string("bmo_spot_stats: ") + cudaGetErrorString(e));
    return BMO_OK;
}
