// bmo_psf.cu -- PSFDetector (OpticalComponents/Detectors/PSFDetector.jl): collection of the ray hits a
// trace left on the detector and the coherent point-spread-function sum.
//
//   interact3d(::AbstractSystem, ::PSFDetector, ::Beam{T, Ray{T}}, ::Ray) (:77-89) stores, per hit,
//   position, direction, optical_path_length(beam), |dir . normal| and 2pi/lambda  -> psf_flag / psf_build
//   (a GaussianBeamlet reaches it through the generic interact3d, Gaussian.jl:124-135: one record each for
//   the chief, waist and divergence beam)
//   calc_local_pos / calc_local_lims (:91-141)                                      -> psf_local / psf_reduce
//   intensity(psf; n, ...) (:190-237): I[i, j] = | sum_h proj_h cis(k_h (opl_h + (p_ij - hit_h) . dir_h)) |^2
//                                                                                  -> psf_intensity_kernel
// The tracer treats the detector like every other absorbing object (interact3d returns nothing); the
// records are rebuilt here from the segment table, so a trace needs BMO_KEEP_SEGMENTS.
// Compiled with FMA contraction (tolerance of the path: 1e-8 relative L2 of the intensity map).
#include <cstdlib>
#include "bmo_host.cuh"

namespace bmo {

enum { S_PX = 0, S_PY, S_PZ, S_DX, S_DY, S_DZ, S_N, S_T, S_NX, S_NY, S_NZ };   // segment rows (bmo_trace.cu)

struct PsfView {
    const double* seg_d; const int32_t* seg_part; int64_t rows; int nsd;   // segment table: row records [rows][nsd]
    const int32_t *nseg, *status, *lam, *parent;
    const long long* first_seg;
    const double* popl;    // beamlets: OPL of the parent's chief beam (the tracer's running sum, also read by K4)
    int64_t n_beams;
    int rays;              // rows per segment: 1, or 3 for beamlets (chief, waist, divergence interleaved)
};

// flags[b] = 1 if beam b ended on object `psf` (its last stored ray -- a beamlet's chief ray -- has an intersection with it).
// A torn or clipped beamlet never reached interact3d (System.jl:288-304): its status is not BMO_ST_ABSORBED.
__global__ void psf_flag(PsfView R, SysView S, int psf_object, int32_t* flags) {
    const int64_t b = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= R.n_beams) return;
    int f = 0;
    if ((R.status[b] & 0xff) == BMO_ST_ABSORBED && R.nseg[b] > 0) {
        const int part = R.seg_part[(R.first_seg[b] + R.nseg[b] - 1) * R.rays];
        if (part >= 0 && S.parts[part].object == psf_object) f = 1;
    }
    flags[b] = f;
}
// optical_path_length(beam) (Beam.jl:137-149): the parent's OPL first, then the beam's own rays in order.  The ancestor of
// each generation is found by walking up from b again (O(depth^2) parent reads, paid only by deep records), so a beam tree of
// any depth sums root first without a fixed-size chain.
__device__ double beam_opl(const PsfView& R, int b) {
    int depth = 0;
    for (int c = R.parent[b]; c >= 0; c = R.parent[c]) depth++;
    double l0 = 0.0;
    for (int d = depth; d >= 0; d--) {
        int c = b;
        for (int u = 0; u < d; u++) c = R.parent[c];
        const int64_t f = R.first_seg[c];
        for (int s = 0; s < R.nseg[c]; s++) {
            const double t = R.seg_d[(size_t)(f + s) * R.nsd + S_T];
            if (isinf(t)) break;
            l0 += t * R.seg_d[(size_t)(f + s) * R.nsd + S_N];
        }
    }
    return l0;
}
// optical_path_length of ray q of beamlet b (Beam.jl:137-149): only the chief beam has a parent (Gaussian.jl:107-111), whose
// OPL the tracer kept in popl; then the beam's own rows in order.  No walk up the beamlet tree, so its depth is unbounded.
__device__ double beamlet_opl(const PsfView& R, int64_t b, int q) {
    double l0 = q == 0 ? R.popl[b] : 0.0;
    const int64_t f = R.first_seg[b];
    for (int s = 0; s < R.nseg[b]; s++) {
        const int64_t row = (f + s) * 3 + q;
        const double t = R.seg_d[(size_t)row * R.nsd + S_T];
        if (isinf(t)) break;
        l0 += t * R.seg_d[(size_t)row * R.nsd + S_N];
    }
    return l0;
}
// one thread per record: record q of flagged beam b goes to base + rays * offs[b] + q (a beamlet: chief, waist, divergence)
__global__ void psf_build(PsfView R, SysView S, const int32_t* flags, const long long* offs, int64_t base, double* rec, double* fast) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= R.n_beams * R.rays) return;
    const int64_t b = i / R.rays;
    const int q = (int)(i - b * R.rays);
    if (!flags[b]) return;
    const int64_t row = (R.first_seg[b] + R.nseg[b] - 1) * R.rays + q;
    const double* d = R.seg_d;
    const V3 pos = mk3(d[(size_t)(row) * R.nsd + S_PX], d[(size_t)(row) * R.nsd + S_PY], d[(size_t)(row) * R.nsd + S_PZ]);
    const V3 dir = mk3(d[(size_t)(row) * R.nsd + S_DX], d[(size_t)(row) * R.nsd + S_DY], d[(size_t)(row) * R.nsd + S_DZ]);
    const V3 nrm = mk3(d[(size_t)(row) * R.nsd + S_NX], d[(size_t)(row) * R.nsd + S_NY], d[(size_t)(row) * R.nsd + S_NZ]);
    const double t = d[(size_t)(row) * R.nsd + S_T];
    const V3 hit = pos + t * dir;
    const double opl = R.rays == 1 ? beam_opl(R, (int)b) : beamlet_opl(R, b, q);
    const double proj = fabs(dot(dir, nrm));
    const double k = kTwoPi / S.lambdas[R.lam[b]];
    const int64_t o = base + R.rays * offs[b] + q;
    double* r = rec + o * PSF_NREC;
    r[0] = hit.x; r[1] = hit.y; r[2] = hit.z; r[3] = dir.x; r[4] = dir.y; r[5] = dir.z; r[6] = opl; r[7] = proj; r[8] = k;
    double* qf = fast + o * PSF_NFAST;
    qf[0] = k * (opl - dot(hit, dir)); qf[1] = k * dir.x; qf[2] = k * dir.y; qf[3] = k * dir.z; qf[4] = proj;
}

// local (x, z) of every hit (calc_local_pos, PSFDetector.jl:91-101)
__global__ void psf_local(const double* rec, int64_t n, const double* dp, double* xs, double* zs) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const double* r = rec + i * PSF_NREC;
    const V3 loc = mk3(r[0] - dp[0], r[1] - dp[1], r[2] - dp[2]);
    xs[i] = dot(loc, mk3(dp[3], dp[6], dp[9]));     // orientation[:, 1]
    zs[i] = dot(loc, mk3(dp[5], dp[8], dp[11]));    // orientation[:, 3]
}
// single-block reductions for calc_local_lims (:112-141).  mode 0: out = (sum w, sum w x, sum w z, min x, max x, min z, max z);
// mode 1: out = (max |x - x0|, max |z - z0|)
__global__ void __launch_bounds__(512) psf_reduce(const double* rec, const double* xs, const double* zs, int64_t n, int mode, double x0, double z0, double* out) {
    __shared__ double s[7][512];
    double a[7] = {0, 0, 0, INFINITY, -INFINITY, INFINITY, -INFINITY};
    if (mode == 1) { a[0] = 0; a[1] = 0; }
    for (int64_t i = threadIdx.x; i < n; i += blockDim.x) {
        const double x = xs[i], z = zs[i];
        if (mode == 0) {
            const double w = rec[i * PSF_NREC + 7];
            a[0] += w; a[1] += w * x; a[2] += w * z;
            a[3] = fmin(a[3], x); a[4] = fmax(a[4], x); a[5] = fmin(a[5], z); a[6] = fmax(a[6], z);
        } else { a[0] = fmax(a[0], fabs(x - x0)); a[1] = fmax(a[1], fabs(z - z0)); }
    }
    for (int k = 0; k < 7; k++) s[k][threadIdx.x] = a[k];
    __syncthreads();
    for (int o = blockDim.x / 2; o > 0; o >>= 1) {
        if (threadIdx.x < o) {
            if (mode == 0) {
                for (int k = 0; k < 3; k++) s[k][threadIdx.x] += s[k][threadIdx.x + o];
                s[3][threadIdx.x] = fmin(s[3][threadIdx.x], s[3][threadIdx.x + o]); s[4][threadIdx.x] = fmax(s[4][threadIdx.x], s[4][threadIdx.x + o]);
                s[5][threadIdx.x] = fmin(s[5][threadIdx.x], s[5][threadIdx.x + o]); s[6][threadIdx.x] = fmax(s[6][threadIdx.x], s[6][threadIdx.x + o]);
            } else {
                s[0][threadIdx.x] = fmax(s[0][threadIdx.x], s[0][threadIdx.x + o]); s[1][threadIdx.x] = fmax(s[1][threadIdx.x], s[1][threadIdx.x + o]);
            }
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) for (int k = 0; k < (mode == 0 ? 7 : 2); k++) out[k] = s[k][0];
}

// ---- K6: PSF sum, one thread per pixel, hit records staged through shared memory ---------------------
// Per pixel-hit pair: phase = c0_h + p . (k dir)_h  (= k (opl + (p - hit) . dir), PSFDetector.jl:229-230, with
// the hit-only terms folded into c0), sincos of the O(1e6 rad) phase by the Cody-Waite reduction of
// bmo_math.cuh, acc += proj (cos, sin): 3 FMA + 17 FMA-class + 2 FMA, FP64-pipe bound.
constexpr int PSF_TX = 32, PSF_TY = 8, PSF_BATCH = 256;
struct PsfParams {
    const double* fast; int64_t n_hits;
    const double* dp;            // detector pose: pos(3), dir(9 row-major)
    double x_lo, x_hi, z_lo, z_hi, x_shift, z_shift;
    int32_t n, j0, j1, pad;      // columns [j0, j1) of the n x n map
    double* out;                 // [n][j1 - j0] column-major [i + n*(j - j0)]
};
BMO_D double lin_coord(int i, int n, double lo, double hi) {   // LinRange getindex (Base.lerpi)
    const double t = n == 1 ? 0.0 : (double)i / (double)(n - 1);
    return (1 - t) * lo + t * hi;
}
__global__ void __launch_bounds__(PSF_TX* PSF_TY, 4) psf_intensity_kernel(const PsfParams P) {
    __shared__ double s_h[PSF_BATCH * PSF_NFAST];
    const int i = blockIdx.x * PSF_TX + threadIdx.x, j = P.j0 + blockIdx.y * PSF_TY + threadIdx.y;
    const int tid = threadIdx.y * PSF_TX + threadIdx.x;
    const bool inside = i < P.n && j < P.j1;
    const double x = lin_coord(min(i, P.n - 1), P.n, P.x_lo, P.x_hi) + P.x_shift;
    const double z = lin_coord(min(j, P.n - 1), P.n, P.z_lo, P.z_hi) + P.z_shift;
    const double* dp = P.dp;
    // p = origin + x e1 + z e2 (:226)
    const double px = dp[0] + x * dp[3] + z * dp[5], py = dp[1] + x * dp[6] + z * dp[8], pz = dp[2] + x * dp[9] + z * dp[11];
    double are = 0.0, aim = 0.0;
    for (int64_t h0 = 0; h0 < P.n_hits; h0 += PSF_BATCH) {
        const int m = (int)min((int64_t)PSF_BATCH, P.n_hits - h0);
        __syncthreads();
        for (int w = tid; w < m * PSF_NFAST; w += PSF_TX * PSF_TY) s_h[w] = P.fast[h0 * PSF_NFAST + w];
        __syncthreads();
#pragma unroll 2
        for (int h = 0; h < m; h++) {
            const double* q = s_h + h * PSF_NFAST;
            const double phase = fma(px, q[1], fma(py, q[2], fma(pz, q[3], q[0])));
            double sn, cs;
            sincos_reduced(phase, &sn, &cs);
            are = fma(q[4], cs, are);
            aim = fma(q[4], sn, aim);
        }
    }
    if (inside) P.out[(int64_t)i + (int64_t)P.n * (j - P.j0)] = are * are + aim * aim;
}

}  // namespace bmo

using namespace bmo;

namespace bmo { __global__ void scan_flags(const int32_t* in, int64_t n, long long* out, long long* total); }

int32_t bmo::psf_reserve(bmo_psf* p, int64_t need, cudaStream_t st) {
    if (need <= p->cap) return BMO_OK;
    const int64_t cap = std::max<int64_t>(need, 2 * p->cap);
    DevBuf<double> nr, nf;
    BMO_CUDA(nr.alloc((size_t)cap * PSF_NREC, st));
    BMO_CUDA(nf.alloc((size_t)cap * PSF_NFAST, st));
    if (p->n > 0) {
        BMO_CUDA(cudaMemcpyAsync(nr.get(), p->rec, (size_t)p->n * PSF_NREC * sizeof(double), cudaMemcpyDeviceToDevice, st));
        BMO_CUDA(cudaMemcpyAsync(nf.get(), p->fast, (size_t)p->n * PSF_NFAST * sizeof(double), cudaMemcpyDeviceToDevice, st));
    }
    dev_free(p->rec, st); dev_free(p->fast, st);
    p->rec = nr.release(); p->fast = nf.release(); p->cap = cap;
    return BMO_OK;
}

static int32_t psf_check(bmo_sys* sys, int32_t psf_object, const char* who) {
    if (!sys) return fail(BMO_EINVAL, std::string(who) + ": sys NULL");
    if (psf_object < 0 || psf_object >= (int)sys->objects.size() || sys->objects[psf_object].kind != BMO_OBJ_PSFDETECTOR)
        return fail(BMO_EINVAL, std::string(who) + ": object is not a PSFDetector");
    return BMO_OK;
}

int32_t bmo_psf_collect(bmo_sys* sys, bmo_result* r, int32_t psf_object, bmo_psf** psf, int64_t* n_total) {
    int32_t rc;
    if ((rc = psf_check(sys, psf_object, "bmo_psf_collect"))) return rc;
    if (!r || !psf) return fail(BMO_EINVAL, "bmo_psf_collect: NULL argument");
    if (!r->keep || !r->seg_d) return fail(BMO_ESTATE, "bmo_psf_collect: the result has no segment table (trace with BMO_KEEP_SEGMENTS)");
    bmo_ctx* ctx = sys->ctx;
    BMO_CUDA(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    std::unique_ptr<bmo_psf, FreeWith<bmo_psf_free>> fresh;   // a new record set: the caller's once the call succeeds
    if (!*psf) { fresh.reset(new bmo_psf()); fresh->ctx = ctx; }
    bmo_psf* p = *psf ? *psf : fresh.get();
    if (p->ctx != ctx) return fail(BMO_EINVAL, "bmo_psf_collect: detector data lives on another context");
    if (r->mode != 1) {   // PolarizedRay: no interact3d method -> no data (AbstractSystem.jl:30-33)
        const int64_t nb = r->n_beams;
        DevBuf<int32_t> d_flags;
        DevBuf<long long> d_offs;
        BMO_CUDA(d_flags.alloc((size_t)nb, st));
        BMO_CUDA(d_offs.alloc((size_t)nb, st));
        PsfView v;
        v.seg_d = r->seg_d; v.seg_part = r->seg_part; v.rows = r->seg_rows; v.nsd = r->nsd; v.nseg = r->nseg; v.status = r->status; v.lam = r->lam;
        v.parent = r->parent; v.first_seg = r->first_seg; v.popl = r->popl; v.n_beams = nb; v.rays = r->mode == 2 ? 3 : 1;
        psf_flag<<<(unsigned)((nb + 255) / 256), 256, 0, st>>>(v, sys->view, psf_object, d_flags.get());
        BMO_LAUNCH(ctx, "psf_flag");
        scan_flags<<<1, 1024, 0, st>>>(d_flags.get(), nb, d_offs.get(), ctx->d_totals);
        BMO_LAUNCH(ctx, "scan_flags");
        BMO_CUDA(cudaMemcpyAsync(ctx->h_totals, ctx->d_totals, sizeof(long long), cudaMemcpyDeviceToHost, st));
        BMO_CUDA(cudaStreamSynchronize(st));
        const int64_t m = ctx->h_totals[0] * v.rays;    // records: one per ray of every flagged beam
        if (m > 0) {
            if ((rc = psf_reserve(p, p->n + m, st))) return rc;
            psf_build<<<(unsigned)((nb * v.rays + 255) / 256), 256, 0, st>>>(v, sys->view, d_flags.get(), d_offs.get(), p->n, p->rec, p->fast);
            BMO_LAUNCH(ctx, "psf_build");
            p->n += m;
        }
        BMO_CUDA(cudaStreamSynchronize(st));
    }
    if (fresh) *psf = fresh.release();
    if (n_total) *n_total = p->n;
    return BMO_OK;
}

int32_t bmo_psf_data(bmo_psf* p, double* records) {
    if (!p || !records) return fail(BMO_EINVAL, "bmo_psf_data: NULL argument");
    BMO_CUDA(cudaSetDevice(p->ctx->device));
    BMO_CUDA(cudaMemcpyAsync(records, p->rec, (size_t)p->n * PSF_NREC * sizeof(double), cudaMemcpyDeviceToHost, p->ctx->stream));
    BMO_CUDA(cudaStreamSynchronize(p->ctx->stream));
    return BMO_OK;
}

int32_t bmo_psf_lims(bmo_sys* sys, bmo_psf* p, int32_t psf_object, int32_t pose, double crop_factor, int32_t center, double* lims) {
    int32_t rc;
    if ((rc = psf_check(sys, psf_object, "bmo_psf_lims"))) return rc;
    if (!p || !lims) return fail(BMO_EINVAL, "bmo_psf_lims: NULL argument");
    if (p->n == 0) return fail(BMO_ESTATE, "bmo_psf_lims: the detector holds no data");
    if (pose < 0 || pose >= sys->view.n_poses) return fail(BMO_EINVAL, "bmo_psf_lims: pose out of range");
    bmo_ctx* ctx = sys->ctx;
    BMO_CUDA(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    DevBuf<double> xs, zs, d_out;
    BMO_CUDA(xs.alloc((size_t)p->n, st)); BMO_CUDA(zs.alloc((size_t)p->n, st)); BMO_CUDA(d_out.alloc(8, st));
    const double* dp = sys->view.det_pose + 12 * ((int64_t)pose * sys->view.n_objects + psf_object);
    psf_local<<<(unsigned)((p->n + 255) / 256), 256, 0, st>>>(p->rec, p->n, dp, xs.get(), zs.get());
    BMO_LAUNCH(ctx, "psf_local");
    psf_reduce<<<1, 512, 0, st>>>(p->rec, xs.get(), zs.get(), p->n, 0, 0.0, 0.0, d_out.get());
    BMO_LAUNCH(ctx, "psf_reduce");
    double h[7];
    BMO_CUDA(cudaMemcpyAsync(h, d_out.get(), sizeof(h), cudaMemcpyDeviceToHost, st));
    BMO_CUDA(cudaStreamSynchronize(st));
    double x0, z0;
    if (center == 0) { x0 = h[1] / h[0]; z0 = h[2] / h[0]; }          // :122-125 projection-weighted centroid
    else { x0 = (h[3] + h[4]) / 2; z0 = (h[5] + h[6]) / 2; }           // :127-128 bounding-box midpoint
    psf_reduce<<<1, 512, 0, st>>>(p->rec, xs.get(), zs.get(), p->n, 1, x0, z0, d_out.get());
    BMO_LAUNCH(ctx, "psf_reduce");
    BMO_CUDA(cudaMemcpyAsync(h, d_out.get(), 2 * sizeof(double), cudaMemcpyDeviceToHost, st));
    BMO_CUDA(cudaStreamSynchronize(st));
    const double hwx = h[0] * crop_factor, hwz = h[1] * crop_factor;
    lims[0] = x0 - hwx; lims[1] = x0 + hwx; lims[2] = z0 - hwz; lims[3] = z0 + hwz;
    return BMO_OK;
}

// bmo_psf_intensity's argument checks (`who` names the caller in the message)
int32_t bmo::psf_intensity_check(const char* who, bmo_sys* sys, const bmo_psf* p, int32_t psf_object, int32_t pose, int32_t n,
                                 const double* lims, const double* intensity) {
    int32_t rc;
    if ((rc = psf_check(sys, psf_object, who))) return rc;
    if (!p || !lims || !intensity) return fail(BMO_EINVAL, std::string(who) + ": NULL argument");
    if (n < 1) return fail(BMO_EINVAL, std::string(who) + ": n must be >= 1");
    if (pose < 0 || pose >= sys->view.n_poses) return fail(BMO_EINVAL, std::string(who) + ": pose out of range");
    return BMO_OK;
}

// K6 on columns [j0, j1) of the map, enqueued on the context's stream between evk0 and evk1; no launch for an empty range
int32_t bmo::psf_intensity_band(bmo_sys* sys, const bmo_psf* p, int32_t psf_object, int32_t pose, int32_t n, const double* lims,
                                double x0_shift, double z0_shift, int32_t j0, int32_t j1, double* d_out) {
    if (j1 == j0) return BMO_OK;
    bmo_ctx* ctx = sys->ctx;
    cudaStream_t st = ctx->stream;
    PsfParams pp{};
    pp.fast = p->fast; pp.n_hits = p->n; pp.dp = sys->view.det_pose + 12 * ((int64_t)pose * sys->view.n_objects + psf_object);
    pp.x_lo = lims[0]; pp.x_hi = lims[1]; pp.z_lo = lims[2]; pp.z_hi = lims[3]; pp.x_shift = x0_shift; pp.z_shift = z0_shift;
    pp.n = n; pp.j0 = j0; pp.j1 = j1; pp.out = d_out;
    dim3 grid((n + PSF_TX - 1) / PSF_TX, (j1 - j0 + PSF_TY - 1) / PSF_TY), block(PSF_TX, PSF_TY);
    BMO_CUDA(cudaEventRecord(ctx->evk0, st));
    psf_intensity_kernel<<<grid, block, 0, st>>>(pp);
    BMO_LAUNCH(ctx, "psf_intensity");
    BMO_CUDA(cudaEventRecord(ctx->evk1, st));
    ctx->psf_pairs += (int64_t)n * (j1 - j0) * p->n;
    return BMO_OK;
}

// bmo_psf_intensity and bmo_psf_intensity_cols: columns [j0, j1) to a host or device buffer of n * (j1 - j0) doubles
static int32_t psf_intensity_cols(const char* who, bmo_sys* sys, bmo_psf* p, int32_t psf_object, int32_t pose, int32_t n, const double* lims,
                                  double x0_shift, double z0_shift, int32_t j0, int32_t j1, double* intensity, uint32_t flags) {
    int32_t rc;
    if ((rc = psf_intensity_check(who, sys, p, psf_object, pose, n, lims, intensity))) return rc;
    if (!(0 <= j0 && j0 <= j1 && j1 <= n)) return fail(BMO_EINVAL, std::string(who) + ": column range outside 0 <= j0 <= j1 <= n");
    if (j1 == j0) return BMO_OK;
    bmo_ctx* ctx = sys->ctx;
    BMO_CUDA(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    const bool on_dev = flags & BMO_INPUT_DEVICE;
    const size_t n_out = (size_t)n * (size_t)(j1 - j0);
    double* d_out = intensity;
    DevBuf<double> out_copy;   // of a host map
    if (!on_dev) {
        BMO_CUDA(out_copy.alloc(n_out, st));
        d_out = out_copy.get();
    }
    if ((rc = psf_intensity_band(sys, p, psf_object, pose, n, lims, x0_shift, z0_shift, j0, j1, d_out))) return rc;
    if (!on_dev) BMO_CUDA(cudaMemcpyAsync(intensity, d_out, n_out * sizeof(double), cudaMemcpyDeviceToHost, st));
    BMO_CUDA(cudaStreamSynchronize(st));
    float kms = 0;
    BMO_CUDA(cudaEventElapsedTime(&kms, ctx->evk0, ctx->evk1));
    ctx->psf_ms = kms;
    return BMO_OK;
}

int32_t bmo_psf_intensity(bmo_sys* sys, bmo_psf* p, int32_t psf_object, int32_t pose, int32_t n, const double* lims, double x0_shift,
                          double z0_shift, double* intensity, uint32_t flags) {
    NvtxRange nvtx_("bmo_psf_intensity");
    return psf_intensity_cols("bmo_psf_intensity", sys, p, psf_object, pose, n, lims, x0_shift, z0_shift, 0, n, intensity, flags);
}

int32_t bmo_psf_intensity_cols(bmo_sys* sys, bmo_psf* p, int32_t psf_object, int32_t pose, int32_t n, const double* lims, double x0_shift,
                               double z0_shift, int32_t j0, int32_t j1, double* intensity, uint32_t flags) {
    NvtxRange nvtx_("bmo_psf_intensity_cols");
    return psf_intensity_cols("bmo_psf_intensity_cols", sys, p, psf_object, pose, n, lims, x0_shift, z0_shift, j0, j1, intensity, flags);
}

int32_t bmo_psf_count(bmo_psf* p, int64_t* n) {
    if (!p || !n) return fail(BMO_EINVAL, "bmo_psf_count: NULL argument");
    *n = p->n;
    return BMO_OK;
}

int32_t bmo_psf_free(bmo_psf* p) {
    if (!p) return BMO_OK;
    cudaSetDevice(p->ctx->device);
    dev_free(p->rec, p->ctx->stream); dev_free(p->fast, p->ctx->stream);
    delete p;
    return BMO_OK;
}
