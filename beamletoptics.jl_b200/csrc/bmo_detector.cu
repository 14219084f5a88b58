// bmo_detector.cu -- Photodetector: coherent superposition of Gaussian beamlet fields (K4).
//
// Restates interact3d(::Photodetector, ::GaussianBeamlet, ray_id) (Photodetector.jl:69-107) ->
// electric_field(gauss, r, z) (Gaussian.jl:381-392) -> point_on_beam (Beam.jl:177-205) +
// gauss_parameters (Gaussian.jl:298-353) -> electric_field(r, z, E0, w0, w, k, psi, R)
// (OpticUtils.jl:87-89), one thread per pixel, beamlet records staged through shared memory.
// Two kernels:
//   pd_field_fast (default)  the per-pair arithmetic is strength-reduced: along one chief segment the
//       waist / divergence ray heights are affine in the arclength s (y0_r = A_r + s B_r), so the two
//       line-plane intersections, the normalisations and tan(pi/2 - acos(c)) collapse to
//       m_r = c_r / sqrt(1 - c_r^2) with c_r^2 = (alpha_r + s beta_r)^2 / |y0_r|^2; the local waist w0
//       cancels out of E0 (w0_beam / w0) * w0 / w; the Gouy phase enters as (cos psi, sin psi) =
//       (sqrt(1 - R zeta), -+ sqrt(R zeta)) instead of atan2 + sincos; k z (O(1e7) rad) is reduced by
//       2 pi with two FMAs before sincos.  Algebraically identical to the reference, rounding differs
//       at the 1e-9 rad level (the reference's own k*z carries 1 ulp(1e7) = 2e-9 rad); tolerance of
//       the path: 1e-8 relative L2 (north_star).  Pixels whose z falls on an earlier chief segment
//       (tilted detectors, Beam.jl:186-199) take the reference-order path below.
//   pd_field (BMO_PD_REFERENCE_ORDER)  every pair evaluated in the reference's operation order;
//       kept as the cross-check of the fast kernel at full detector sizes.
#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>
#include "bmo_host.cuh"
#include "bmo_interact.cuh"

namespace bmo {

// segment table rows (must match bmo_trace.cu)
enum { S_PX = 0, S_PY, S_PZ, S_DX, S_DY, S_DZ, S_N, S_T, S_NX, S_NY, S_NZ };

// One leaf beamlet that ends on the detector.  Plain doubles so a tile can be copied to smem as words.
struct PdRec {
    double p0[3], d0[3];      // chief ray of the last segment (ray_id)
    double wp[3], wd[3];      // waist ray
    double dp[3], dd[3];      // divergence ray
    double cn;                // refractive index of the chief segment
    double l0;                // length(gauss) - length(ray)              (Photodetector.jl:74)
    double temp;              // cumulative length before the last segment (Beam.jl:179-199, parent-first sum)
    double plen;              // length(parent)
    double lambda, k;         // wavelength, 2pi/lambda                   (Gaussian.jl:384)
    double w0b, e0r, e0i;     // beam_waist(gauss), electric_field(gauss)
    double cr, ci;            // exp(im * ref_phi), ref_phi = (OPL - L)/lambda * 2pi   (Gaussian.jl:388-391)
    double sq;                // sqrt(|d0 . n_hit|)                       (Photodetector.jl:84,103)
    double first_row;         // first chief row of this beam in the segment table (as double; slow path)
    double nseg;
    double pose;
    double pad;
};
static_assert(sizeof(PdRec) % 8 == 0, "PdRec must be a whole number of doubles");

// Strength-reduced record of the same beamlet (last chief segment), see pd_field_fast.
struct PdFast {
    double p0[3], d0[3];
    double Ad[3], Bd[3], alpd, betd;   // divergence ray: y0(s) = Ad + s Bd, (y0 . dir_d)/|dir_d| = alpd + s betd
    double Aw[3], Bw[3], alpw, betw;   // waist ray
    double l0, temp, k;
    double cre, cim;                   // E0_beam * w0_beam * sqrt(proj) * exp(i ref_phi)
    double multi;                      // > 0: the beam has earlier segments (z < temp must be checked)
    double generic;                    // > 0: degenerate geometry, use the reference-order path for every pixel
    double pad;
};
static_assert(sizeof(PdFast) % 8 == 0, "PdFast must be a whole number of doubles");

struct ResView {
    const double* seg_d; const int32_t* seg_part; int64_t rows; int nsd;   // segment table: row records [rows][nsd]
    const int32_t *nseg, *status, *lam, *pose;
    const long long* first_seg;
    const double *w0, *e0, *plen, *popl;
    int64_t n_beams;
};

// flags[b] = 1 if beam b of a pose in [pose_lo, pose_hi) ended on detector `pd` after a full interaction (all three rays on
// the PD shape)
__global__ void pd_flag(ResView R, SysView S, int pd_object, int pose_lo, int pose_hi, int32_t* flags) {
    const int64_t b = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= R.n_beams) return;
    int f = 0;
    if ((R.status[b] & 0xff) == BMO_ST_ABSORBED && R.nseg[b] > 0 && R.pose[b] >= pose_lo && R.pose[b] < pose_hi) {
        const int64_t row = (R.first_seg[b] + R.nseg[b] - 1) * 3;
        const int part = R.seg_part[row];
        if (part >= 0 && S.parts[part].object == pd_object) f = 1;
    }
    flags[b] = f;
}
__global__ void pd_build(ResView R, SysView S, const int32_t* flags, const long long* offs, PdRec* recs) {
    const int64_t b = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= R.n_beams || !flags[b]) return;
    PdRec rc;
    const int n = R.nseg[b];
    const int64_t f = R.first_seg[b];
    const int nsd = R.nsd;
    const double plen = R.plen[b], popl = R.popl[b];
    // running sums with the reference's association (Beam.jl:125-205)
    double lsum = 0.0, lpar = plen, opl = popl;
    for (int s = 0; s < n - 1; s++) {
        const int64_t row = (f + s) * 3;
        const double t = R.seg_d[(size_t)(row) * nsd + S_T], nn = R.seg_d[(size_t)(row) * nsd + S_N];
        lsum += t; lpar += t; opl += t * nn;
    }
    const int64_t rc_ = (f + n - 1) * 3, rw = rc_ + 1, rd = rc_ + 2;
    const double* d = R.seg_d;
    const double t_last = d[(size_t)(rc_) * nsd + S_T];
    rc.cn = d[(size_t)(rc_) * nsd + S_N];
    for (int k = 0; k < 3; k++) {
        rc.p0[k] = d[(size_t)(rc_) * nsd + (S_PX + k)]; rc.d0[k] = d[(size_t)(rc_) * nsd + (S_DX + k)];
        rc.wp[k] = d[(size_t)(rw) * nsd + (S_PX + k)]; rc.wd[k] = d[(size_t)(rw) * nsd + (S_DX + k)];
        rc.dp[k] = d[(size_t)(rd) * nsd + (S_PX + k)]; rc.dd[k] = d[(size_t)(rd) * nsd + (S_DX + k)];
    }
    const double L = (lsum + t_last) + plen;          // length(gauss) = l + l0
    const double OPL = opl + t_last * rc.cn;           // optical_path_length(gauss)
    rc.l0 = L - t_last;
    rc.temp = lpar;
    rc.plen = plen;
    rc.lambda = S.lambdas[R.lam[b]];
    rc.k = kTwoPi / rc.lambda;
    rc.w0b = R.w0[b]; rc.e0r = R.e0[2 * b]; rc.e0i = R.e0[2 * b + 1];
    const double dl = OPL - L;
    const double ref_phi = dl / rc.lambda * kTwoPi;
    Cx c = cis(ref_phi);
    rc.cr = c.re; rc.ci = c.im;
    V3 nrm = mk3(d[(size_t)(rc_) * nsd + S_NX], d[(size_t)(rc_) * nsd + S_NY], d[(size_t)(rc_) * nsd + S_NZ]);
    rc.sq = sqrt(fabs(dot(mk3(rc.d0[0], rc.d0[1], rc.d0[2]), nrm)));
    rc.first_row = (double)f; rc.nseg = (double)n; rc.pose = (double)R.pose[b]; rc.pad = 0;
    recs[offs[b]] = rc;
}
// Grouping the records of a sweep by pose, on the device (pd_run):
//   pd_pose_count  cnt[p - pose0] = records of pose p (the beams flagged by pd_flag), and *unsorted = 1 when some beam's pose id
//                  is smaller than its predecessor's.  Records are numbered in beam order, so without such a beam they are
//                  already grouped; the test looks at every beam, flagged or not, which can only ask for a sort that was not needed.
//   pd_pose_keys   (pose - pose0, record index) of every record: the pairs a stable radix sort orders by pose
//   pd_gather      out[i] = in[order[i]]
__global__ void pd_pose_count(const int32_t* pose, const int32_t* flags, int64_t nb, int32_t pose0, unsigned long long* cnt,
                              long long* unsorted) {
    const int64_t b0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) * POSE_RUN, b1 = min(nb, b0 + POSE_RUN);
    int32_t cur = -1;
    unsigned long long c = 0;
    bool down = false;
    for (int64_t b = b0; b < b1; b++) {
        const int32_t p = pose[b];
        down |= b > 0 && pose[b - 1] > p;
        if (!flags[b]) continue;
        if (p != cur && c) { atomicAdd(cnt + (cur - pose0), c); c = 0; }
        cur = p; c++;
    }
    add_pose_count(cnt, cur - pose0, c, c > 0);
    if (down) *unsorted = 1;
}
__global__ void pd_pose_keys(const int32_t* pose, const int32_t* flags, const long long* offs, int64_t nb, int32_t pose0, int32_t* keys,
                             int32_t* idx) {
    const int64_t b = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= nb || !flags[b]) return;
    const long long q = offs[b];
    keys[q] = pose[b] - pose0;
    idx[q] = (int32_t)q;
}
__global__ void pd_gather(const PdRec* in, const int32_t* order, PdRec* out, int64_t m) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < m) out[i] = in[order[i]];
}

// PdRec -> PdFast (after the records have been grouped by pose)
__global__ void pd_make_fast(const PdRec* recs, PdFast* fast, int64_t m) {
    const int64_t b = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= m) return;
    const PdRec rc = recs[b];
    const int n = (int)rc.nseg;
    PdFast fr;
    const V3 p0 = mk3(rc.p0[0], rc.p0[1], rc.p0[2]), d0 = mk3(rc.d0[0], rc.d0[1], rc.d0[2]);
    fr.generic = 0.0;
    for (int q = 0; q < 2; q++) {
        const V3 rp = q == 0 ? mk3(rc.dp[0], rc.dp[1], rc.dp[2]) : mk3(rc.wp[0], rc.wp[1], rc.wp[2]);
        const V3 rd = q == 0 ? mk3(rc.dd[0], rc.dd[1], rc.dd[2]) : mk3(rc.wd[0], rc.wd[1], rc.wd[2]);
        const double denom = dot(d0, rd);                     // line_plane_distance3d, LinearAlgebraUtils.jl:127-136
        if (!(fabs(denom) > 1e-6)) fr.generic = 1.0;
        const double a = dot(p0 - rp, d0) / denom, bq = dot(d0, d0) / denom;   // il(s) = a + s bq for point = p0 + s d0
        const V3 A = rp + a * rd - p0, B = bq * rd - d0;
        const double ind = 1.0 / norm(rd);
        double* Ao = q == 0 ? fr.Ad : fr.Aw; double* Bo = q == 0 ? fr.Bd : fr.Bw;
        Ao[0] = A.x; Ao[1] = A.y; Ao[2] = A.z; Bo[0] = B.x; Bo[1] = B.y; Bo[2] = B.z;
        (q == 0 ? fr.alpd : fr.alpw) = dot(A, rd) * ind;
        (q == 0 ? fr.betd : fr.betw) = dot(B, rd) * ind;
    }
    for (int k = 0; k < 3; k++) { fr.p0[k] = rc.p0[k]; fr.d0[k] = rc.d0[k]; }
    fr.l0 = rc.l0; fr.temp = rc.temp; fr.k = rc.k;
    const Cx C = ((mkc(rc.e0r, rc.e0i) * rc.w0b) * mkc(rc.cr, rc.ci)) * rc.sq;
    fr.cre = C.re; fr.cim = C.im;
    fr.multi = n > 1 ? 1.0 : 0.0;
    fr.pad = 0;
    fast[b] = fr;
}

constexpr int PD_TILE = 16;   // 16 x 16 pixels per block
constexpr int PD_BATCH = 32;  // beamlet records staged per smem tile

struct PdParams {
    const PdRec* recs; const PdFast* fast; int64_t n_recs;
    ResView R;
    double* field;            // [n_fields][n*n*2] column-major [i + n*j], re/im interleaved
    const double* det_pose;   // [n_poses][n_objects][12]
    const long long* pose_off;// NULL (single field) or [n_fields+1] record ranges per pose
    int32_t n, pd_object, n_objects, pose0;
    double lo, hi;
};

// LinRange getindex: lerpi(i, n-1, lo, hi) = (1 - t)*lo + t*hi, t = i/(n-1)
BMO_D double lin_coord(int i, int n, double lo, double hi) {
    const double t = (n == 1) ? 0.0 : (double)i / (double)(n - 1);
    return (1 - t) * lo + t * hi;
}

// One pixel-beamlet pair in the reference's operation order (Photodetector.jl:98-103, Beam.jl:177-205,
// Gaussian.jl:298-353, 381-392, OpticUtils.jl:87-89)
BMO_NI Cx pd_pair_reference(const PdRec& rc, V3 p1, const double* seg_d, int nsd) {
    const V3 p0 = mk3(rc.p0[0], rc.p0[1], rc.p0[2]), d0 = mk3(rc.d0[0], rc.d0[1], rc.d0[2]);
    // projection of the pixel onto the beamlet axis (Photodetector.jl:98-101)
    const double l1 = dot(p1 - p0, d0);
    const V3 p2 = p0 + l1 * d0;
    const double r = norm(p1 - p2);
    const double z = rc.l0 + l1;
    // point_on_beam(gauss, z) (Beam.jl:177-205)
    V3 point, c_dir = d0, w_pos = mk3(rc.wp[0], rc.wp[1], rc.wp[2]), w_dir = mk3(rc.wd[0], rc.wd[1], rc.wd[2]),
              d_pos = mk3(rc.dp[0], rc.dp[1], rc.dp[2]), d_dir = mk3(rc.dd[0], rc.dd[1], rc.dd[2]);
    double c_n = rc.cn;
    bool found = false;
    if (rc.nseg > 1.0 && z < rc.temp) {   // an earlier segment: replay the reference's loop
        const int ns = (int)rc.nseg;
        const int64_t f = (int64_t)rc.first_row;
        const double* d = seg_d;
        double temp = rc.plen;
        for (int s = 0; s < ns - 1; s++) {
            const int64_t row = (f + s) * 3;
            const double len = d[(size_t)(row) * nsd + S_T];
            temp += len;
            if (z < temp) {
                const double b = temp - z;
                const V3 sp = mk3(d[(size_t)(row) * nsd + S_PX], d[(size_t)(row) * nsd + S_PY], d[(size_t)(row) * nsd + S_PZ]);
                c_dir = mk3(d[(size_t)(row) * nsd + S_DX], d[(size_t)(row) * nsd + S_DY], d[(size_t)(row) * nsd + S_DZ]);
                point = sp + (len - b) * c_dir;
                c_n = d[(size_t)(row) * nsd + S_N];
                w_pos = mk3(d[(size_t)(row + 1) * nsd + S_PX], d[(size_t)(row + 1) * nsd + S_PY], d[(size_t)(row + 1) * nsd + S_PZ]);
                w_dir = mk3(d[(size_t)(row + 1) * nsd + S_DX], d[(size_t)(row + 1) * nsd + S_DY], d[(size_t)(row + 1) * nsd + S_DZ]);
                d_pos = mk3(d[(size_t)(row + 2) * nsd + S_PX], d[(size_t)(row + 2) * nsd + S_PY], d[(size_t)(row + 2) * nsd + S_PZ]);
                d_dir = mk3(d[(size_t)(row + 2) * nsd + S_DX], d[(size_t)(row + 2) * nsd + S_DY], d[(size_t)(row + 2) * nsd + S_DZ]);
                found = true;
                break;
            }
        }
    }
    if (!found) point = p0 + (z - rc.temp) * d0;
    double w, Rc, psi, w0;
    gauss_parameters(point, c_dir, c_n, w_pos, w_dir, d_pos, d_dir, rc.lambda, w, Rc, psi, w0);
    // electric_field(gauss, r, z) (Gaussian.jl:381-392, OpticUtils.jl:87-89)
    const Cx E0 = mkc(rc.e0r, rc.e0i) * (rc.w0b / w0);
    Cx e = ((E0 * w0) / w) * exp(-(r * r) / (w * w));
    e = e * cis(rc.k * z + psi + (rc.k * (r * r) * Rc) / 2);
    e = e * mkc(rc.cr, rc.ci);
    return e * rc.sq;
}

// pixel (i, j) -> world: p1 = dir' * (x, 0, y) + pos   (Photodetector.jl:78,92-96 -- transposed orientation)
BMO_D V3 pd_pixel(const double* dp, int i, int j, int n, double lo, double hi) {
    const double x = lin_coord(min(i, n - 1), n, lo, hi), y = lin_coord(min(j, n - 1), n, lo, hi);
    // T = transpose(dir): T[r][c] = dir[c][r]; dir row-major at dp[3 + 3*r + c]
    return mk3(dp[3 + 0] * x + dp[3 + 6] * y + dp[0],      // T[1,1]*x + T[1,3]*y + p[1]
               dp[3 + 1] * x + dp[3 + 7] * y + dp[1],      // T[2,1]*x + T[2,3]*y + p[2]
               dp[3 + 2] * x + dp[3 + 8] * y + dp[2]);     // T[3,1]*x + T[3,3]*y + p[3]
}

__global__ void __launch_bounds__(PD_TILE* PD_TILE) pd_field(const PdParams P) {
    __shared__ PdRec s_rec[PD_BATCH];
    const int i = blockIdx.x * PD_TILE + threadIdx.x, j = blockIdx.y * PD_TILE + threadIdx.y;
    const int tid = threadIdx.y * PD_TILE + threadIdx.x;
    const int fld = blockIdx.z;
    const int pose = P.pose0 + fld;
    const bool inside = i < P.n && j < P.n;
    const V3 p1 = pd_pixel(P.det_pose + 12 * ((int64_t)pose * P.n_objects + P.pd_object), i, j, P.n, P.lo, P.hi);
    int64_t rb = 0, re = P.n_recs;
    if (P.pose_off) { rb = P.pose_off[fld]; re = P.pose_off[fld + 1]; }
    Cx acc = mkc(0, 0);
    for (int64_t base = rb; base < re; base += PD_BATCH) {
        const int nb = (int)min((int64_t)PD_BATCH, re - base);
        __syncthreads();
        {
            const int nw = nb * (int)(sizeof(PdRec) / 8);
            const double* src = reinterpret_cast<const double*>(P.recs + base);
            double* dst = reinterpret_cast<double*>(s_rec);
            for (int k = tid; k < nw; k += PD_TILE * PD_TILE) dst[k] = src[k];
        }
        __syncthreads();
        if (!inside) continue;
        for (int q = 0; q < nb; q++) acc = acc + pd_pair_reference(s_rec[q], p1, P.R.seg_d, P.R.nsd);
    }
    if (inside) {
        double* f = P.field + ((int64_t)fld * P.n * P.n + (int64_t)i + (int64_t)P.n * j) * 2;
        f[0] += acc.re;
        f[1] += acc.im;
    }
}

constexpr int PDF_TX = 32, PDF_TY = 8;   // 256 threads; each thread owns PX pixels (rows j, j + 8, ...) of a 32 x (8 PX) tile
constexpr int PDF_BATCH = 48;                        // beamlet records per shared-memory tile

// Reciprocal, reciprocal square root and square root for the detector kernel: the hardware approximation (MUFU, 2^-22)
// followed by ONE Newton step in FMAs -- relative error < 1e-13, four to six FP64 instructions instead of the ten to fourteen
// of the correctly rounded library routines (which add a second Newton step and a fix-up).  The field is held to 1e-8 relative
// L2; arguments are positive and far from the subnormal range (squared lengths in metres, 1 - cos^2).  0 -> NaN (the library
// returns Inf): the waist-plane guards below treat both alike (Gaussian.jl:348-351).
BMO_D double rcp13(double x) {
    double y;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(x));
    const double e = fma(-x, y, 1.0);
    return fma(y, e, y);
}
BMO_D double rsqrt13(double x) {
    double y;
    asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(x));
    const double e = fma(-x * y, y, 1.0);
    return fma(0.5 * y, e, y);
}
BMO_D double sqrt13(double x) { return x > 0.0 ? x * rsqrt13(x) : (x == 0.0 ? 0.0 : NAN); }

BMO_D Cx pd_pair_fast(const PdFast& rc, V3 p1, bool& slow) {
    const double vx = p1.x - rc.p0[0], vy = p1.y - rc.p0[1], vz = p1.z - rc.p0[2];
    const double l1 = vx * rc.d0[0] + vy * rc.d0[1] + vz * rc.d0[2];
    const double qx = vx - l1 * rc.d0[0], qy = vy - l1 * rc.d0[1], qz = vz - l1 * rc.d0[2];   // p1 - p2
    const double r2 = qx * qx + qy * qy + qz * qz;
    const double z = rc.l0 + l1;
    slow = rc.generic > 0.0 || (rc.multi > 0.0 && z < rc.temp);
    const double s = z - rc.temp;
    // ray heights / slopes in the plane through point_on_beam(z), perpendicular to the chief
    const double ydx = rc.Ad[0] + s * rc.Bd[0], ydy = rc.Ad[1] + s * rc.Bd[1], ydz = rc.Ad[2] + s * rc.Bd[2];
    const double ywx = rc.Aw[0] + s * rc.Bw[0], ywy = rc.Aw[1] + s * rc.Bw[1], ywz = rc.Aw[2] + s * rc.Bw[2];
    const double y2d = ydx * ydx + ydy * ydy + ydz * ydz, y2w = ywx * ywx + ywy * ywy + ywz * ywz;
    const double nd = rc.alpd + s * rc.betd, nw = rc.alpw + s * rc.betw;
    // cos^2 of the angle between height vector and ray, c_r^2 = n_r^2 / y_r^2: one reciprocal serves both
    // (NaN at y = 0, like the reference's y0 / 0)
    const double ip = rcp13(y2d * y2w);
    double c2d = (nd * nd) * (y2w * ip), c2w = (nw * nw) * (y2d * ip);
    c2d = c2d > 1.0 ? 1.0 : c2d; c2w = c2w > 1.0 ? 1.0 : c2w;  // clamp of angle3d (LinearAlgebraUtils.jl:103-108)
    const double id = rsqrt13(1.0 - c2d), iw = rsqrt13(1.0 - c2w);
    const double E = nd * id + nw * iw;                          // E_kt = y_d m_d + y_w m_w
    const double F2 = c2d * (id * id) + c2w * (iw * iw);         // F_kt^2 = m_d^2 + m_w^2
    const double rw = rsqrt13(y2d + y2w);                        // 1 / w
    const double iw2 = rw * rw;
    double R = E * iw2;                                          // curvature E_kt / w^2
    // psi = -atan2(1, sqrt(1/(R zeta) - 1)), R zeta = E^2 / (w^2 F^2):  sin|psi| = |E| / (w F), cos psi = sqrt(1 - sin^2)
    double spsi = fabs(E) * rw * rsqrt13(F2);
    spsi = spsi > 1.0 ? 1.0 : spsi;
    double cpsi = sqrt13(1.0 - spsi * spsi);
    if (!(R < 0.0)) spsi = -spsi;                                // R < 0 flips the sign of psi
    if (isnan(R)) R = 0.0;                                       // Gaussian.jl:348-351
    if (isnan(spsi) || isnan(cpsi)) { cpsi = 1.0; spsi = 0.0; }
    const double amp = rw * exp_neg(-r2 * iw2);                  // (w0 / w) exp(-r^2/w^2) with w0 cancelled against E0
    double sn, cs;
    sincos_reduced(rc.k * z + (rc.k * r2 * R) * 0.5, &sn, &cs);
    const double re = cs * cpsi - sn * spsi, im = sn * cpsi + cs * spsi;
    return mkc((rc.cre * re - rc.cim * im) * amp, (rc.cre * im + rc.cim * re) * amp);
}

// One pixel per thread, 3 resident blocks per SM (80 registers): the fastest configuration measured (DESIGN §5).
constexpr int PDF_PX = 1;
__global__ void __launch_bounds__(PDF_TX* PDF_TY, 3) pd_field_fast(const PdParams P) {
    __shared__ PdFast s_rec[PDF_BATCH];
    const int tid = threadIdx.y * PDF_TX + threadIdx.x;
    const int i = blockIdx.x * PDF_TX + threadIdx.x;
    const int j0 = blockIdx.y * (PDF_TY * PDF_PX) + threadIdx.y;
    const int fld = blockIdx.z;
    const int pose = P.pose0 + fld;
    const double* dp = P.det_pose + 12 * ((int64_t)pose * P.n_objects + P.pd_object);
    V3 p1[PDF_PX];
    Cx acc[PDF_PX];
    bool inside[PDF_PX];
#pragma unroll
    for (int u = 0; u < PDF_PX; u++) {
        const int j = j0 + u * PDF_TY;
        inside[u] = i < P.n && j < P.n;
        p1[u] = pd_pixel(dp, i, j, P.n, P.lo, P.hi);
        acc[u] = mkc(0, 0);
    }
    int64_t rb = 0, re = P.n_recs;
    if (P.pose_off) { rb = P.pose_off[fld]; re = P.pose_off[fld + 1]; }
    for (int64_t base = rb; base < re; base += PDF_BATCH) {
        const int nb = (int)min((int64_t)PDF_BATCH, re - base);
        __syncthreads();
        {
            const int nw = nb * (int)(sizeof(PdFast) / 8);
            const double* src = reinterpret_cast<const double*>(P.fast + base);
            double* dst = reinterpret_cast<double*>(s_rec);
            for (int k = tid; k < nw; k += PDF_TX * PDF_TY) dst[k] = src[k];
        }
        __syncthreads();
        // Pairs that need the reference-order routine (the pixel's z falls on an earlier chief segment, degenerate geometry) are
        // only noted here, one bit per record of the batch, and evaluated after the batch: the out-of-line call and the
        // registers it forces the compiler to save stay out of the pair loop.  The sum then takes those pairs last, which
        // changes its rounding at the 1e-16 level (the field is held to 1e-8 relative L2).
        unsigned long long later[PDF_PX];
#pragma unroll
        for (int u = 0; u < PDF_PX; u++) later[u] = 0ull;
        static_assert(PDF_BATCH <= 64, "one bit per record of a batch");
        for (int q = 0; q < nb; q++) {
#pragma unroll
            for (int u = 0; u < PDF_PX; u++) {
                bool slow;
                const Cx e = pd_pair_fast(s_rec[q], p1[u], slow);
                if (slow) later[u] |= 1ull << q;
                else acc[u] = acc[u] + e;
            }
        }
#pragma unroll
        for (int u = 0; u < PDF_PX; u++) {
            unsigned long long m = later[u];
            while (m) {
                const int q = __ffsll((long long)m) - 1;
                m &= m - 1;
                acc[u] = acc[u] + pd_pair_reference(P.recs[base + q], p1[u], P.R.seg_d, P.R.nsd);
            }
        }
    }
#pragma unroll
    for (int u = 0; u < PDF_PX; u++) {
        if (!inside[u]) continue;
        const int j = j0 + u * PDF_TY;
        double* f = P.field + ((int64_t)fld * P.n * P.n + (int64_t)i + (int64_t)P.n * j) * 2;
        f[0] += acc[u].re;
        f[1] += acc[u].im;
    }
}

// optical_power = trapz((x, y), |E|^2 / (2 Z0)) (Photodetector.jl:109-116, Trapz.jl) in two steps:
//   pd_power_columns  one warp per pixel column j: s_j = sum_i (x_{i+1} - x_i) (I_ij + I_{i+1,j}) / 2, lanes stride over i so that
//                     a warp reads consecutive complex values (the field is stored [i + n j]); grid = (column groups, fields)
//   pd_power_reduce   one block per field: sum_j (y_{j+1} - y_j) (s_j + s_{j+1}) / 2
// Deterministic (no atomics); the order of the additions differs from a serial loop at the 1e-16 level.
constexpr int PWR_WARPS = 8;
__global__ void __launch_bounds__(32 * PWR_WARPS) pd_power_columns(const double* fields, int n, double lo, double hi, double* s_col) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int j = blockIdx.x * PWR_WARPS + warp;
    if (j >= n) return;
    const double* f = fields + ((int64_t)blockIdx.y * n * n + (int64_t)n * j) * 2;
    double s = 0;
    for (int i = lane; i + 1 < n; i += 32) {
        const double2 a = *reinterpret_cast<const double2*>(f + 2 * i), b = *reinterpret_cast<const double2*>(f + 2 * i + 2);
        const double ia = (a.x * a.x + a.y * a.y) / (2 * kZvac), ib = (b.x * b.x + b.y * b.y) / (2 * kZvac);
        s += (lin_coord(i + 1, n, lo, hi) - lin_coord(i, n, lo, hi)) * (ia + ib) / 2;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if (lane == 0) s_col[(int64_t)blockIdx.y * n + j] = s;
}
__global__ void __launch_bounds__(256) pd_power_reduce(const double* s_col, int n, double lo, double hi, double* power) {
    __shared__ double s_w[8];
    const double* c = s_col + (int64_t)blockIdx.x * n;
    double p = 0;
    for (int j = threadIdx.x; j + 1 < n; j += 256) p += (lin_coord(j + 1, n, lo, hi) - lin_coord(j, n, lo, hi)) * (c[j] + c[j + 1]) / 2;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) p += __shfl_xor_sync(0xffffffffu, p, o);
    if ((threadIdx.x & 31) == 0) s_w[threadIdx.x >> 5] = p;
    __syncthreads();
    if (threadIdx.x == 0) {
        double t = 0;
        for (int k = 0; k < 8; k++) t += s_w[k];
        power[blockIdx.x] = t;
    }
}
// both steps on stream st; d_power: [n_fields] on the device
static int32_t pd_power_launch(bmo_ctx* ctx, const double* d_fields, int n_fields, int n, double lo, double hi, double* d_power, cudaStream_t st) {
    DevBuf<double> s_col;
    BMO_CUDA(s_col.alloc((size_t)n_fields * n, st));
    pd_power_columns<<<dim3((n + PWR_WARPS - 1) / PWR_WARPS, n_fields), 32 * PWR_WARPS, 0, st>>>(d_fields, n, lo, hi, s_col.get());
    BMO_LAUNCH(ctx, "pd_power_columns");
    pd_power_reduce<<<n_fields, 256, 0, st>>>(s_col.get(), n, lo, hi, d_power);
    BMO_LAUNCH(ctx, "pd_power_reduce");
    return BMO_OK;
}

__global__ void scan_flags(const int32_t* in, int64_t n, long long* out, long long* total);

}  // namespace bmo

using namespace bmo;

// single-block chunked exclusive scan (same scheme as scan_counts in bmo_trace.cu)
__global__ void __launch_bounds__(1024) bmo::scan_flags(const int32_t* in, int64_t n, long long* out, long long* total) {
    __shared__ long long s_sum[1024];
    const int T = blockDim.x;
    const int64_t chunk = (n + T - 1) / T;
    const int64_t b = (int64_t)threadIdx.x * chunk, e = min(b + chunk, n);
    long long s = 0;
    for (int64_t i = b; i < e; i++) s += in[i];
    s_sum[threadIdx.x] = s;
    __syncthreads();
    for (int o = 1; o < T; o <<= 1) {
        long long v = threadIdx.x >= o ? s_sum[threadIdx.x - o] : 0;
        __syncthreads();
        s_sum[threadIdx.x] += v;
        __syncthreads();
    }
    long long run = threadIdx.x == 0 ? 0 : s_sum[threadIdx.x - 1];
    for (int64_t i = b; i < e; i++) { out[i] = run; run += in[i]; }
    if (threadIdx.x == T - 1) *total = s_sum[T - 1];
}

static ResView res_view(bmo_result* r) {
    ResView v;
    v.seg_d = r->seg_d; v.seg_part = r->seg_part; v.rows = r->seg_rows; v.nsd = r->nsd; v.nseg = r->nseg; v.status = r->status; v.lam = r->lam;
    v.pose = r->pose; v.first_seg = r->first_seg; v.w0 = r->w0; v.e0 = r->e0; v.plen = r->plen; v.popl = r->popl; v.n_beams = r->n_beams;
    return v;
}

static int32_t pd_run(bmo_sys* sys, bmo_result* r, int32_t pd_object, int32_t pose0, int32_t n_fields, double* fields, uint32_t flags,
                      bool per_pose) {
    NvtxRange nvtx_("bmo_pd_accumulate");
    if (!sys || !r || !fields) return fail(BMO_EINVAL, "bmo_pd_accumulate: NULL argument");
    if (r->mode != 2) return fail(BMO_EINVAL, "bmo_pd_accumulate: result does not hold Gaussian beamlets (Photodetector.jl:57-60)");
    if (pd_object < 0 || pd_object >= (int)sys->objects.size() || sys->objects[pd_object].kind != BMO_OBJ_PHOTODETECTOR)
        return fail(BMO_EINVAL, "bmo_pd_accumulate: object is not a Photodetector");
    if (pose0 < 0 || pose0 + n_fields > sys->view.n_poses) return fail(BMO_EINVAL, "bmo_pd_accumulate: pose out of range");
    bmo_ctx* ctx = sys->ctx;
    BMO_CUDA(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    const bmo_object& ob = sys->objects[pd_object];
    const int n = ob.pd_n;
    const size_t fbytes = (size_t)n_fields * n * n * 2 * sizeof(double);
    const bool on_dev = flags & BMO_INPUT_DEVICE;
    BMO_CUDA(cudaEventRecord(ctx->ev0, st));
    double* d_field = fields;
    DevBuf<double> field_copy;   // of a host field
    if (!on_dev) {
        BMO_CUDA(field_copy.alloc((size_t)n_fields * n * n * 2, st));
        d_field = field_copy.get();
        BMO_CUDA(cudaMemcpyAsync(d_field, fields, fbytes, cudaMemcpyHostToDevice, st));
    }
    DevBuf<int32_t> d_flags;
    DevBuf<long long> d_offs, d_pose_off;
    DevBuf<PdRec> d_recs;
    DevBuf<PdFast> d_fast;
    const bool ref_order = flags & BMO_PD_REFERENCE_ORDER;
    const int64_t nb = r->n_beams;
    BMO_CUDA(d_flags.alloc((size_t)nb, st));
    BMO_CUDA(d_offs.alloc((size_t)nb, st));
    ResView rv = res_view(r);
    // only the records of poses [pose0, pose0 + n_fields) are built
    pd_flag<<<(unsigned)((nb + 255) / 256), 256, 0, st>>>(rv, sys->view, pd_object, pose0, pose0 + n_fields, d_flags.get());
    BMO_LAUNCH(ctx, "pd_flag");
    scan_flags<<<1, 1024, 0, st>>>(d_flags.get(), nb, d_offs.get(), ctx->d_totals);
    BMO_LAUNCH(ctx, "scan_flags");
    // per pose: the record count of every pose (cnt, closed by a zero so that its exclusive scan ends with m) and, next to m,
    // whether the records need sorting -- read back with m
    DevBuf<unsigned long long> cnt;
    if (per_pose) {
        BMO_CUDA(cnt.alloc((size_t)n_fields + 1, st));
        BMO_CUDA(cudaMemsetAsync(cnt.get(), 0, ((size_t)n_fields + 1) * sizeof(unsigned long long), st));
        BMO_CUDA(cudaMemsetAsync(ctx->d_totals + 1, 0, sizeof(long long), st));
        const int64_t runs = (nb + POSE_RUN - 1) / POSE_RUN;
        pd_pose_count<<<(unsigned)((runs + 255) / 256), 256, 0, st>>>(r->pose, d_flags.get(), nb, pose0, cnt.get(), ctx->d_totals + 1);
        BMO_LAUNCH(ctx, "pd_pose_count");
    }
    BMO_CUDA(cudaMemcpyAsync(ctx->h_totals, ctx->d_totals, (per_pose ? 2 : 1) * sizeof(long long), cudaMemcpyDeviceToHost, st));
    BMO_CUDA(cudaStreamSynchronize(st));
    const int64_t m = ctx->h_totals[0];
    const bool unsorted = per_pose && ctx->h_totals[1] != 0;
    if (m > 0) {
        BMO_CUDA(d_recs.alloc((size_t)m, st));
        pd_build<<<(unsigned)((nb + 255) / 256), 256, 0, st>>>(rv, sys->view, d_flags.get(), d_offs.get(), d_recs.get());
        BMO_LAUNCH(ctx, "pd_build");
        if (per_pose) {
            // group the records by pose, stably (the order std::stable_sort by pose gives), on the device; one pose needs no sort
            if (unsorted && n_fields > 1) {
                if (m > INT32_MAX) return fail(BMO_EINVAL, "bmo_pd_accumulate_poses: more records than a 32-bit index can number");
                DevBuf<int32_t> keys, idx, keys_out, order;
                DevBuf<PdRec> sorted;
                DevBuf<char> tmp;
                size_t tmp_bytes = 0;
                const int end_bit = 32 - __builtin_clz((unsigned)(n_fields - 1));
                BMO_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, tmp_bytes, keys.get(), keys_out.get(), idx.get(), order.get(), (int)m, 0, end_bit, st));
                BMO_CUDA(keys.alloc((size_t)m, st));
                BMO_CUDA(idx.alloc((size_t)m, st));
                BMO_CUDA(keys_out.alloc((size_t)m, st));
                BMO_CUDA(order.alloc((size_t)m, st));
                BMO_CUDA(tmp.alloc(tmp_bytes, st));
                pd_pose_keys<<<(unsigned)((nb + 255) / 256), 256, 0, st>>>(r->pose, d_flags.get(), d_offs.get(), nb, pose0, keys.get(), idx.get());
                BMO_LAUNCH(ctx, "pd_pose_keys");
                BMO_CUDA(cub::DeviceRadixSort::SortPairs(tmp.get(), tmp_bytes, keys.get(), keys_out.get(), idx.get(), order.get(), (int)m, 0, end_bit, st));
                BMO_LAUNCH(ctx, "radix sort by pose");
                BMO_CUDA(sorted.alloc((size_t)m, st));
                pd_gather<<<(unsigned)((m + 255) / 256), 256, 0, st>>>(d_recs.get(), order.get(), sorted.get(), m);
                BMO_LAUNCH(ctx, "pd_gather");
                d_recs = std::move(sorted);
            }
            size_t scan_bytes = 0;
            BMO_CUDA(d_pose_off.alloc((size_t)n_fields + 1, st));
            long long* cnt_in = reinterpret_cast<long long*>(cnt.get());
            BMO_CUDA(cub::DeviceScan::ExclusiveSum(nullptr, scan_bytes, cnt_in, d_pose_off.get(), n_fields + 1, st));
            DevBuf<char> scan_tmp;
            BMO_CUDA(scan_tmp.alloc(scan_bytes, st));
            BMO_CUDA(cub::DeviceScan::ExclusiveSum(scan_tmp.get(), scan_bytes, cnt_in, d_pose_off.get(), n_fields + 1, st));
            BMO_LAUNCH(ctx, "pose offsets");
        }
        if (!ref_order) {
            BMO_CUDA(d_fast.alloc((size_t)m, st));
            pd_make_fast<<<(unsigned)((m + 127) / 128), 128, 0, st>>>(d_recs.get(), d_fast.get(), m);
            BMO_LAUNCH(ctx, "pd_make_fast");
        }
        PdParams pp{};
        pp.recs = d_recs.get(); pp.fast = d_fast.get(); pp.n_recs = m; pp.R = rv; pp.field = d_field; pp.det_pose = sys->view.det_pose;
        pp.pose_off = d_pose_off.get();
        pp.n = n; pp.pd_object = pd_object; pp.n_objects = sys->view.n_objects; pp.pose0 = pose0; pp.lo = ob.pd_lo; pp.hi = ob.pd_hi;
        BMO_CUDA(cudaEventRecord(ctx->evk0, st));
        if (ref_order) {
            dim3 grid((n + PD_TILE - 1) / PD_TILE, (n + PD_TILE - 1) / PD_TILE, n_fields), block(PD_TILE, PD_TILE);
            pd_field<<<grid, block, 0, st>>>(pp);
        } else {
            dim3 grid((n + PDF_TX - 1) / PDF_TX, (n + PDF_TY * PDF_PX - 1) / (PDF_TY * PDF_PX), n_fields), block(PDF_TX, PDF_TY);
            pd_field_fast<<<grid, block, 0, st>>>(pp);
        }
        BMO_LAUNCH(ctx, "pd_field");
        BMO_CUDA(cudaEventRecord(ctx->evk1, st));
        ctx->px_beamlets += m * (int64_t)n * n;
    }
    if (!on_dev) {
        BMO_CUDA(cudaMemcpyAsync(fields, d_field, fbytes, cudaMemcpyDeviceToHost, st));
    }
    BMO_CUDA(cudaEventRecord(ctx->ev1, st));
    BMO_CUDA(cudaStreamSynchronize(st));
    float ms = 0;
    BMO_CUDA(cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1));
    ctx->pd_ms = ms;
    if (m > 0) { float kms = 0; BMO_CUDA(cudaEventElapsedTime(&kms, ctx->evk0, ctx->evk1)); ctx->k4_ms += kms; }
    return BMO_OK;
}

int32_t bmo_pd_accumulate(bmo_sys* sys, bmo_result* r, int32_t pd_object, int32_t pose, double* field, uint32_t flags) {
    return pd_run(sys, r, pd_object, pose, 1, field, flags, false);
}
int32_t bmo_pd_accumulate_poses(bmo_sys* sys, bmo_result* r, int32_t pd_object, int32_t n_poses, double* fields, uint32_t flags) {
    return pd_run(sys, r, pd_object, 0, n_poses, fields, flags, true);
}
// Pose sweep in one call (the loop "move -> empty!(pd) -> solve_system! -> optical_power(pd)" of test/runtests.jl:2092-2120,
// batched): the per-pose fields start from zero on the device, the power integrals are taken there, and only what the
// caller asks for comes back -- n_poses doubles instead of n_poses * n^2 complex numbers when `fields` is NULL.
int32_t bmo_pd_sweep(bmo_sys* sys, bmo_result* r, int32_t pd_object, int32_t n_poses, double* fields, double* power, uint32_t flags) {
    if (!sys || !r) return fail(BMO_EINVAL, "bmo_pd_sweep: NULL argument");
    if (!fields && !power) return fail(BMO_EINVAL, "bmo_pd_sweep: neither fields nor power requested");
    if (pd_object < 0 || pd_object >= (int)sys->objects.size() || sys->objects[pd_object].kind != BMO_OBJ_PHOTODETECTOR)
        return fail(BMO_EINVAL, "bmo_pd_sweep: object is not a Photodetector");
    if (n_poses < 1 || n_poses > sys->view.n_poses) return fail(BMO_EINVAL, "bmo_pd_sweep: n_poses out of range");
    bmo_ctx* ctx = sys->ctx;
    BMO_CUDA(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    const int n = sys->objects[pd_object].pd_n;
    const size_t cnt = (size_t)n_poses * n * n * 2;
    DevBuf<double> d_field, d_p;
    BMO_CUDA(d_field.alloc(cnt, st));
    if (power) BMO_CUDA(d_p.alloc((size_t)n_poses, st));
    const int32_t rc = pd_sweep_device(sys, r, pd_object, n_poses, d_field.get(), d_p.get(), flags);
    if (rc) return rc;
    if (power) BMO_CUDA(cudaMemcpyAsync(power, d_p.get(), (size_t)n_poses * sizeof(double), cudaMemcpyDeviceToHost, st));
    if (fields) BMO_CUDA(cudaMemcpyAsync(fields, d_field.get(), cnt * sizeof(double), cudaMemcpyDeviceToHost, st));
    BMO_CUDA(cudaStreamSynchronize(st));
    return BMO_OK;
}
int32_t bmo::pd_sweep_device(bmo_sys* sys, bmo_result* r, int32_t pd_object, int32_t n_poses, double* d_field, double* d_power, uint32_t flags) {
    bmo_ctx* ctx = sys->ctx;
    const bmo_object& ob = sys->objects[pd_object];
    const int n = ob.pd_n;
    BMO_CUDA(cudaMemsetAsync(d_field, 0, (size_t)n_poses * n * n * 2 * sizeof(double), ctx->stream));
    int32_t rc = pd_run(sys, r, pd_object, 0, n_poses, d_field, (flags | BMO_INPUT_DEVICE), true);
    if (!rc && d_power) rc = pd_power_launch(ctx, d_field, n_poses, n, ob.pd_lo, ob.pd_hi, d_power, ctx->stream);
    return rc;
}
int32_t bmo_pd_power(bmo_sys* sys, int32_t pd_object, int32_t n_fields, const double* fields, double* power, uint32_t flags) {
    if (!sys || !fields || !power) return fail(BMO_EINVAL, "bmo_pd_power: NULL argument");
    if (pd_object < 0 || pd_object >= (int)sys->objects.size() || sys->objects[pd_object].kind != BMO_OBJ_PHOTODETECTOR)
        return fail(BMO_EINVAL, "bmo_pd_power: object is not a Photodetector");
    bmo_ctx* ctx = sys->ctx;
    BMO_CUDA(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    const bmo_object& ob = sys->objects[pd_object];
    const int n = ob.pd_n;
    const bool on_dev = flags & BMO_INPUT_DEVICE;
    const double* d_f = fields;
    double* d_p = power;
    DevBuf<double> f_copy, p_copy;   // of host fields and power
    if (!on_dev) {
        BMO_CUDA(f_copy.alloc((size_t)n_fields * n * n * 2, st));
        BMO_CUDA(cudaMemcpyAsync(f_copy.get(), fields, (size_t)n_fields * n * n * 2 * sizeof(double), cudaMemcpyHostToDevice, st));
        d_f = f_copy.get();
        BMO_CUDA(p_copy.alloc((size_t)n_fields, st));
        d_p = p_copy.get();
    }
    { int32_t rc = pd_power_launch(ctx, d_f, n_fields, n, ob.pd_lo, ob.pd_hi, d_p, st); if (rc) return rc; }
    if (!on_dev) {
        BMO_CUDA(cudaMemcpyAsync(power, d_p, (size_t)n_fields * sizeof(double), cudaMemcpyDeviceToHost, st));
        BMO_CUDA(cudaStreamSynchronize(st));
    }
    return BMO_OK;
}
