// bmo_comm.cu -- the exchange steps of the path behind the C ABI.
//   * The Photodetector field of a beamlet bundle that was sharded over several GPUs is the sum of the ranks' partial
//     fields (the reference adds the beamlet fields serially, `pd.field[i, j] += ...`, Photodetector.jl:103; its
//     `for beam in beams(bg)` loop, System.jl:463-468, is what gets sharded).  One complex128 all-reduce (2 n^2 doubles)
//     over NVLink / NVSwitch through NCCL.
//   * The spot diagram of a ray bundle sharded over several GPUs (bmo_spot_stats_sharded): every rank reduces its own
//     Spotdetector entries to per-block partials (bmo_source.cu), the partials are all-gathered and combined in global block
//     order on every rank, and the histograms are summed by one int64 all-reduce.  No spot leaves its GPU.
//   * The PSFDetector map of a ray bundle sharded over several GPUs (bmo_psf_allgather, bmo_psf_intensity_sharded): the hit
//     records are all-gathered in rank order, every rank sums all records into its band of pixel columns, and the bands are
//     all-gathered.  Each pixel is summed on one GPU over the records of one trace in order, so the map has one GPU's bits.
//   * The Photodetector pose sweep sharded over GPUs by pose range (bmo_pd_sweep_sharded): every rank sweeps its contiguous
//     poses with bmo_pd_sweep's code, the fields stay where they are, and the powers are all-gathered into pose order.
//   * The spot-diagram pose sweep sharded over GPUs by pose range (bmo_spot_stats_poses_sharded): every rank reduces its
//     contiguous poses with bmo_spot_stats_poses' code, and the statistics and histograms are all-gathered into pose order.
//     Each pose is reduced from its own entries alone, so no sum crosses a rank.
//
// NCCL is bound at run time (dlopen of libnccl.so.2) so that libbmo.so has no link-time dependency on it: a host
// that never shards never needs the library, and inside a process that already carries one (PyTorch's bundled
// NCCL) the same copy is used.  BMO_NCCL_LIB overrides the library path.
//
// Two ways to build the communicator, matching the two host models:
//   * one process per GPU (torchrun, MPI, Julia Distributed): rank 0 calls bmo_comm_unique_id, the 128 bytes travel by
//     whatever transport the host has, every rank calls bmo_comm_init;
//   * one process driving n GPUs (a single Julia session, SURVEY 8(b) `bmo_init(n_gpus)`): bmo_comm_init_local over the
//     contexts of the n devices, bmo_pd_allreduce_local = the grouped all-reduce.
#include <dlfcn.h>
#include <mutex>
#include "bmo_host.cuh"

using namespace bmo;

namespace {
// the slice of nccl.h this file uses (stable since NCCL 2.0; checked against 2.27.3 / 2.28.9)
struct NcclUniqueId { char internal[128]; };
typedef void* NcclComm;
typedef int (*fn_GetUniqueId)(NcclUniqueId*);
typedef int (*fn_CommInitRank)(NcclComm*, int, NcclUniqueId, int);
typedef int (*fn_CommInitAll)(NcclComm*, int, const int*);
typedef int (*fn_CommDestroy)(NcclComm);
typedef int (*fn_AllReduce)(const void*, void*, size_t, int /*dtype*/, int /*op*/, NcclComm, cudaStream_t);
typedef int (*fn_AllGather)(const void*, void*, size_t, int /*dtype*/, NcclComm, cudaStream_t);
typedef int (*fn_Group)(void);
typedef const char* (*fn_ErrStr)(int);
typedef int (*fn_GetVersion)(int*);
constexpr int kNcclInt8 = 0, kNcclInt64 = 4, kNcclDouble = 8, kNcclSum = 0;

struct Nccl {
    void* so = nullptr;
    fn_GetUniqueId GetUniqueId = nullptr;
    fn_CommInitRank CommInitRank = nullptr;
    fn_CommInitAll CommInitAll = nullptr;
    fn_CommDestroy CommDestroy = nullptr;
    fn_AllReduce AllReduce = nullptr;
    fn_AllGather AllGather = nullptr;
    fn_Group GroupStart = nullptr, GroupEnd = nullptr;
    fn_ErrStr GetErrorString = nullptr;
    fn_GetVersion GetVersion = nullptr;
    std::string why;   // load error
};
Nccl g_nccl;
std::once_flag g_nccl_once;

void load_nccl() {
    const char* env = getenv("BMO_NCCL_LIB");
    const char* names[] = {env, "libnccl.so.2", "libnccl.so"};
    for (const char* nm : names) {
        if (!nm || !*nm) continue;
        g_nccl.so = dlopen(nm, RTLD_NOW | RTLD_GLOBAL);
        if (g_nccl.so) break;
        g_nccl.why = dlerror();
    }
    if (!g_nccl.so) return;
#define SYM(field, name) g_nccl.field = (decltype(g_nccl.field))dlsym(g_nccl.so, name); if (!g_nccl.field) { g_nccl.why = std::string("symbol missing: ") + name; g_nccl.so = nullptr; return; }
    SYM(GetUniqueId, "ncclGetUniqueId") SYM(CommInitRank, "ncclCommInitRank") SYM(CommInitAll, "ncclCommInitAll")
    SYM(CommDestroy, "ncclCommDestroy") SYM(AllReduce, "ncclAllReduce") SYM(AllGather, "ncclAllGather") SYM(GroupStart, "ncclGroupStart") SYM(GroupEnd, "ncclGroupEnd")
    SYM(GetErrorString, "ncclGetErrorString") SYM(GetVersion, "ncclGetVersion")
#undef SYM
}
int32_t need_nccl() {
    std::call_once(g_nccl_once, load_nccl);
    if (!g_nccl.so) return fail(BMO_ENCCL, "NCCL is not available (dlopen libnccl.so.2: " + g_nccl.why + "); set BMO_NCCL_LIB");
    return BMO_OK;
}
#define BMO_NCCL(call)                                                                                          \
    do {                                                                                                        \
        int r_ = (call);                                                                                        \
        if (r_ != 0) return fail(BMO_ENCCL, std::string(#call) + ": " + g_nccl.GetErrorString(r_));             \
    } while (0)
}  // namespace

struct bmo_comm {
    bmo_ctx* ctx = nullptr;
    NcclComm comm = nullptr;
    int32_t rank = 0, n_ranks = 1;
    double* stage = nullptr;     // device staging buffer for host fields
    size_t stage_cap = 0;        // doubles
};

int32_t bmo_comm_unique_id(uint8_t* id) {
    if (!id) return fail(BMO_EINVAL, "bmo_comm_unique_id: NULL");
    int32_t rc = need_nccl();
    if (rc) return rc;
    NcclUniqueId u;
    BMO_NCCL(g_nccl.GetUniqueId(&u));
    std::memcpy(id, u.internal, BMO_COMM_ID_BYTES);
    return BMO_OK;
}

int32_t bmo_comm_init(bmo_ctx* ctx, int32_t n_ranks, int32_t rank, const uint8_t* id, bmo_comm** out) {
    if (!ctx || !id || !out) return fail(BMO_EINVAL, "bmo_comm_init: NULL argument");
    if (n_ranks < 1 || rank < 0 || rank >= n_ranks) return fail(BMO_EINVAL, "bmo_comm_init: rank outside [0, n_ranks)");
    int32_t rc = need_nccl();
    if (rc) return rc;
    BMO_CUDA(cudaSetDevice(ctx->device));
    NcclUniqueId u;
    std::memcpy(u.internal, id, BMO_COMM_ID_BYTES);
    std::unique_ptr<bmo_comm, FreeWith<bmo_comm_free>> c(new bmo_comm());
    c->ctx = ctx; c->rank = rank; c->n_ranks = n_ranks;
    int r = g_nccl.CommInitRank(&c->comm, n_ranks, u, rank);
    if (r != 0) return fail(BMO_ENCCL, std::string("ncclCommInitRank: ") + g_nccl.GetErrorString(r));
    *out = c.release();
    return BMO_OK;
}

int32_t bmo_comm_init_local(int32_t n, bmo_ctx* const* ctxs, bmo_comm** comms) {
    if (n < 1 || !ctxs || !comms) return fail(BMO_EINVAL, "bmo_comm_init_local: bad arguments");
    int32_t rc = need_nccl();
    if (rc) return rc;
    std::vector<int> devs((size_t)n);
    for (int k = 0; k < n; k++) {
        if (!ctxs[k]) return fail(BMO_EINVAL, "bmo_comm_init_local: NULL context");
        devs[k] = ctxs[k]->device;
        for (int j = 0; j < k; j++) if (devs[j] == devs[k]) return fail(BMO_EINVAL, "bmo_comm_init_local: two contexts share a device");
    }
    std::vector<NcclComm> cs((size_t)n, nullptr);
    BMO_NCCL(g_nccl.CommInitAll(cs.data(), n, devs.data()));
    for (int k = 0; k < n; k++) {
        bmo_comm* c = new bmo_comm();
        c->ctx = ctxs[k]; c->comm = cs[k]; c->rank = k; c->n_ranks = n;
        comms[k] = c;
    }
    return BMO_OK;
}

int32_t bmo_comm_info(bmo_comm* c, int32_t* rank, int32_t* n_ranks, int32_t* nccl_version) {
    if (!c) return fail(BMO_EINVAL, "bmo_comm_info: NULL");
    if (rank) *rank = c->rank;
    if (n_ranks) *n_ranks = c->n_ranks;
    if (nccl_version) { int v = 0; g_nccl.GetVersion(&v); *nccl_version = v; }
    return BMO_OK;
}

// device pointer of the field on this rank: the caller's (BMO_INPUT_DEVICE) or the staging copy of a host field
static int32_t stage_field(bmo_comm* c, double* field, size_t n_dbl, bool on_dev, double** dptr) {
    if (on_dev) { *dptr = field; return BMO_OK; }
    cudaStream_t st = c->ctx->stream;
    if (c->stage_cap < n_dbl) {
        if (c->stage) cudaFree(c->stage);
        c->stage = nullptr; c->stage_cap = 0;
        BMO_CUDA(cudaMalloc((void**)&c->stage, n_dbl * sizeof(double)));
        c->stage_cap = n_dbl;
    }
    BMO_CUDA(cudaMemcpyAsync(c->stage, field, n_dbl * sizeof(double), cudaMemcpyHostToDevice, st));
    *dptr = c->stage;
    return BMO_OK;
}

int32_t bmo_pd_allreduce(bmo_comm* c, double* field, int64_t n_complex, uint32_t flags) {
    if (!c || !field || n_complex <= 0) return fail(BMO_EINVAL, "bmo_pd_allreduce: bad arguments");
    BMO_CUDA(cudaSetDevice(c->ctx->device));
    cudaStream_t st = c->ctx->stream;
    const bool on_dev = flags & BMO_INPUT_DEVICE;
    const size_t n_dbl = (size_t)2 * (size_t)n_complex;
    double* d = nullptr;
    int32_t rc = stage_field(c, field, n_dbl, on_dev, &d);
    if (rc) return rc;
    if (c->n_ranks > 1) BMO_NCCL(g_nccl.AllReduce(d, d, n_dbl, kNcclDouble, kNcclSum, c->comm, st));
    if (!on_dev) BMO_CUDA(cudaMemcpyAsync(field, d, n_dbl * sizeof(double), cudaMemcpyDeviceToHost, st));
    if (!on_dev || (flags & BMO_COMM_SYNC)) BMO_CUDA(cudaStreamSynchronize(st));
    return BMO_OK;
}

int32_t bmo_pd_allreduce_local(int32_t n, bmo_comm* const* comms, double* const* fields, int64_t n_complex, uint32_t flags) {
    if (n < 1 || !comms || !fields || n_complex <= 0) return fail(BMO_EINVAL, "bmo_pd_allreduce_local: bad arguments");
    const bool on_dev = flags & BMO_INPUT_DEVICE;
    const size_t n_dbl = (size_t)2 * (size_t)n_complex;
    std::vector<double*> d((size_t)n, nullptr);
    int32_t rc;
    for (int k = 0; k < n; k++) {
        if (!comms[k] || !fields[k]) return fail(BMO_EINVAL, "bmo_pd_allreduce_local: NULL entry");
        BMO_CUDA(cudaSetDevice(comms[k]->ctx->device));
        if ((rc = stage_field(comms[k], fields[k], n_dbl, on_dev, &d[k]))) return rc;
    }
    if (n > 1) {
        BMO_NCCL(g_nccl.GroupStart());
        for (int k = 0; k < n; k++) {
            int r = g_nccl.AllReduce(d[k], d[k], n_dbl, kNcclDouble, kNcclSum, comms[k]->comm, comms[k]->ctx->stream);
            if (r != 0) { g_nccl.GroupEnd(); return fail(BMO_ENCCL, std::string("ncclAllReduce: ") + g_nccl.GetErrorString(r)); }
        }
        BMO_NCCL(g_nccl.GroupEnd());
    }
    for (int k = 0; k < n; k++) {
        BMO_CUDA(cudaSetDevice(comms[k]->ctx->device));
        if (!on_dev) BMO_CUDA(cudaMemcpyAsync(fields[k], d[k], n_dbl * sizeof(double), cudaMemcpyDeviceToHost, comms[k]->ctx->stream));
    }
    for (int k = 0; k < n; k++) {
        BMO_CUDA(cudaSetDevice(comms[k]->ctx->device));
        if (!on_dev || (flags & BMO_COMM_SYNC)) BMO_CUDA(cudaStreamSynchronize(comms[k]->ctx->stream));
    }
    return BMO_OK;
}

// the collective steps of bmo_spot_stats_sharded: NCCL on the context's stream; one rank needs no exchange
struct NcclSpotExchange : SpotExchange {
    bmo_comm* c;
    explicit NcclSpotExchange(bmo_comm* comm) : c(comm) {}
    int32_t gather(const void* mine, void* all, size_t bytes) override {
        if (c->n_ranks == 1) { BMO_CUDA(cudaMemcpyAsync(all, mine, bytes, cudaMemcpyDeviceToDevice, c->ctx->stream)); return BMO_OK; }
        BMO_NCCL(g_nccl.AllGather(mine, all, bytes, kNcclInt8, c->comm, c->ctx->stream));
        return BMO_OK;
    }
    int32_t sum(int64_t* v, size_t n) override {
        if (c->n_ranks > 1) BMO_NCCL(g_nccl.AllReduce(v, v, n, kNcclInt64, kNcclSum, c->comm, c->ctx->stream));
        return BMO_OK;
    }
};

// Step 1 of the collectives below: every rank's words, all-gathered into all[k * K + w] (word w of rank k, K = mine.size()).
// Word 0 is the rank's argument verdict: BMO_OK, or the code its own checks returned (g_last_error then holds their message).  The
// first refusal in rank order decides for every rank, so that all ranks take the same branch: that code is returned on every rank,
// with the refusing rank's own message there.  (Only arguments are agreed on: a CUDA or NCCL failure on one rank -- an allocation,
// a launch -- returns on that rank alone and leaves the others in the next collective, as with any NCCL collective.)
static int32_t agree(bmo_comm* c, const std::string& fn, const std::vector<int64_t>& mine, std::vector<int64_t>& all) {
    const std::string why = mine[0] ? g_last_error : std::string();
    const int W = c->n_ranks;
    const size_t K = mine.size();
    all.assign(K * W, 0);
    cudaStream_t st = c->ctx->stream;
    BMO_CUDA(cudaSetDevice(c->ctx->device));
    DevBuf<int64_t> buf;
    BMO_CUDA(buf.alloc(K * (W + 1), st));
    int64_t* d = buf.get();
    BMO_CUDA(cudaMemcpyAsync(d, mine.data(), K * sizeof(int64_t), cudaMemcpyHostToDevice, st));
    const int nr = W == 1 ? cudaMemcpyAsync(d + K, d, K * sizeof(int64_t), cudaMemcpyDeviceToDevice, st) != cudaSuccess
                          : g_nccl.AllGather(d, d + K, K, kNcclInt64, c->comm, st);
    if (nr) return fail(BMO_ENCCL, fn + ": exchanging the arguments: " + (W == 1 ? std::string("copy failed") : std::string(g_nccl.GetErrorString(nr))));
    BMO_CUDA(cudaMemcpyAsync(all.data(), d + K, all.size() * sizeof(int64_t), cudaMemcpyDeviceToHost, st));
    BMO_CUDA(cudaStreamSynchronize(st));
    for (int k = 0; k < W; k++) {
        const int32_t v = (int32_t)all[K * k];
        if (v) {
            if (k == c->rank) { g_last_error = why; return v; }
            return fail(v, fn + ": rank " + std::to_string(k) + " refused its arguments");
        }
    }
    return BMO_OK;
}

int32_t bmo_spot_stats_sharded(bmo_comm* c, bmo_result* r, int32_t det_object, const double* window, int32_t nx, int32_t nz,
                               bmo_spot_info* out, int64_t* counts, uint32_t flags) {
    NvtxRange nvtx_("bmo_spot_stats_sharded");
    const std::string fn = "bmo_spot_stats_sharded";
    if (!c) return fail(BMO_EINVAL, fn + ": communicator NULL");
    // Step 1: every rank's argument verdict, entry count and the arguments that must agree (detector, histogram shape, window)
    int32_t rc = BMO_OK;
    if (!out) rc = fail(BMO_EINVAL, fn + ": NULL argument");
    else if (r && r->ctx != c->ctx) rc = fail(BMO_EINVAL, fn + ": the result belongs to another context than the communicator");
    if (!rc && r) rc = spot_check_result(fn, r, det_object);
    if (!rc) rc = spot_check_args(fn, window, nx, nz, counts);
    const int W = c->n_ranks;
    constexpr int K = 11;   // verdict, entries, then what must agree: det_object, histogram?, nx, nz, window?, window bits [4]
    std::vector<int64_t> mine(K, 0), all;
    mine[0] = rc; mine[1] = r ? r->n_beams * r->R : 0; mine[2] = det_object;
    if (counts) { mine[3] = 1; mine[4] = nx; mine[5] = nz; }
    if (window) { mine[6] = 1; std::memcpy(&mine[7], window, 4 * sizeof(double)); }
    if ((rc = agree(c, fn, mine, all))) return rc;
    std::vector<int64_t> entries((size_t)W);
    int64_t N = 0;
    for (int k = 0; k < W; k++) {
        const int64_t* a = all.data() + (size_t)K * k;
        if (!std::equal(a + 2, a + K, all.data() + 2))
            return fail(BMO_EINVAL, fn + ": rank " + std::to_string(k) + " passes another detector, histogram shape or window than rank 0");
        if (a[1] > INT64_MAX - N) return fail(BMO_EINVAL, fn + ": the ranks' entries overflow int64");
        entries[k] = a[1];
        N += a[1];
    }
    // Step 2: the global blocks must not cross a rank boundary
    const int64_t per = spot_per(N);
    for (int k = 0; k + 1 < W; k++)
        if (entries[k] % per)
            return fail(BMO_EINVAL, fn + ": rank " + std::to_string(k) + " holds " + std::to_string(entries[k]) + " entries, not a multiple of the " +
                                        std::to_string(per) + " entries per block of " + std::to_string(N) + " (cut the shards with parallel.spot_shard_slice)");
    // Steps 3-5: the two passes and the histogram (bmo_source.cu)
    NcclSpotExchange x(c);
    return spot_stats_shard(fn, c->ctx, r, det_object, window, nx, nz, entries, per, x, out, counts, flags);
}

int32_t bmo_psf_allgather(bmo_comm* c, bmo_psf* local, bmo_psf** all_out) {
    NvtxRange nvtx_("bmo_psf_allgather");
    const std::string fn = "bmo_psf_allgather";
    if (!c) return fail(BMO_EINVAL, fn + ": communicator NULL");
    // Step 1: every rank's verdict and record count; the total must fit int64
    int32_t rc = BMO_OK;
    if (!all_out) rc = fail(BMO_EINVAL, fn + ": NULL argument");
    else if (local && local->ctx != c->ctx) rc = fail(BMO_EINVAL, fn + ": the records belong to another context than the communicator");
    std::vector<int64_t> mine{rc, local ? local->n : 0}, all;
    if ((rc = agree(c, fn, mine, all))) return rc;
    const int W = c->n_ranks;
    int64_t total = 0, most = 0;
    std::vector<int64_t> first((size_t)W);
    for (int k = 0; k < W; k++) {
        const int64_t m = all[2 * k + 1];
        if (m > INT64_MAX / (PSF_NREC + PSF_NFAST) / W - total) return fail(BMO_EINVAL, fn + ": the ranks' records overflow int64");
        first[k] = total;
        total += m;
        most = std::max(most, m);
    }
    // Step 2: one all-gather of [most][PSF_NREC] records then [most][PSF_NFAST] fast words per rank, each rank's part copied into place
    bmo_ctx* ctx = c->ctx;
    cudaStream_t st = ctx->stream;
    std::unique_ptr<bmo_psf, FreeWith<bmo_psf_free>> p(new bmo_psf());
    p->ctx = ctx;
    if ((rc = psf_reserve(p.get(), total, st))) return rc;
    p->n = total;
    const int64_t m = local ? local->n : 0;
    constexpr size_t D = sizeof(double);
    const size_t per = (size_t)most * (PSF_NREC + PSF_NFAST);   // doubles per rank
    if (total > 0 && W == 1) {     // no exchange: a copy of this rank's records
        BMO_CUDA(cudaMemcpyAsync(p->rec, local->rec, (size_t)m * PSF_NREC * D, cudaMemcpyDeviceToDevice, st));
        BMO_CUDA(cudaMemcpyAsync(p->fast, local->fast, (size_t)m * PSF_NFAST * D, cudaMemcpyDeviceToDevice, st));
        BMO_CUDA(cudaStreamSynchronize(st));
    } else if (total > 0) {
        DevBuf<double> buf;
        BMO_CUDA(buf.alloc(per * (W + 1), st));
        double* send = buf.get() + per * W;
        if (m) {
            BMO_CUDA(cudaMemcpyAsync(send, local->rec, (size_t)m * PSF_NREC * D, cudaMemcpyDeviceToDevice, st));
            BMO_CUDA(cudaMemcpyAsync(send + (size_t)most * PSF_NREC, local->fast, (size_t)m * PSF_NFAST * D, cudaMemcpyDeviceToDevice, st));
        }
        BMO_NCCL(g_nccl.AllGather(send, buf.get(), per, kNcclDouble, c->comm, st));
        for (int k = 0; k < W; k++) {
            const int64_t mk = all[2 * k + 1];
            if (!mk) continue;
            const double* part = buf.get() + per * k;
            BMO_CUDA(cudaMemcpyAsync(p->rec + first[k] * PSF_NREC, part, (size_t)mk * PSF_NREC * D, cudaMemcpyDeviceToDevice, st));
            BMO_CUDA(cudaMemcpyAsync(p->fast + first[k] * PSF_NFAST, part + (size_t)most * PSF_NREC, (size_t)mk * PSF_NFAST * D,
                                     cudaMemcpyDeviceToDevice, st));
        }
        BMO_CUDA(cudaStreamSynchronize(st));
    }
    *all_out = p.release();
    return BMO_OK;
}

int32_t bmo_psf_intensity_sharded(bmo_comm* c, bmo_sys* sys, bmo_psf* all, int32_t psf_object, int32_t pose, int32_t n, const double* lims,
                                  double x0_shift, double z0_shift, double* intensity, uint32_t flags) {
    NvtxRange nvtx_("bmo_psf_intensity_sharded");
    const std::string fn = "bmo_psf_intensity_sharded";
    if (!c) return fail(BMO_EINVAL, fn + ": communicator NULL");
    // Step 1: every rank's verdict and the arguments that must agree: n, pose, psf_object, the bits of lims and the shifts, and the
    // record count (a rank that passes its own rather than the gathered records holds another count)
    int32_t rc = psf_intensity_check(fn.c_str(), sys, all, psf_object, pose, n, lims, intensity);
    if (!rc && sys->ctx != c->ctx) rc = fail(BMO_EINVAL, fn + ": the system belongs to another context than the communicator");
    if (!rc && all->ctx != c->ctx) rc = fail(BMO_EINVAL, fn + ": the records belong to another context than the communicator");
    constexpr int K = 11;   // verdict, n, pose, psf_object, lims bits [4], x0_shift bits, z0_shift bits, records
    std::vector<int64_t> mine(K, 0), agreed;
    mine[0] = rc; mine[1] = n; mine[2] = pose; mine[3] = psf_object;
    if (lims) std::memcpy(&mine[4], lims, 4 * sizeof(double));
    std::memcpy(&mine[8], &x0_shift, sizeof(double)); std::memcpy(&mine[9], &z0_shift, sizeof(double));
    mine[10] = all ? all->n : 0;
    if ((rc = agree(c, fn, mine, agreed))) return rc;
    const int W = c->n_ranks;
    for (int k = 1; k < W; k++)
        if (!std::equal(agreed.begin() + (size_t)K * k + 1, agreed.begin() + (size_t)K * (k + 1), agreed.begin() + 1))
            return fail(BMO_EINVAL, fn + ": rank " + std::to_string(k) + " passes another n, pose, detector, window, shift or record count than rank 0");
    // Step 2: K6 on this rank's band of B = ceil(n / W) columns, then the bands all-gathered.  The map is column-major, so rank r's band
    // of n * B doubles lands at n * (r * B): the first n * n doubles of the gathered bands are the map.
    bmo_ctx* ctx = c->ctx;
    BMO_CUDA(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    const int64_t B = ((int64_t)n + W - 1) / W;
    const int32_t j0 = (int32_t)std::min<int64_t>(n, c->rank * B), j1 = (int32_t)std::min<int64_t>(n, (c->rank + 1) * B);
    const size_t nn = (size_t)n * n, band = (size_t)n * B;
    const bool on_dev = flags & BMO_INPUT_DEVICE;
    double* d_map = intensity;      // the caller's device buffer when the bands exactly fill it
    DevBuf<double> map_copy;
    if (!on_dev || band * W != nn) {
        BMO_CUDA(map_copy.alloc(band * W, st));
        d_map = map_copy.get();
    }
    if ((rc = psf_intensity_band(sys, all, psf_object, pose, n, lims, x0_shift, z0_shift, j0, j1, d_map + band * c->rank))) return rc;
    if (W > 1) BMO_NCCL(g_nccl.AllGather(d_map + band * c->rank, d_map, band, kNcclDouble, c->comm, st));
    if (d_map != intensity)
        BMO_CUDA(cudaMemcpyAsync(intensity, d_map, nn * sizeof(double), on_dev ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost, st));
    BMO_CUDA(cudaStreamSynchronize(st));
    if (j1 > j0) {
        float kms = 0;
        BMO_CUDA(cudaEventElapsedTime(&kms, ctx->evk0, ctx->evk1));
        ctx->psf_ms = kms;
    }
    return BMO_OK;
}

// The pose ranges of a sweep sharded by pose range (bmo_pd_sweep_sharded, bmo_spot_stats_poses_sharded).  Step 1 agrees on K words
// per rank: the verdict, the words that must equal rank 0's, then the rank's first pose and pose count.  Every rank's items of one
// pose -- a power, a bmo_spot_info, a histogram -- have the same size, so step 3 is one all-gather of each rank's items, padded to
// the largest count, and one copy of each rank's part into pose order.
struct PoseShards {
    bmo_comm* c;
    int W;
    std::vector<int64_t> first, count;
    int64_t most = 0;        // the largest count
    explicit PoseShards(bmo_comm* comm) : c(comm), W(comm->n_ranks), first((size_t)W), count((size_t)W) {}

    // Step 1, once `all` is agreed: another `what` than rank 0's, or ranges that do not tile [0, n_poses) in rank order, is refused
    int32_t check(const std::string& fn, const std::vector<int64_t>& all, int64_t n_poses, const char* what) {
        const size_t K = all.size() / W;
        int64_t next = 0;
        for (int k = 0; k < W; k++) {
            const int64_t* a = all.data() + K * k;
            if (!std::equal(a + 1, a + K - 2, all.data() + 1))
                return fail(BMO_EINVAL, fn + ": rank " + std::to_string(k) + " passes another " + what + " than rank 0");
            first[k] = a[K - 2];
            count[k] = a[K - 1];
            if (first[k] != next)
                return fail(BMO_EINVAL, fn + ": rank " + std::to_string(k) + " sweeps from pose " + std::to_string(first[k]) + ", not " +
                                            std::to_string(next) + " (the ranks' poses must tile [0, n_poses) in rank order)");
            next += count[k];
            most = std::max(most, count[k]);
        }
        if (next != n_poses)
            return fail(BMO_EINVAL, fn + ": the ranks sweep " + std::to_string(next) + " of " + std::to_string(n_poses) + " poses");
        return BMO_OK;
    }
    // The device buffer of step 3 holds items() items: [W][most] gathered, then this rank's own `most` from item mine() (one rank:
    // only its own, from item 0).
    size_t items() const { return (size_t)most * (W > 1 ? W + 1 : 1); }
    size_t mine() const { return W > 1 ? (size_t)most * W : 0; }
    // Step 3 on the context's stream, not synchronised: buf's own items (`item` bytes each) of every rank into dst, pose p at item p
    // (dst: host pointer, or device pointer with kind cudaMemcpyDeviceToDevice).  With one rank a copy, no NCCL call.
    int32_t gather(void* buf, size_t item, void* dst, cudaMemcpyKind kind) {
        cudaStream_t st = c->ctx->stream;
        char* b = (char*)buf;
        const size_t part = (size_t)most * item;
        if (W > 1) BMO_NCCL(g_nccl.AllGather(b + mine() * item, b, part, kNcclInt8, c->comm, st));
        for (int k = 0; k < W; k++)
            if (count[k])
                BMO_CUDA(cudaMemcpyAsync((char*)dst + (size_t)first[k] * item, b + (W > 1 ? part * k : 0), (size_t)count[k] * item, kind, st));
        return BMO_OK;
    }
};

int32_t bmo_pd_sweep_sharded(bmo_comm* c, bmo_sys* sys, bmo_result* r, int32_t pd_object, int32_t n_poses, int32_t first, int32_t count,
                             double* fields, double* power, uint32_t flags) {
    NvtxRange nvtx_("bmo_pd_sweep_sharded");
    const std::string fn = "bmo_pd_sweep_sharded";
    if (!c) return fail(BMO_EINVAL, fn + ": communicator NULL");
    // Step 1: every rank's verdict (bmo_pd_sweep's checks on this rank's poses) and the arguments that must agree
    int32_t rc = BMO_OK;
    if (!sys || !power) rc = fail(BMO_EINVAL, fn + ": NULL argument");
    else if (sys->ctx != c->ctx) rc = fail(BMO_EINVAL, fn + ": the system belongs to another context than the communicator");
    else if (n_poses < 1 || first < 0 || count < 0 || count > n_poses - first)
        rc = fail(BMO_EINVAL, fn + ": poses [first, first + count) outside [0, n_poses)");
    else if (count > sys->view.n_poses) rc = fail(BMO_EINVAL, fn + ": the system holds fewer poses than count");
    else if (pd_object < 0 || pd_object >= (int)sys->objects.size() || sys->objects[pd_object].kind != BMO_OBJ_PHOTODETECTOR)
        rc = fail(BMO_EINVAL, fn + ": object is not a Photodetector");
    else if (count > 0 && !r) rc = fail(BMO_EINVAL, fn + ": NULL result on a rank with poses");
    else if (count > 0 && r->ctx != c->ctx) rc = fail(BMO_EINVAL, fn + ": the result belongs to another context than the communicator");
    else if (count > 0 && r->mode != 2) rc = fail(BMO_EINVAL, fn + ": result does not hold Gaussian beamlets (Photodetector.jl:57-60)");
    const int n = rc ? 0 : sys->objects[pd_object].pd_n;
    // verdict, then pd_object, n, n_poses (as rank 0's), first, count (tiling [0, n_poses) in rank order)
    std::vector<int64_t> mine{rc, pd_object, n, n_poses, first, count}, all;
    if ((rc = agree(c, fn, mine, all))) return rc;
    PoseShards ps(c);
    if ((rc = ps.check(fn, all, n_poses, "detector, detector size or pose count"))) return rc;
    // Step 2: this rank's fields and powers, on the device
    bmo_ctx* ctx = c->ctx;
    BMO_CUDA(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    const bool on_dev = flags & BMO_INPUT_DEVICE;
    const size_t fcount = (size_t)count * n * n * 2;
    DevBuf<double> f_buf, p_buf;
    BMO_CUDA(p_buf.alloc(ps.items(), st));
    if (count > 0) {
        double* d_field = fields;     // the caller's device buffer
        if (!on_dev || !fields) {
            BMO_CUDA(f_buf.alloc(fcount, st));
            d_field = f_buf.get();
        }
        if ((rc = pd_sweep_device(sys, r, pd_object, count, d_field, p_buf.get() + ps.mine(), flags))) return rc;
        if (fields && !on_dev) BMO_CUDA(cudaMemcpyAsync(fields, d_field, fcount * sizeof(double), cudaMemcpyDeviceToHost, st));
    }
    // Step 3: the powers of all ranks in pose order
    if ((rc = ps.gather(p_buf.get(), sizeof(double), power, on_dev ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost))) return rc;
    BMO_CUDA(cudaStreamSynchronize(st));
    return BMO_OK;
}

int32_t bmo_spot_stats_poses_sharded(bmo_comm* c, bmo_result* r, int32_t det_object, int32_t n_poses, int32_t first, int32_t count,
                                     const double* window, int32_t nx, int32_t nz, bmo_spot_info* out, int64_t* counts, uint32_t flags) {
    NvtxRange nvtx_("bmo_spot_stats_poses_sharded");
    const std::string fn = "bmo_spot_stats_poses_sharded";
    if (!c) return fail(BMO_EINVAL, fn + ": communicator NULL");
    // Step 1: every rank's verdict (bmo_spot_stats_poses' checks on this rank's poses) and the arguments that must agree
    int32_t rc = BMO_OK;
    if (!out) rc = fail(BMO_EINVAL, fn + ": NULL argument");
    else if (n_poses < 1 || first < 0 || count < 0 || count > n_poses - first)
        rc = fail(BMO_EINVAL, fn + ": poses [first, first + count) outside [0, n_poses)");
    else if (count > 0 && !r) rc = fail(BMO_EINVAL, fn + ": NULL result on a rank with poses");
    else if (count > 0 && r->ctx != c->ctx) rc = fail(BMO_EINVAL, fn + ": the result belongs to another context than the communicator");
    else if (count > 0 && r->n_poses != count)
        rc = fail(BMO_EINVAL, fn + ": count " + std::to_string(count) + " differs from the " + std::to_string(r->n_poses) +
                                  " poses the result was traced with");
    else if (count > 0) rc = spot_check_result(fn, r, det_object);
    if (!rc) rc = spot_check_args(fn, window, nx, nz, counts);
    // verdict, then det_object, n_poses, histogram?, nx, nz, window?, window bits [4] (as rank 0's), first, count (tiling [0, n_poses))
    std::vector<int64_t> mine(13, 0), all;
    mine[0] = rc; mine[1] = det_object; mine[2] = n_poses;
    if (counts) { mine[3] = 1; mine[4] = nx; mine[5] = nz; }
    if (window) { mine[6] = 1; std::memcpy(&mine[7], window, 4 * sizeof(double)); }
    mine[11] = first; mine[12] = count;
    if ((rc = agree(c, fn, mine, all))) return rc;
    PoseShards ps(c);
    if ((rc = ps.check(fn, all, n_poses, "detector, pose count, histogram shape or window"))) return rc;
    // Step 2: this rank's statistics with bmo_spot_stats_poses' code, its histograms into the device buffer of step 3
    bmo_ctx* ctx = c->ctx;
    BMO_CUDA(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    const size_t bins = counts ? (size_t)nx * (size_t)nz : 0;
    DevBuf<bmo_spot_info> i_buf;
    DevBuf<int64_t> h_buf;
    BMO_CUDA(i_buf.alloc(ps.items(), st));
    if (counts) BMO_CUDA(h_buf.alloc(ps.items() * bins, st));
    std::vector<bmo_spot_info> info((size_t)count);
    if (count > 0) {
        if ((rc = spot_stats(fn.c_str(), 1, &r, det_object, count, window, nx, nz, info.data(), counts ? h_buf.get() + ps.mine() * bins : nullptr,
                             BMO_INPUT_DEVICE)))
            return rc;
        BMO_CUDA(cudaMemcpyAsync(i_buf.get() + ps.mine(), info.data(), (size_t)count * sizeof(bmo_spot_info), cudaMemcpyHostToDevice, st));
    }
    // Step 3: the statistics and histograms of all ranks in pose order
    if ((rc = ps.gather(i_buf.get(), sizeof(bmo_spot_info), out, cudaMemcpyDeviceToHost))) return rc;
    if (counts && (rc = ps.gather(h_buf.get(), bins * sizeof(int64_t), counts,
                                  (flags & BMO_INPUT_DEVICE) ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost)))
        return rc;
    BMO_CUDA(cudaStreamSynchronize(st));
    return BMO_OK;
}

int32_t bmo_comm_free(bmo_comm* c) {
    if (!c) return BMO_OK;
    cudaSetDevice(c->ctx->device);
    cudaStreamSynchronize(c->ctx->stream);
    if (c->comm && g_nccl.so) g_nccl.CommDestroy(c->comm);
    if (c->stage) cudaFree(c->stage);
    delete c;
    return BMO_OK;
}
