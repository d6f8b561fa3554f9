// capi.cu — implementation of the C ABI declared in include/tinympc_b200.h.
//
// Host glue only: handle management, problem upload, workspace sizing, kernel-family selection,
// launch + CUDA-event timing, and the host-pointer convenience path (pinned staging, chunked so that
// H2D copies, the solve kernel and D2H copies of consecutive chunks overlap on three streams).
// No CPU fallback exists: every solve goes through a CUDA kernel of this library or returns an error.
#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <thread>
#include <vector>

#include "host_precompute.h"
#include "launch.h"

#define TM_DECL(nx, nu) extern "C" const tmpc::DimEntry *tm_dim_entry_##nx##_##nu();
TM_DIMS(TM_DECL)
#undef TM_DECL

namespace {

// x0[b] <- (A x0[b] + B u[b][:,0]) + f ; one thread per (instance, row); matrices column-major in the blob
template <typename T>
__global__ void advance_kernel(int nx, int nu, int64_t ustride, int64_t B, const T *__restrict__ blob, T *x0, const T *__restrict__ u) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const bool valid = t < B * nx;
    T r = T(0);
    if (valid) {
        const int64_t b = t / nx;
        const int i = (int)(t - b * nx);
        const T *A = blob, *Bm = blob + nx * nx, *f = Bm + nx * nu;
        const T *xb = x0 + b * nx, *ub = u + b * ustride;
        T ax = A[i] * xb[0];
        for (int m = 1; m < nx; ++m) ax = ax + A[i + nx * m] * xb[m];
        T bu = Bm[i] * ub[0];
        for (int j = 1; j < nu; ++j) bu = bu + Bm[i + nx * j] * ub[j];
        r = (ax + bu) + f[i];
    }
    __syncthreads();  // blockDim is a multiple of nx: all rows of an instance have read x0 before any row writes it
    if (valid) x0[t] = r;
}

thread_local std::string g_err;
int fail(int code, const std::string &msg) {
    g_err = msg;
    return code;
}
#define CUDA_TRY(expr)                                                                             \
    do {                                                                                           \
        cudaError_t e_ = (expr);                                                                   \
        if (e_ != cudaSuccess)                                                                     \
            return fail(TINYMPC_ERR_CUDA, std::string(#expr) + ": " + cudaGetErrorString(e_));     \
    } while (0)

const tmpc::DimEntry *find_dim(int nx, int nu) {
#define TM_FIND(a, b) \
    if (nx == a && nu == b) return tm_dim_entry_##a##_##b();
    TM_DIMS(TM_FIND)
#undef TM_FIND
    return nullptr;
}

size_t esize(int dtype) { return dtype == TINYMPC_F64 ? 8 : 4; }

struct DevBuf {
    void *p = nullptr;
    size_t bytes = 0;
    int ensure(size_t n) {
        if (n <= bytes) return 0;
        if (p) cudaFree(p);
        p = nullptr;
        bytes = 0;
        if (cudaMalloc(&p, n) != cudaSuccess) return -1;
        bytes = n;
        return 0;
    }
    void release() {
        if (p) cudaFree(p);
        p = nullptr;
        bytes = 0;
    }
};
struct PinBuf {
    void *p = nullptr;
    size_t bytes = 0;
    int ensure(size_t n) {
        if (n <= bytes) return 0;
        if (p) cudaFreeHost(p);
        p = nullptr;
        bytes = 0;
        if (cudaMallocHost(&p, n) != cudaSuccess) return -1;
        bytes = n;
        return 0;
    }
    void release() {
        if (p) cudaFreeHost(p);
        p = nullptr;
        bytes = 0;
    }
};

std::vector<char> copy_bytes(const void *p, size_t n) {
    std::vector<char> v(n);
    if (n) std::memcpy(v.data(), p, n);
    return v;
}

}  // namespace

struct tinympc_b200_solver {
    int device = 0;
    int sm_count = 0;
    int max_smem_optin = 0;
    int l2_bytes = 0;
    int nx = 0, nu = 0, N = 0, dtype = 0;
    double rho = 0;
    const tmpc::DimEntry *dim = nullptr;
    // host copies (native dtype, column-major)
    std::vector<char> A, Bm, f, Qd, Rd, Kinf, Pinf, Quu, AmBKt, APf, BPf;
    std::vector<char> h_xlo, h_xhi, h_ulo, h_uhi;  // column 0 of the bounds
    bool has_xb = false, has_ub = false;
    int ncx = 0, ncu = 0, nlx = 0, nlu = 0, ntvx = 0, ntvu = 0;
    int cone_x_start[4] = {0, 0, 0, 0}, cone_u_start[4] = {0, 0, 0, 0};
    double cone_x_mu[4] = {0, 0, 0, 0}, cone_u_mu[4] = {0, 0, 0, 0};
    // device copies
    DevBuf d_xmin, d_xmax, d_umin, d_umax, d_blob;
    int bounds_tv = 0;
    int bounds_zero_free = 1;
    DevBuf d_Alin_x, d_blin_x, d_Alin_u, d_blin_u, d_tvA_x, d_tvb_x, d_tvA_u, d_tvb_u;
    tinympc_settings_t settings;
    int mode = TINYMPC_MODE_STRICT;
    int family = TINYMPC_KERNEL_AUTO;
    // launch scratch (one solve at a time per handle: enqueue() serialises launches issued on different streams)
    DevBuf ws;          // TPI / GPS workspace
    DevBuf queue;
    DevBuf vscratch;    // GPI: work->v / work->z staging
    DevBuf shared_ref;  // host path: references shared by the whole batch
    cudaEvent_t ev_last = nullptr;  // recorded after the last enqueue
    cudaStream_t last_stream = nullptr;
    bool have_last = false;
    // host-path staging (per pipeline slot)
    static constexpr int SLOTS = 3;
    DevBuf dio[SLOTS];
    PinBuf pin_in[SLOTS], pin_out[SLOTS];
    cudaStream_t st_h2d = nullptr, st_k = nullptr, st_d2h = nullptr;
    cudaEvent_t ev_in[SLOTS] = {}, ev_k[SLOTS] = {}, ev_out[SLOTS] = {};
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    bool timed = false;
    tinympc_b200_stats_t stats;
};

namespace {

int upload(DevBuf &b, const void *src, size_t n) {
    if (!src || n == 0) return 0;
    if (b.ensure(n)) return -1;
    return cudaMemcpy(b.p, src, n, cudaMemcpyHostToDevice) == cudaSuccess ? 0 : -1;
}

// grow a launch buffer of the handle to n bytes; the previous solve may still be using it, so wait for that one first
int grow(tinympc_b200_solver *s, DevBuf &b, size_t n, const char *what) {
    if (n <= b.bytes) return 0;
    if (s->have_last) CUDA_TRY(cudaEventSynchronize(s->ev_last));
    if (b.ensure(n)) return fail(TINYMPC_ERR_CUDA, std::string(what) + " allocation failed");
    return 0;
}

struct Features {
    int soc_x, soc_u, lin_x, lin_u, tvl_x, tvl_u, ext;
};
Features features(const tinympc_b200_solver *s) {
    Features f;
    const tinympc_settings_t &st = s->settings;
    f.soc_x = st.en_state_soc && s->ncx > 0;
    f.soc_u = st.en_input_soc && s->ncu > 0;
    f.lin_x = st.en_state_linear != 0;
    f.lin_u = st.en_input_linear != 0;
    f.tvl_x = st.en_tv_state_linear != 0;
    f.tvl_u = st.en_tv_input_linear != 0;
    f.ext = f.soc_x || f.soc_u || f.lin_x || f.lin_u || f.tvl_x || f.tvl_u;
    return f;
}

int check_ready(const tinympc_b200_solver *s) {
    const tinympc_settings_t &st = s->settings;
    if ((st.en_state_bound && !s->has_xb) || (st.en_input_bound && !s->has_ub))
        return fail(TINYMPC_ERR_NO_BOUNDS, "en_state_bound/en_input_bound set but bounds were never provided");
    if ((st.en_state_linear && s->nlx > 0 && (!s->d_Alin_x.p || !s->d_blin_x.p)) || (st.en_input_linear && s->nlu > 0 && (!s->d_Alin_u.p || !s->d_blin_u.p)) ||
        (st.en_tv_state_linear && s->ntvx > 0 && (!s->d_tvA_x.p || !s->d_tvb_x.p)) || (st.en_tv_input_linear && s->ntvu > 0 && (!s->d_tvA_u.p || !s->d_tvb_u.p)))
        return fail(TINYMPC_ERR_ARG, "linear constraints enabled but their matrices were not uploaded");
    if (st.check_termination <= 0) return fail(TINYMPC_ERR_ARG, "check_termination must be >= 1");
    return 0;
}

// Which kernel family serves a solve.  GPI = lane groups, state on chip (box constraints, horizon fits in shared + tensor
// memory); GPS = lane groups, state streamed (everything else the lane mapping covers); TPI = one thread per instance.
// `gpi` / `gps`: the plans of the two lane-group families for this solve (family 0 = not available).  Returns -1 when an
// explicit request cannot be honoured.
int resolve_family(const tinympc_b200_solver *s, const Features &ft, const tmpc::LaunchPlan &gpi, const tmpc::LaunchPlan &gps, int64_t B) {
    const bool gpi_ok = gpi.family != 0, gps_ok = gps.family != 0;
    if (s->family == TINYMPC_KERNEL_GPI) return gpi_ok ? TINYMPC_KERNEL_GPI : (gps_ok ? TINYMPC_KERNEL_GPS : -1);
    if (s->family == TINYMPC_KERNEL_GPS) return gps_ok ? TINYMPC_KERNEL_GPS : -1;
    if (s->family == TINYMPC_KERNEL_TPI) return TINYMPC_KERNEL_TPI;
    // AUTO (measured rules; evidence: profiles/r02_auto_rule_sweep.md, profiles/r01_sweep_1gpu.md)
    const bool gps_two = gps.group_instances == 2;  // two instances per lane group: the small shapes
    const bool big_batch = B >= (int64_t)s->sm_count * 384;  // one thread per instance fills the GPU
    // cones / hyperplanes: streamed lane groups (rocket landing, fp64: 3.3x the thread-per-instance kernel)
    if (ft.ext) return gps_ok ? TINYMPC_KERNEL_GPS : TINYMPC_KERNEL_TPI;
    // box constraints, streamed alternative when the state does not stay on chip: for big batches the streamed lane groups
    // beat one thread per instance on the small fp64 shapes ((6,3,100): 28.1 vs 36.7 ms, (4,2,50): 9.1 vs 11.6 ms) and lose
    // on the wide ones ((12,4,50) fp64: 61.6 vs 35.8 ms; fp32 N = 100: 41-113 vs 36-71 ms); small batches cannot fill the
    // GPU with one thread per instance
    const int streamed = !gps_ok ? TINYMPC_KERNEL_TPI
                                 : ((!big_batch || (s->dtype == TINYMPC_F64 && gps_two)) ? TINYMPC_KERNEL_GPS : TINYMPC_KERNEL_TPI);
    if (!gpi_ok) return streamed;
    // fp32: on chip (GPI) unless shared + tensor memory hold fewer than 32 instances per SM (long horizons with wide inputs)
    // AND the batch is large.  Measured on B200 (B = 131 072, N = 100): at 16 instances/SM the streamed kernels win by 10-35 %
    // for every shape except (16,8), where the thread-per-instance register footprint costs more than the low on-chip
    // occupancy; at >= 32 instances/SM GPI always wins.
    const int ipc = gpi.instances_per_cta, gpi_warps = gpi.warps_resident;
    if (s->dtype == TINYMPC_F64) {
        // fp64 (rows re-read per sweep, duals in tensor memory): on chip wins as soon as four warps per SM are resident
        // ((12,4,50): 29.6 vs 35.9 ms TPI at 16 instances/SM; (16,8,50): 57.3 vs 88.4 ms at 8/SM), and loses badly with one
        // warp per SM ((6,3,100): 83 vs 28.4 ms on the streamed lane groups)
        if (gpi_warps > 0 && gpi_warps < 4 && big_batch) return streamed;
        return TINYMPC_KERNEL_GPI;
    }
    const bool tpi_heavy = s->nx >= 16 && s->nu >= 8;
    if (ipc > 0 && ipc < 32 && !tpi_heavy && big_batch) return streamed;
    return TINYMPC_KERNEL_GPI;
}

// the launch descriptor of a solve of `io` on the handle's problem
void base_desc(const tinympc_b200_solver *s, tmpc::LaunchDesc &d, const Features &ft, const tinympc_batch_t &io) {
    std::memset(&d, 0, sizeof(d));
    d.io = io;
    d.Bpad = (io.B + 31) / 32 * 32;
    d.dtype = s->dtype;
    d.fast = s->mode == TINYMPC_MODE_FAST;
    d.ext = ft.ext;
    d.A = s->A.data(); d.Bm = s->Bm.data(); d.f = s->f.data(); d.Qd = s->Qd.data(); d.Rd = s->Rd.data();
    d.Kinf = s->Kinf.data(); d.Pinf = s->Pinf.data(); d.Quu = s->Quu.data(); d.AmBKt = s->AmBKt.data();
    d.APf = s->APf.data(); d.BPf = s->BPf.data();
    d.rho = s->rho;
    const tinympc_settings_t &st = s->settings;
    d.pri_tol = st.abs_pri_tol; d.dua_tol = st.abs_dua_tol;
    d.N = s->N; d.max_iter = st.max_iter; d.check_termination = st.check_termination;
    d.en_state_bound = st.en_state_bound; d.en_input_bound = st.en_input_bound;
    d.soc_x = ft.soc_x; d.soc_u = ft.soc_u;
    d.ncx = st.en_state_soc ? s->ncx : 0; d.ncu = st.en_input_soc ? s->ncu : 0;
    d.lin_x = ft.lin_x; d.lin_u = ft.lin_u; d.nlx = s->nlx; d.nlu = s->nlu;
    d.tvl_x = ft.tvl_x; d.tvl_u = ft.tvl_u; d.ntvx = s->ntvx; d.ntvu = s->ntvu;
    for (int c = 0; c < 4; ++c) {
        d.cone_x_start[c] = s->cone_x_start[c]; d.cone_u_start[c] = s->cone_u_start[c];
        d.cone_x_mu[c] = s->cone_x_mu[c]; d.cone_u_mu[c] = s->cone_u_mu[c];
    }
    d.x_min = s->d_xmin.p; d.x_max = s->d_xmax.p; d.u_min = s->d_umin.p; d.u_max = s->d_umax.p;
    d.Alin_x = s->d_Alin_x.p; d.blin_x = s->d_blin_x.p; d.Alin_u = s->d_Alin_u.p; d.blin_u = s->d_blin_u.p;
    d.tv_Alin_x = s->d_tvA_x.p; d.tv_blin_x = s->d_tvb_x.p; d.tv_Alin_u = s->d_tvA_u.p; d.tv_blin_u = s->d_tvb_u.p;
    d.gmat = s->d_blob.p;
    d.bounds_tv = s->bounds_tv;
    d.bounds_zero_free = s->bounds_zero_free;
    d.h_xlo = s->h_xlo.empty() ? nullptr : s->h_xlo.data(); d.h_xhi = s->h_xhi.empty() ? nullptr : s->h_xhi.data();
    d.h_ulo = s->h_ulo.empty() ? nullptr : s->h_ulo.data(); d.h_uhi = s->h_uhi.empty() ? nullptr : s->h_uhi.data();
    d.sm_count = s->sm_count;
    d.smem_budget = s->max_smem_optin - 64;
}

// enqueue one batched solve on `stream` (device pointers); fills stats
int enqueue(tinympc_b200_solver *s, const tinympc_batch_t *io, cudaStream_t stream, bool timed) {
    if (int rc = check_ready(s)) return rc;
    if (!io->x0 || !io->Xref) return fail(TINYMPC_ERR_ARG, "x0 and Xref are required");
    if (io->B <= 0) return TINYMPC_OK;
    const Features ft = features(s);
    tmpc::LaunchDesc d;
    base_desc(s, d, ft, *io);
    d.stream = stream;
    const tmpc::LaunchPlan gpi = s->dim->plan(d, TINYMPC_KERNEL_GPI), gps = s->dim->plan(d, TINYMPC_KERNEL_GPS);
    int family = resolve_family(s, ft, gpi, gps, io->B);
    if (io->models) {  // per-instance models: on-chip kernel only
        if (!gpi.family || s->family == TINYMPC_KERNEL_TPI || s->family == TINYMPC_KERNEL_GPS)
            return fail(TINYMPC_ERR_UNSUPPORTED, "per-instance models need the on-chip GPI kernel (box constraints, horizon fitting in shared memory)");
        family = TINYMPC_KERNEL_GPI;
    }
    if (family < 0) return fail(TINYMPC_ERR_UNSUPPORTED, "the requested lane-group kernel does not cover this problem shape");
    const tmpc::LaunchPlan plan = family == TINYMPC_KERNEL_GPI ? gpi : family == TINYMPC_KERNEL_GPS ? gps : s->dim->plan(d, family);
    if (!plan.family) return fail(TINYMPC_ERR_UNSUPPORTED, "no compiled kernel for this (dtype, mode, family) combination");
    // The launch scratch of a handle (work queue, workspaces, timing events) is single-buffered: a solve enqueued on a
    // different stream than the previous one first waits for it.
    if (s->have_last && s->last_stream != stream) CUDA_TRY(cudaStreamWaitEvent(stream, s->ev_last, 0));
    if (int rc = grow(s, s->ws, plan.workspace_bytes, "workspace")) return rc;
    if (int rc = grow(s, s->vscratch, plan.scratch_bytes, "GPI v-scratch")) return rc;
    d.workspace = s->ws.p;
    d.scratch = plan.scratch_bytes ? s->vscratch.p : nullptr;
    if (timed) CUDA_TRY(cudaEventRecord(s->ev0, stream));
    if (family != TINYMPC_KERNEL_TPI) {
        if (s->queue.ensure(256)) return fail(TINYMPC_ERR_CUDA, "queue allocation failed");
        CUDA_TRY(cudaMemsetAsync(s->queue.p, 0, 256, stream));
        d.work_queue = s->queue.p;
    }
    const int rc = s->dim->launch(&d, plan);
    if (rc == TINYMPC_ERR_CUDA) return fail(rc, std::string("kernel launch failed: ") + cudaGetErrorString(cudaGetLastError()));
    if (rc) return fail(rc, "no compiled kernel for this (dtype, mode, family) combination");
    if (timed) CUDA_TRY(cudaEventRecord(s->ev1, stream));
    CUDA_TRY(cudaEventRecord(s->ev_last, stream));
    s->last_stream = stream;
    s->have_last = true;
    s->timed = timed;
    s->stats.instances = io->B;
    s->stats.kernel_launches = 1;
    s->stats.kernel_family = family;
    s->stats.lanes_per_instance = plan.lanes;
    s->stats.instances_per_cta = plan.instances_per_cta;
    s->stats.smem_bytes_per_cta = (int)plan.smem;
    s->stats.threads_per_cta = plan.threads;
    s->stats.tmem_cols_per_cta = plan.tmem_cols;
    s->stats.ctas = plan.ctas;
    s->stats.gpi_instances = family == TINYMPC_KERNEL_TPI ? 0 : io->B;
    s->stats.workspace_bytes = (int64_t)plan.workspace_bytes;
    return TINYMPC_OK;
}

}  // namespace

namespace {
template <typename T>
int precompute_batch_T(int nx, int nu, int64_t B, const T *A, const T *Bm, const T *f, const T *Qd, const T *Rd, const T *rho,
                       T *out, int nthreads, int64_t *bad_index = nullptr) {
    const int64_t M = tinympc_b200_model_blob_elems(nx, nu);
    nthreads = (int)std::max<int64_t>(1, std::min<int64_t>(nthreads, B));
    std::vector<int64_t> bad(nthreads, 0);
    auto work = [&](int t) {
        std::vector<T> Qw(nx), Rw(nu);
        for (int64_t b = t; b < B; b += nthreads) {
            const T *Ab = A + b * nx * nx, *Bb = Bm + b * nx * nu, *fb = f + b * nx;
            T *o = out + b * M;
            T *oA = o, *oB = oA + nx * nx, *oF = oB + nx * nu, *oQ = oF + nx, *oR = oQ + nx, *oK = oR + nu, *oP = oK + nu * nx,
              *oQuu = oP + nx * nx, *oAm = oQuu + nu * nu, *oAPf = oAm + nx * nx, *oBPf = oAPf + nx;
            const T r = rho[b];
            for (int i = 0; i < nx; ++i) Qw[i] = Qd[b * nx + i] + r;  // tiny_api.cpp:117
            for (int j = 0; j < nu; ++j) Rw[j] = Rd[b * nu + j] + r;  // tiny_api.cpp:118
            std::copy(Ab, Ab + nx * nx, oA);
            std::copy(Bb, Bb + nx * nu, oB);
            std::copy(fb, fb + nx, oF);
            std::copy(Qw.begin(), Qw.end(), oQ);
            std::copy(Rw.begin(), Rw.end(), oR);
            const int rc = tmpc::precompute_cache<T>(nx, nu, (double)r, Ab, Bb, fb, Qw.data(), Rw.data(), oK, oP, oQuu, oAm, oAPf, oBPf);
            oBPf[nu] = r;
            if (rc < 0 && bad[t] == 0) bad[t] = b + 1;
        }
    };
    std::vector<std::thread> th;
    for (int t = 1; t < nthreads; ++t) th.emplace_back(work, t);
    work(0);
    for (auto &x : th) x.join();
    int64_t first = 0;
    for (int64_t v : bad)
        if (v && (!first || v < first)) first = v;
    if (first) {
        fail(TINYMPC_ERR_SINGULAR, "singular R + B'PB in the Riccati recursion of instance " + std::to_string(first - 1));
        if (bad_index) *bad_index = first - 1;
        return TINYMPC_ERR_SINGULAR;
    }
    if (bad_index) *bad_index = -1;
    return 0;
}
}  // namespace

extern "C" {

const char *tinympc_b200_last_error(void) { return g_err.c_str(); }
const char *tinympc_b200_version(void) { return "tinympc_b200 0.1 (sm_100a)"; }

int tinympc_b200_supported(int32_t dtype, int32_t nx, int32_t nu) {
    return (dtype == TINYMPC_F32 || dtype == TINYMPC_F64) && find_dim(nx, nu) != nullptr;
}

int tinympc_b200_default_settings(tinympc_settings_t *s) {
    if (!s) return fail(TINYMPC_ERR_ARG, "settings is null");
    s->abs_pri_tol = 1e-3;  // tiny_api_constants.hpp:5-16
    s->abs_dua_tol = 1e-3;
    s->max_iter = 1000;
    s->check_termination = 1;
    s->en_state_bound = 1;
    s->en_input_bound = 1;
    s->en_state_soc = 0;
    s->en_input_soc = 0;
    s->en_state_linear = 0;
    s->en_input_linear = 0;
    s->en_tv_state_linear = 0;
    s->en_tv_input_linear = 0;
    return TINYMPC_OK;
}

int tinympc_b200_precompute_cache(int32_t dtype, int32_t nx, int32_t nu, double rho, const void *A, const void *B,
                                  const void *f, const void *Q, const void *R, void *Kinf, void *Pinf, void *Quu_inv,
                                  void *AmBKt, void *APf, void *BPf) {
    if (!A || !B || !f || !Q || !R || !Kinf || !Pinf || !Quu_inv || !AmBKt || !APf || !BPf || nx <= 0 || nu <= 0)
        return fail(TINYMPC_ERR_ARG, "null pointer or bad size");
    int rc;
    if (dtype == TINYMPC_F64)
        rc = tmpc::precompute_cache<double>(nx, nu, rho, (const double *)A, (const double *)B, (const double *)f,
                                            (const double *)Q, (const double *)R, (double *)Kinf, (double *)Pinf,
                                            (double *)Quu_inv, (double *)AmBKt, (double *)APf, (double *)BPf);
    else if (dtype == TINYMPC_F32)
        rc = tmpc::precompute_cache<float>(nx, nu, rho, (const float *)A, (const float *)B, (const float *)f,
                                           (const float *)Q, (const float *)R, (float *)Kinf, (float *)Pinf,
                                           (float *)Quu_inv, (float *)AmBKt, (float *)APf, (float *)BPf);
    else
        return fail(TINYMPC_ERR_ARG, "bad dtype");
    if (rc < 0) return fail(TINYMPC_ERR_ARG, "singular R + B'PB in the Riccati recursion");
    return rc;
}

int64_t tinympc_b200_model_blob_elems(int32_t nx, int32_t nu) {
    return (int64_t)3 * nx * nx + 2 * nx * nu + nu * nu + 3 * nx + 2 * nu + 1;
}

int tinympc_b200_precompute_cache_batch(int32_t dtype, int32_t nx, int32_t nu, int64_t B, const void *A, const void *Bm,
                                        const void *f, const void *Qdiag, const void *Rdiag, const void *rho,
                                        void *models_out, int32_t nthreads) {
    if (!A || !Bm || !f || !Qdiag || !Rdiag || !rho || !models_out || nx <= 0 || nu <= 0 || B < 0)
        return fail(TINYMPC_ERR_ARG, "null pointer or bad size");
    if (dtype == TINYMPC_F64)
        return precompute_batch_T<double>(nx, nu, B, (const double *)A, (const double *)Bm, (const double *)f, (const double *)Qdiag,
                                          (const double *)Rdiag, (const double *)rho, (double *)models_out, nthreads);
    if (dtype == TINYMPC_F32)
        return precompute_batch_T<float>(nx, nu, B, (const float *)A, (const float *)Bm, (const float *)f, (const float *)Qdiag,
                                         (const float *)Rdiag, (const float *)rho, (float *)models_out, nthreads);
    return fail(TINYMPC_ERR_ARG, "bad dtype");
}

int tinympc_b200_precompute_cache_batch_device(tinympc_b200_solver_t *s, int64_t B, const void *A, const void *Bm, const void *f,
                                               const void *Qdiag, const void *Rdiag, const void *rho, void *models_out,
                                               int32_t *sweeps_out, void *stream) {
    if (!s) return fail(TINYMPC_ERR_ARG, "null handle");
    if (!A || !Bm || !f || !Qdiag || !Rdiag || !rho || !models_out || B < 0) return fail(TINYMPC_ERR_ARG, "null pointer or bad size");
    if (B == 0) return TINYMPC_OK;
    CUDA_TRY(cudaSetDevice(s->device));
    const int rc = s->dim->precompute_batch(s->dtype, B, A, Bm, f, Qdiag, Rdiag, rho, models_out, sweeps_out, s->sm_count,
                                            (cudaStream_t)stream);
    if (rc == TINYMPC_ERR_CUDA) return fail(rc, std::string("precompute kernel launch failed: ") + cudaGetErrorString(cudaGetLastError()));
    if (rc) return fail(rc, "precompute kernel unavailable for this dtype");
    return TINYMPC_OK;
}

int tinympc_b200_create(const tinympc_problem_t *p, int32_t device, tinympc_b200_solver_t **out) {
    if (!p || !out) return fail(TINYMPC_ERR_ARG, "null argument");
    *out = nullptr;
    if (p->nx <= 0 || p->nu <= 0 || p->N < 2) return fail(TINYMPC_ERR_ARG, "need nx>0, nu>0, N>=2");
    if (p->dtype != TINYMPC_F32 && p->dtype != TINYMPC_F64) return fail(TINYMPC_ERR_ARG, "bad dtype");
    if (!p->Adyn || !p->Bdyn || !p->fdyn || !p->Q || !p->R || !p->Kinf || !p->Pinf || !p->Quu_inv || !p->AmBKt ||
        !p->APf || !p->BPf)
        return fail(TINYMPC_ERR_ARG, "model / cache pointer is null");
    const tmpc::DimEntry *dim = find_dim(p->nx, p->nu);
    if (!dim) return fail(TINYMPC_ERR_UNSUPPORTED, "no kernel compiled for this (nx, nu); add it to TM_DIMS in csrc/launch.h");
    if (p->num_state_cones > 4 || p->num_input_cones > 4) return fail(TINYMPC_ERR_UNSUPPORTED, "at most 4 cones per side");
    for (int c = 0; c < p->num_state_cones && p->Acx && p->qcx; ++c)
        if (p->qcx[c] != 3 || p->Acx[c] < 0 || p->Acx[c] + 3 > p->nx) return fail(TINYMPC_ERR_CONE_DIM, "state cone must be 3-dimensional and inside the state");
    for (int c = 0; c < p->num_input_cones && p->Acu && p->qcu; ++c)
        if (p->qcu[c] != 3 || p->Acu[c] < 0 || p->Acu[c] + 3 > p->nu) return fail(TINYMPC_ERR_CONE_DIM, "input cone must be 3-dimensional and inside the input");

    if (p->num_state_linear < 0 || p->num_input_linear < 0 || p->num_tv_state_linear < 0 || p->num_tv_input_linear < 0)
        return fail(TINYMPC_ERR_ARG, "negative constraint count");
    if ((p->num_state_linear > 0 && (!p->Alin_x || !p->blin_x)) || (p->num_input_linear > 0 && (!p->Alin_u || !p->blin_u)) ||
        (p->num_tv_state_linear > 0 && (!p->tv_Alin_x || !p->tv_blin_x)) ||
        (p->num_tv_input_linear > 0 && (!p->tv_Alin_u || !p->tv_blin_u)))
        return fail(TINYMPC_ERR_ARG, "hyperplane count > 0 with a NULL normal matrix or offset vector");
    if ((p->num_state_cones > 0 && (!p->Acx || !p->qcx || !p->cx)) || (p->num_input_cones > 0 && (!p->Acu || !p->qcu || !p->cu)))
        return fail(TINYMPC_ERR_ARG, "cone count > 0 with a NULL index / mu vector");

    int ndev = 0;
    CUDA_TRY(cudaGetDeviceCount(&ndev));
    if (device < 0 || device >= ndev) return fail(TINYMPC_ERR_ARG, "bad device index");
    CUDA_TRY(cudaSetDevice(device));
    cudaDeviceProp prop;
    CUDA_TRY(cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10) return fail(TINYMPC_ERR_UNSUPPORTED, "this library is built for sm_100a (B200) only");

    tinympc_b200_solver *s = new tinympc_b200_solver();
    s->device = device;
    s->sm_count = prop.multiProcessorCount;
    s->max_smem_optin = (int)prop.sharedMemPerBlockOptin;
    s->l2_bytes = prop.l2CacheSize;
    s->nx = p->nx; s->nu = p->nu; s->N = p->N; s->dtype = p->dtype; s->rho = p->rho;
    s->dim = dim;
    const size_t es = esize(p->dtype), nx = p->nx, nu = p->nu, N = p->N;
    s->A = copy_bytes(p->Adyn, es * nx * nx); s->Bm = copy_bytes(p->Bdyn, es * nx * nu); s->f = copy_bytes(p->fdyn, es * nx);
    s->Qd = copy_bytes(p->Q, es * nx); s->Rd = copy_bytes(p->R, es * nu);
    s->Kinf = copy_bytes(p->Kinf, es * nu * nx); s->Pinf = copy_bytes(p->Pinf, es * nx * nx);
    s->Quu = copy_bytes(p->Quu_inv, es * nu * nu); s->AmBKt = copy_bytes(p->AmBKt, es * nx * nx);
    s->APf = copy_bytes(p->APf, es * nx); s->BPf = copy_bytes(p->BPf, es * nu);
    tinympc_b200_default_settings(&s->settings);
    bool ok = true;
    {   // packed cache blob for the GPI kernel's TMA staging: A,B,f,Qd,Rd,Kinf,Pinf,Quu,AmBKt,APf,BPf
        std::vector<char> blob;
        for (const std::vector<char> *v : {&s->A, &s->Bm, &s->f, &s->Qd, &s->Rd, &s->Kinf, &s->Pinf, &s->Quu, &s->AmBKt, &s->APf, &s->BPf})
            blob.insert(blob.end(), v->begin(), v->end());
        blob.resize((blob.size() + 63) / 64 * 64, 0);
        ok &= !upload(s->d_blob, blob.data(), blob.size());
    }
    auto varies = [&](const void *m, size_t rows, size_t cols) {  // does a (rows x cols) column-major matrix vary along columns?
        if (!m) return false;
        const char *c = (const char *)m;
        for (size_t k = 1; k < cols; ++k)
            if (std::memcmp(c, c + k * rows * es, rows * es) != 0) return true;
        return false;
    };
    auto has_zero = [&](const void *m, size_t n) {  // any element == +-0 ?
        if (!m) return false;
        for (size_t i = 0; i < n; ++i)
            if ((es == 8 ? ((const double *)m)[i] : (double)((const float *)m)[i]) == 0.0) return true;
        return false;
    };
    s->bounds_zero_free = !(has_zero(p->x_min, (size_t)nx * N) || has_zero(p->x_max, (size_t)nx * N) ||
                            has_zero(p->u_min, (size_t)nu * (N - 1)) || has_zero(p->u_max, (size_t)nu * (N - 1)));
    s->bounds_tv = varies(p->x_min, nx, N) || varies(p->x_max, nx, N) || varies(p->u_min, nu, N - 1) || varies(p->u_max, nu, N - 1);
    if (p->x_min && p->x_max) {
        ok &= !upload(s->d_xmin, p->x_min, es * nx * N) && !upload(s->d_xmax, p->x_max, es * nx * N);
        s->has_xb = true;
        s->h_xlo = copy_bytes(p->x_min, es * nx); s->h_xhi = copy_bytes(p->x_max, es * nx);
    }
    if (p->u_min && p->u_max) {
        ok &= !upload(s->d_umin, p->u_min, es * nu * (N - 1)) && !upload(s->d_umax, p->u_max, es * nu * (N - 1));
        s->has_ub = true;
        s->h_ulo = copy_bytes(p->u_min, es * nu); s->h_uhi = copy_bytes(p->u_max, es * nu);
    }
    auto rd = [&](const void *base, int i) { return p->dtype == TINYMPC_F64 ? ((const double *)base)[i] : (double)((const float *)base)[i]; };
    s->ncx = p->num_state_cones; s->ncu = p->num_input_cones;
    for (int c = 0; c < s->ncx; ++c) { s->cone_x_start[c] = p->Acx[c]; s->cone_x_mu[c] = rd(p->cx, c); }
    for (int c = 0; c < s->ncu; ++c) { s->cone_u_start[c] = p->Acu[c]; s->cone_u_mu[c] = rd(p->cu, c); }
    s->nlx = p->num_state_linear; s->nlu = p->num_input_linear;
    if (s->nlx > 0) ok &= !upload(s->d_Alin_x, p->Alin_x, es * s->nlx * nx) && !upload(s->d_blin_x, p->blin_x, es * s->nlx);
    if (s->nlu > 0) ok &= !upload(s->d_Alin_u, p->Alin_u, es * s->nlu * nu) && !upload(s->d_blin_u, p->blin_u, es * s->nlu);
    s->ntvx = p->num_tv_state_linear; s->ntvu = p->num_tv_input_linear;
    if (s->ntvx > 0) ok &= !upload(s->d_tvA_x, p->tv_Alin_x, es * s->ntvx * N * nx) && !upload(s->d_tvb_x, p->tv_blin_x, es * s->ntvx * N);
    if (s->ntvu > 0) ok &= !upload(s->d_tvA_u, p->tv_Alin_u, es * s->ntvu * (N - 1) * nu) && !upload(s->d_tvb_u, p->tv_blin_u, es * s->ntvu * (N - 1));
    ok &= cudaEventCreate(&s->ev0) == cudaSuccess && cudaEventCreate(&s->ev1) == cudaSuccess &&
          cudaEventCreateWithFlags(&s->ev_last, cudaEventDisableTiming) == cudaSuccess;
    if (!ok) {
        tinympc_b200_destroy(s);
        return fail(TINYMPC_ERR_CUDA, std::string("problem upload failed: ") + cudaGetErrorString(cudaGetLastError()));
    }
    std::memset(&s->stats, 0, sizeof(s->stats));
    *out = s;
    return TINYMPC_OK;
}

int tinympc_b200_destroy(tinympc_b200_solver_t *s) {
    if (!s) return TINYMPC_OK;
    cudaSetDevice(s->device);
    DevBuf *bufs[] = {&s->d_xmin, &s->d_xmax, &s->d_umin, &s->d_umax, &s->d_Alin_x, &s->d_blin_x, &s->d_Alin_u,
                      &s->d_blin_u, &s->d_tvA_x, &s->d_tvb_x, &s->d_tvA_u, &s->d_tvb_u, &s->ws, &s->queue, &s->d_blob, &s->vscratch,
                      &s->shared_ref};
    for (DevBuf *b : bufs) b->release();
    for (int i = 0; i < tinympc_b200_solver::SLOTS; ++i) {
        s->dio[i].release();
        s->pin_in[i].release();
        s->pin_out[i].release();
        if (s->ev_in[i]) cudaEventDestroy(s->ev_in[i]);
        if (s->ev_k[i]) cudaEventDestroy(s->ev_k[i]);
        if (s->ev_out[i]) cudaEventDestroy(s->ev_out[i]);
    }
    if (s->st_h2d) cudaStreamDestroy(s->st_h2d);
    if (s->st_k) cudaStreamDestroy(s->st_k);
    if (s->st_d2h) cudaStreamDestroy(s->st_d2h);
    if (s->ev_last) cudaEventDestroy(s->ev_last);
    if (s->ev0) cudaEventDestroy(s->ev0);
    if (s->ev1) cudaEventDestroy(s->ev1);
    delete s;
    return TINYMPC_OK;
}

int tinympc_b200_update_settings(tinympc_b200_solver_t *s, const tinympc_settings_t *st) {
    if (!s || !st) return fail(TINYMPC_ERR_ARG, "null argument");
    if (st->check_termination <= 0) return fail(TINYMPC_ERR_ARG, "check_termination must be >= 1");
    s->settings = *st;
    return TINYMPC_OK;
}

int tinympc_b200_get_settings(const tinympc_b200_solver_t *s, tinympc_settings_t *st) {
    if (!s || !st) return fail(TINYMPC_ERR_ARG, "null argument");
    *st = s->settings;
    return TINYMPC_OK;
}

int tinympc_b200_set_mode(tinympc_b200_solver_t *s, int32_t mode, int32_t family) {
    if (!s) return fail(TINYMPC_ERR_ARG, "null solver");
    if (mode != TINYMPC_MODE_STRICT && mode != TINYMPC_MODE_FAST) return fail(TINYMPC_ERR_ARG, "bad mode");
    if (family != TINYMPC_KERNEL_AUTO && family != TINYMPC_KERNEL_TPI && family != TINYMPC_KERNEL_GPI && family != TINYMPC_KERNEL_GPS)
        return fail(TINYMPC_ERR_ARG, "bad kernel family");
    s->mode = mode;
    s->family = family;
    return TINYMPC_OK;
}

int tinympc_b200_solve(tinympc_b200_solver_t *s, const tinympc_batch_t *io, void *cuda_stream) {
    if (!s || !io) return fail(TINYMPC_ERR_ARG, "null argument");
    CUDA_TRY(cudaSetDevice(s->device));
    return enqueue(s, io, (cudaStream_t)cuda_stream, true);
}

int tinympc_b200_advance(tinympc_b200_solver_t *s, int64_t B, void *x0, const void *u, int64_t u_stride, void *cuda_stream) {
    if (!s || !x0 || !u) return fail(TINYMPC_ERR_ARG, "null argument");
    if (B <= 0) return TINYMPC_OK;
    CUDA_TRY(cudaSetDevice(s->device));
    // threads per block = a multiple of nx so that all rows of an instance read x0 before any row writes it
    const int per = std::max(1, 256 / s->nx) * s->nx;
    const int64_t total = B * s->nx;
    const unsigned blocks = (unsigned)((total + per - 1) / per);
    cudaStream_t st = (cudaStream_t)cuda_stream;
    if (s->dtype == TINYMPC_F32)
        advance_kernel<float><<<blocks, per, 0, st>>>(s->nx, s->nu, u_stride, B, (const float *)s->d_blob.p, (float *)x0, (const float *)u);
    else
        advance_kernel<double><<<blocks, per, 0, st>>>(s->nx, s->nu, u_stride, B, (const double *)s->d_blob.p, (double *)x0, (const double *)u);
    CUDA_TRY(cudaGetLastError());
    return TINYMPC_OK;
}

int tinympc_b200_get_stats(const tinympc_b200_solver_t *s, tinympc_b200_stats_t *out) {
    if (!s || !out) return fail(TINYMPC_ERR_ARG, "null argument");
    tinympc_b200_solver *m = const_cast<tinympc_b200_solver *>(s);
    if (m->timed) {
        CUDA_TRY(cudaSetDevice(s->device));
        CUDA_TRY(cudaEventSynchronize(m->ev1));
        float ms = 0.f;
        CUDA_TRY(cudaEventElapsedTime(&ms, m->ev0, m->ev1));
        m->stats.kernel_ms = ms;
        m->timed = false;
    }
    *out = m->stats;
    return TINYMPC_OK;
}

// ---------------------------------------------------------------------------------------------------------
// Host-pointer path.  The batch is cut into chunks; chunk c uses slot c % SLOTS (its own pinned in/out
// buffers and device io buffers).  Three streams: H2D, kernels, D2H, chained by events, so that the copy
// of chunk c+1 overlaps the solve of chunk c and the read-back of chunk c-1.
// ---------------------------------------------------------------------------------------------------------
namespace {

struct Field {
    const void *src;   // host input (may be null)
    void *dst;         // host output (may be null)
    size_t per_inst;   // bytes per instance
    bool is_in, is_out;
    void **dev_slot;   // where the device pointer goes in the device-side tinympc_batch_t
    bool pinned = false;  // the caller's buffer is page-locked: DMA straight from/to it, no staging copy
};

bool is_pinned(const void *p) {
    if (!p) return false;
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) {
        cudaGetLastError();
        return false;
    }
    return a.type == cudaMemoryTypeHost;
}

}  // namespace

int tinympc_b200_solve_host(tinympc_b200_solver_t *s, const tinympc_batch_t *io) {
    if (!s || !io) return fail(TINYMPC_ERR_ARG, "null argument");
    if (!io->x0 || !io->Xref) return fail(TINYMPC_ERR_ARG, "x0 and Xref are required");
    CUDA_TRY(cudaSetDevice(s->device));
    if (int rc = check_ready(s)) return rc;
    const int64_t B = io->B;
    if (B <= 0) return TINYMPC_OK;
    const size_t es = esize(s->dtype);
    const size_t bx = es * s->nx * s->N, bu = es * s->nu * (s->N - 1);
    constexpr int SLOTS = tinympc_b200_solver::SLOTS;
    if (!s->st_h2d) {
        CUDA_TRY(cudaStreamCreateWithFlags(&s->st_h2d, cudaStreamNonBlocking));
        CUDA_TRY(cudaStreamCreateWithFlags(&s->st_k, cudaStreamNonBlocking));
        CUDA_TRY(cudaStreamCreateWithFlags(&s->st_d2h, cudaStreamNonBlocking));
        for (int i = 0; i < SLOTS; ++i) {
            CUDA_TRY(cudaEventCreateWithFlags(&s->ev_in[i], cudaEventDisableTiming));
            CUDA_TRY(cudaEventCreateWithFlags(&s->ev_k[i], cudaEventDisableTiming));
            CUDA_TRY(cudaEventCreateWithFlags(&s->ev_out[i], cudaEventDisableTiming));
        }
    }

    // shared (not per-instance) references are uploaded once, into a buffer the handle keeps
    DevBuf &shared_ref = s->shared_ref;
    tinympc_batch_t dev = *io;  // template for the device-side descriptor
    const bool cold = io->cold_start != 0;
    std::vector<Field> fields;
    fields.push_back({io->x0, nullptr, es * s->nx, true, false, (void **)&dev.x0});
    if (io->xref_per_instance) fields.push_back({io->Xref, nullptr, bx, true, false, (void **)&dev.Xref});
    if (io->Uref && io->uref_per_instance) fields.push_back({io->Uref, nullptr, bu, true, false, (void **)&dev.Uref});
    if (io->models) fields.push_back({io->models, nullptr, es * (size_t)tinympc_b200_model_blob_elems(s->nx, s->nu), true, false, (void **)&dev.models});
    {
        size_t need = (io->xref_per_instance ? 0 : bx) + ((io->Uref && !io->uref_per_instance) ? bu : 0);
        if (need) {
            if (int rc = grow(s, shared_ref, need + 256, "shared reference")) return rc;
            char *c = (char *)shared_ref.p;
            if (!io->xref_per_instance) {
                CUDA_TRY(cudaMemcpyAsync(c, io->Xref, bx, cudaMemcpyHostToDevice, s->st_h2d));
                dev.Xref = c;
                c += (bx + 255) / 256 * 256;
            }
            if (io->Uref && !io->uref_per_instance) {
                CUDA_TRY(cudaMemcpyAsync(c, io->Uref, bu, cudaMemcpyHostToDevice, s->st_h2d));
                dev.Uref = c;
            }
        }
    }
    {
        void *const *sp = (void *const *)&io->state;
        void **dp = (void **)&dev.state;
        const int nfields = sizeof(tinympc_state_t) / sizeof(void *);
        for (int i = 0; i < nfields; ++i) {
            if (!sp[i]) continue;
            const bool is_x = (i % 2) == 0;  // x,v,vnew,g,... alternate with u,z,znew,y,...
            fields.push_back({cold ? nullptr : sp[i], sp[i], is_x ? bx : bu, !cold, true, &dp[i]});
        }
    }
    if (io->sol_x) fields.push_back({nullptr, io->sol_x, bx, false, true, (void **)&dev.sol_x});
    if (io->sol_u) fields.push_back({nullptr, io->sol_u, bu, false, true, (void **)&dev.sol_u});
    if (io->u0) fields.push_back({nullptr, io->u0, es * s->nu, false, true, (void **)&dev.u0});
    if (io->iter) fields.push_back({nullptr, io->iter, sizeof(int32_t), false, true, (void **)&dev.iter});
    if (io->solved) fields.push_back({nullptr, io->solved, sizeof(int32_t), false, true, (void **)&dev.solved});
    if (io->residuals) fields.push_back({nullptr, io->residuals, 4 * es, false, true, (void **)&dev.residuals});

    for (Field &f : fields) f.pinned = is_pinned(f.is_out ? f.dst : f.src) && (!f.is_in || !f.src || is_pinned(f.src));
    // chunking: big enough to fill the GPU several times over, small enough to pipeline
    int64_t chunk = B;
    if (B > 16384) chunk = std::max<int64_t>(8192, (B + 7) / 8);
    chunk = (chunk + 31) / 32 * 32;
    {   // the persistent GPI kernel holds sm_count * instances_per_cta instances at a time: make a chunk a whole
        // number of such waves so that no chunk ends on a mostly empty wave
        const Features ft = features(s);
        tinympc_batch_t first = *io;
        first.B = chunk;
        tmpc::LaunchDesc d;
        base_desc(s, d, ft, first);
        const tmpc::LaunchPlan gpi = s->dim->plan(d, TINYMPC_KERNEL_GPI);
        if (B > 16384 && resolve_family(s, ft, gpi, s->dim->plan(d, TINYMPC_KERNEL_GPS), chunk) == TINYMPC_KERNEL_GPI) {
            const int64_t wave = (int64_t)s->sm_count * gpi.instances_per_cta;
            if (wave > 0 && wave < B) chunk = std::max<int64_t>(1, (chunk + wave / 2) / wave) * wave;
        }
    }
    if (const char *e = std::getenv("TINYMPC_HOST_CHUNK")) {  // experiment knob
        long long v = std::atoll(e);
        if (v > 0) chunk = std::min<int64_t>(B, (v + 31) / 32 * 32);
    }
    const int64_t nchunks = (B + chunk - 1) / chunk;
    const size_t align = 256;
    auto padded = [&](size_t n) { return (n + align - 1) / align * align; };
    size_t dev_bytes = 0, in_bytes = 0, out_bytes = 0;
    for (const Field &f : fields) {
        dev_bytes += padded(f.per_inst * chunk);
        if (f.is_in) in_bytes += padded(f.per_inst * chunk);
        if (f.is_out) out_bytes += padded(f.per_inst * chunk);
    }
    const int used_slots = (int)std::min<int64_t>(SLOTS, nchunks);
    for (int i = 0; i < used_slots; ++i) {
        if (s->dio[i].ensure(dev_bytes) || s->pin_in[i].ensure(in_bytes + align) || s->pin_out[i].ensure(out_bytes + align))
            return fail(TINYMPC_ERR_CUDA, "staging allocation failed");
    }
    int64_t launches = 0;
    struct Pending { int64_t b0, nb; bool active; };
    Pending pend[SLOTS] = {};
    auto drain = [&](int slot) -> int {  // copy the pinned outputs of a finished chunk to the user's buffers
        if (!pend[slot].active) return 0;
        if (cudaEventSynchronize(s->ev_out[slot]) != cudaSuccess) return -1;
        char *po = (char *)s->pin_out[slot].p;
        for (const Field &f : fields) {
            if (!f.is_out) continue;
            if (!f.pinned) std::memcpy((char *)f.dst + f.per_inst * pend[slot].b0, po, f.per_inst * pend[slot].nb);
            po += padded(f.per_inst * chunk);
        }
        pend[slot].active = false;
        return 0;
    };
    for (int64_t c = 0; c < nchunks; ++c) {
        const int slot = (int)(c % SLOTS);
        const int64_t b0 = c * chunk, nb = std::min<int64_t>(chunk, B - b0);
        if (drain(slot)) return fail(TINYMPC_ERR_CUDA, "event sync failed");
        // stage inputs into pinned memory, then one async copy per field
        char *pi = (char *)s->pin_in[slot].p, *pd = (char *)s->dio[slot].p;
        tinympc_batch_t d = dev;
        d.B = nb;
        // device layout
        {
            char *cur = pd;
            const char *base = (const char *)&dev;
            for (const Field &f : fields) {
                size_t off = (const char *)f.dev_slot - base;
                *(void **)((char *)&d + off) = cur;
                cur += padded(f.per_inst * chunk);
            }
        }
        {
            char *cur = pd;
            for (const Field &f : fields) {
                if (f.is_in && f.src) {
                    const char *hsrc = (const char *)f.src + f.per_inst * b0;
                    if (!f.pinned) {
                        std::memcpy(pi, hsrc, f.per_inst * nb);
                        hsrc = pi;
                    }
                    CUDA_TRY(cudaMemcpyAsync(cur, hsrc, f.per_inst * nb, cudaMemcpyHostToDevice, s->st_h2d));
                    pi += padded(f.per_inst * chunk);
                }
                cur += padded(f.per_inst * chunk);
            }
        }
        CUDA_TRY(cudaEventRecord(s->ev_in[slot], s->st_h2d));
        CUDA_TRY(cudaStreamWaitEvent(s->st_k, s->ev_in[slot], 0));
        if (int rc = enqueue(s, &d, s->st_k, false)) return rc;
        launches += s->stats.kernel_launches;
        CUDA_TRY(cudaEventRecord(s->ev_k[slot], s->st_k));
        CUDA_TRY(cudaStreamWaitEvent(s->st_d2h, s->ev_k[slot], 0));
        {
            char *cur = pd, *po = (char *)s->pin_out[slot].p;
            for (const Field &f : fields) {
                if (f.is_out) {
                    char *hdst = f.pinned ? (char *)f.dst + f.per_inst * b0 : po;
                    CUDA_TRY(cudaMemcpyAsync(hdst, cur, f.per_inst * nb, cudaMemcpyDeviceToHost, s->st_d2h));
                    po += padded(f.per_inst * chunk);
                }
                cur += padded(f.per_inst * chunk);
            }
        }
        CUDA_TRY(cudaEventRecord(s->ev_out[slot], s->st_d2h));
        // the next use of this slot's pinned input buffer must wait for its H2D copy: ev_in is synchronised
        // implicitly because drain() waits for ev_out, which is ordered after ev_in.
        pend[slot] = {b0, nb, true};
    }
    for (int i = 0; i < SLOTS; ++i)
        if (drain(i)) return fail(TINYMPC_ERR_CUDA, "event sync failed");
    CUDA_TRY(cudaStreamSynchronize(s->st_h2d));
    s->stats.instances = B;
    s->stats.kernel_launches = launches;
    s->timed = false;
    s->stats.kernel_ms = 0.f;
    return TINYMPC_OK;
}

}  // extern "C"
