// kernels_inst.cu — compiled three times per supported (nx, nu) with -DTM_NX=.. -DTM_NU=.. -DTM_PART=0|1|2 (see Makefile):
//   part 0: thread-per-instance kernels (tpi_kernel.cuh), device precompute, and the type-erased DimEntry
//   part 1: on-chip lane-group kernels (gpi_kernel.cuh)
//   part 2: streamed lane-group kernels (gps_kernel.cuh)
// Three objects per dimension pair keep `make -j` busy and an edit of one kernel family from recompiling the others.
#include <algorithm>
#include <cstdlib>
#include <cstring>
#include <limits>

#include "kparams_fill.h"
#include "launch.h"

#if !defined(TM_NX) || !defined(TM_NU) || !defined(TM_PART)
#error "compile with -DTM_NX=<nx> -DTM_NU=<nu> -DTM_PART=<0|1|2>"
#endif

#define TM_CAT3(a, b, c) a##b##_##c
#define TM_CAT(a, b, c) TM_CAT3(a, b, c)
#define TM_SYM(prefix) TM_CAT(prefix, TM_NX, TM_NU)

// cross-part entry points of this dimension pair
extern "C" tmpc::LaunchPlan TM_SYM(tm_gpi_plan_)(const tmpc::LaunchDesc &d);
extern "C" int TM_SYM(tm_gpi_launch_)(tmpc::LaunchDesc *d, const tmpc::LaunchPlan &plan);
extern "C" tmpc::LaunchPlan TM_SYM(tm_gps_plan_)(const tmpc::LaunchDesc &d);
extern "C" int TM_SYM(tm_gps_launch_)(tmpc::LaunchDesc *d, const tmpc::LaunchPlan &plan);

#if TM_PART == 0
// =========================================================================================================
#include "precompute_kernel.cuh"
#include "tpi_kernel.cuh"

namespace tmpc {
namespace {

// bytes of one [N][vectors][Bpad] state / input array of the structure-of-arrays workspace
template <typename T>
size_t tpi_szx(const LaunchDesc &d) { return (size_t)d.N * SoA<T, TM_NX>::NV * 16 * d.Bpad; }
template <typename T>
size_t tpi_szu(const LaunchDesc &d) { return (size_t)(d.N - 1) * SoA<T, TM_NU>::NV * 16 * d.Bpad; }

template <typename T>
LaunchPlan tpi_plan(const LaunchDesc &d) {
    LaunchPlan p;
    if (d.io.models) return p;  // per-instance models live in the on-chip kernel's per-lane registers only
    p.family = TINYMPC_KERNEL_TPI;
    p.lanes = 1;
    p.threads = p.instances_per_cta = TPI_THREADS;
    p.ctas = (int)((d.io.B + TPI_THREADS - 1) / TPI_THREADS);
    // vnew (two buffers), g, znew (two buffers), y, d, and a slack / dual pair per enabled constraint family; 256 bytes slack
    const size_t nx_arrays = 3 + 2 * (d.soc_x + d.lin_x + d.tvl_x), nu_arrays = 4 + 2 * (d.soc_u + d.lin_u + d.tvl_u);
    p.workspace_bytes = nx_arrays * tpi_szx<T>(d) + nu_arrays * tpi_szu<T>(d) + 256;
    return p;
}

template <typename T, bool FAST, bool EXT>
int launch_tpi(LaunchDesc *d, const LaunchPlan &plan) {
    KParams<T, TM_NX, TM_NU> P;
    fill_params<T, TM_NX, TM_NU>(P, *d);
    // carve the workspace in tpi_plan's order (the arrays of disabled families stay null)
    const size_t szx = tpi_szx<T>(*d), szu = tpi_szu<T>(*d);
    char *c = (char *)d->workspace;
    auto take = [&](size_t n) {
        void *r = c;
        c += n;
        return r;
    };
    P.w_v[0] = take(szx); P.w_v[1] = take(szx); P.w_g = take(szx);
    P.w_z[0] = take(szu); P.w_z[1] = take(szu); P.w_y = take(szu); P.w_d = take(szu);
    if (d->soc_x) { P.w_vc = take(szx); P.w_gc = take(szx); }
    if (d->soc_u) { P.w_zc = take(szu); P.w_yc = take(szu); }
    if (d->lin_x) { P.w_vl = take(szx); P.w_gl = take(szx); }
    if (d->lin_u) { P.w_zl = take(szu); P.w_yl = take(szu); }
    if (d->tvl_x) { P.w_vlt = take(szx); P.w_glt = take(szx); }
    if (d->tvl_u) { P.w_zlt = take(szu); P.w_ylt = take(szu); }
    tpi_solve_kernel<T, TM_NX, TM_NU, FAST, EXT><<<(unsigned)plan.ctas, plan.threads, 0, d->stream>>>(P);
    return cudaGetLastError() == cudaSuccess ? TINYMPC_OK : TINYMPC_ERR_CUDA;
}

template <typename T>
int launch_T(LaunchDesc *d, const LaunchPlan &plan) {
    if (d->ext) return d->fast ? launch_tpi<T, true, true>(d, plan) : launch_tpi<T, false, true>(d, plan);
    return d->fast ? launch_tpi<T, true, false>(d, plan) : launch_tpi<T, false, false>(d, plan);
}

LaunchPlan plan(const LaunchDesc &d, int family) {
    if (family == TINYMPC_KERNEL_GPI) return TM_SYM(tm_gpi_plan_)(d);
    if (family == TINYMPC_KERNEL_GPS) return TM_SYM(tm_gps_plan_)(d);
    if (family != TINYMPC_KERNEL_TPI) return {};
    if (d.dtype == TINYMPC_F32) return tpi_plan<float>(d);
    if (d.dtype == TINYMPC_F64) return tpi_plan<double>(d);
    return {};
}

int launch(LaunchDesc *d, const LaunchPlan &plan) {
    if (plan.family == TINYMPC_KERNEL_GPI) return TM_SYM(tm_gpi_launch_)(d, plan);
    if (plan.family == TINYMPC_KERNEL_GPS) return TM_SYM(tm_gps_launch_)(d, plan);
    if (plan.family != TINYMPC_KERNEL_TPI) return TINYMPC_ERR_UNSUPPORTED;
    if (d->dtype == TINYMPC_F32) return launch_T<float>(d, plan);
    if (d->dtype == TINYMPC_F64) return launch_T<double>(d, plan);
    return TINYMPC_ERR_ARG;
}

int precompute_batch(int dtype, int64_t B, const void *A, const void *Bm, const void *f, const void *Qdiag, const void *Rdiag,
                     const void *rho, void *models_out, int32_t *sweeps_out, int sm_count, cudaStream_t stream) {
    if (dtype == TINYMPC_F32)
        return launch_precompute_T<float, TM_NX, TM_NU>(B, A, Bm, f, Qdiag, Rdiag, rho, models_out, sweeps_out, sm_count, stream);
    if (dtype == TINYMPC_F64)
        return launch_precompute_T<double, TM_NX, TM_NU>(B, A, Bm, f, Qdiag, Rdiag, rho, models_out, sweeps_out, sm_count, stream);
    return TINYMPC_ERR_ARG;
}

}  // namespace
}  // namespace tmpc

extern "C" const tmpc::DimEntry *TM_SYM(tm_dim_entry_)() {
    static const tmpc::DimEntry e = {TM_NX, TM_NU, &tmpc::plan, &tmpc::launch, &tmpc::precompute_batch};
    return &e;
}

#elif TM_PART == 1
// =========================================================================================================
#include "tpi_kernel.cuh"  // Vec16
#include "gpi_kernel.cuh"

namespace tmpc {
namespace {

template <typename T, int NX, int NU, bool FAST>
int launch_gpi(LaunchDesc *d, const LaunchPlan &plan) {
    KParams<T, NX, NU> P;
    fill_params<T, NX, NU>(P, *d);
    const T *gmat = (const T *)d->gmat;
    const bool het = d->io.models != nullptr;  // heterogeneous batch: per-instance model blobs
    const bool tm = plan.tmem_cols != 0;
    // STRICT, shared model, tensor-memory plan (the headline path): min / max clamp when no bound is a signed zero
#define TM_GPI_CASE(LL, HH, TT)                                                                                          \
    if (plan.lanes == LL && het == HH && tm == TT) {                                                                     \
        if constexpr (!FAST && !HH && TT && sizeof(T) == 4) {                                                            \
            if (d->bounds_zero_free) return launch_gpi_L<T, NX, NU, LL, FAST, HH, TT, true>(d, plan, P, gmat);           \
        }                                                                                                                \
        return launch_gpi_L<T, NX, NU, LL, FAST, HH, TT>(d, plan, P, gmat);                                              \
    }
#define TM_GPI_L(LL) TM_GPI_CASE(LL, false, false) TM_GPI_CASE(LL, true, false) TM_GPI_CASE(LL, false, true) TM_GPI_CASE(LL, true, true)
    TM_GPI_L(4)
    TM_GPI_L(8)
#ifdef TM_GPI_L16
    TM_GPI_L(16)
#else
    if constexpr (sizeof(T) == 8) {  // fp64 may need L = 16 for the widest states (see gpi_plan)
        TM_GPI_L(16)
    }
#endif
#undef TM_GPI_L
#undef TM_GPI_CASE
    return TINYMPC_ERR_UNSUPPORTED;
}

}  // namespace
}  // namespace tmpc

extern "C" tmpc::LaunchPlan TM_SYM(tm_gpi_plan_)(const tmpc::LaunchDesc &d) {
    if (d.ext) return {};  // the on-chip kernel covers box constraints; the rest streams (gps)
    if (d.dtype == TINYMPC_F32) return tmpc::gpi_plan<float, TM_NX, TM_NU>(d);
    if (d.dtype == TINYMPC_F64) return tmpc::gpi_plan<double, TM_NX, TM_NU>(d);
    return {};
}
extern "C" int TM_SYM(tm_gpi_launch_)(tmpc::LaunchDesc *d, const tmpc::LaunchPlan &plan) {
    if (d->dtype == TINYMPC_F32) return d->fast ? tmpc::launch_gpi<float, TM_NX, TM_NU, true>(d, plan) : tmpc::launch_gpi<float, TM_NX, TM_NU, false>(d, plan);
    if (d->dtype == TINYMPC_F64) return d->fast ? tmpc::launch_gpi<double, TM_NX, TM_NU, true>(d, plan) : tmpc::launch_gpi<double, TM_NX, TM_NU, false>(d, plan);
    return TINYMPC_ERR_ARG;
}

#else
// =========================================================================================================
#include "gps_kernel.cuh"

namespace tmpc {
namespace {

template <typename T>
LaunchPlan plan_T(const LaunchDesc &d) {
    if (d.io.models) return {};  // per-instance models live in the on-chip kernel only
    return gps_variant<T, TM_NX, TM_NU>(d, gps_env_int("TINYMPC_GPS_NI", 0), LaunchPlan{}, [&](auto l, auto ni, auto fam) {
        return gps_plan_L<T, TM_NX, TM_NU, decltype(l)::value, decltype(ni)::value, decltype(fam)::value>(d);
    });
}

template <typename T>
int launch_T(LaunchDesc *d, const LaunchPlan &plan) {
    KParams<T, TM_NX, TM_NU> P;
    fill_params<T, TM_NX, TM_NU>(P, *d);
    return gps_variant<T, TM_NX, TM_NU>(*d, plan.group_instances, (int)TINYMPC_ERR_UNSUPPORTED, [&](auto l, auto ni, auto fam) {
        constexpr int L = decltype(l)::value, NI = decltype(ni)::value, FAM = decltype(fam)::value;
        return d->fast ? launch_gps_cfg<T, TM_NX, TM_NU, L, NI, FAM, true>(d, plan, P) : launch_gps_cfg<T, TM_NX, TM_NU, L, NI, FAM, false>(d, plan, P);
    });
}

}  // namespace
}  // namespace tmpc

extern "C" tmpc::LaunchPlan TM_SYM(tm_gps_plan_)(const tmpc::LaunchDesc &d) {
    if (d.dtype == TINYMPC_F32) return tmpc::plan_T<float>(d);
    if (d.dtype == TINYMPC_F64) return tmpc::plan_T<double>(d);
    return {};
}
extern "C" int TM_SYM(tm_gps_launch_)(tmpc::LaunchDesc *d, const tmpc::LaunchPlan &plan) {
    if (d->dtype == TINYMPC_F32) return tmpc::launch_T<float>(d, plan);
    if (d->dtype == TINYMPC_F64) return tmpc::launch_T<double>(d, plan);
    return TINYMPC_ERR_ARG;
}
#endif
