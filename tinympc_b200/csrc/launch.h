// launch.h — type-erased launch descriptor between the C-ABI layer (capi.cu) and the per-(nx,nu)
// kernel translation units (kernels_inst.cu compiled once per supported dimension pair).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/tinympc_b200.h"

namespace tmpc {

struct LaunchDesc {
    int dtype;   // TINYMPC_F32 / F64
    int fast;    // TINYMPC_MODE_FAST ?
    int ext;     // any of soc / linear / tv-linear enabled

    // host copies of the model + cache in the native dtype (column-major)
    const void *A, *Bm, *f, *Qd, *Rd, *Kinf, *Pinf, *Quu, *AmBKt, *APf, *BPf;
    double rho, pri_tol, dua_tol;
    int N, max_iter, check_termination;
    int en_state_bound, en_input_bound;
    int soc_x, soc_u, ncx, ncu;
    int lin_x, lin_u, nlx, nlu;
    int tvl_x, tvl_u, ntvx, ntvu;
    int cone_x_start[4], cone_u_start[4];
    double cone_x_mu[4], cone_u_mu[4];  // already rounded to the native dtype

    // device pointers
    const void *x_min, *x_max, *u_min, *u_max;
    const void *Alin_x, *blin_x, *Alin_u, *blin_u, *tv_Alin_x, *tv_blin_x, *tv_Alin_u, *tv_blin_u;
    tinympc_batch_t io;  // device pointers
    int64_t Bpad;
    const void *gmat;  // device blob: A,B,f,Qd,Rd,Kinf,Pinf,Quu,AmBKt,APf,BPf packed (native dtype)
    int bounds_tv;
    int bounds_zero_free;  // no element of the box bounds is +-0 (lets STRICT kernels clamp with min / max instructions)
    const void *h_xlo, *h_xhi, *h_ulo, *h_uhi;  // host copies of column 0 of the bounds (native dtype), may be null
    void *work_queue;  // GPI / GPS: device int64 counter (zeroed by the caller)
    void *workspace;   // TPI / GPS: LaunchPlan::workspace_bytes, allocated by the caller
    void *scratch;     // GPI: LaunchPlan::scratch_bytes, allocated by the caller (null when the plan needs none)

    cudaStream_t stream;
    int sm_count;
    int smem_budget;  // dynamic shared memory a CTA may use: the opt-in limit less 64 bytes of static shared memory
};

// How one solve runs, decided by the kernel family's own translation unit before anything is allocated or launched:
// the caller allocates from it, launches with it and reports it through tinympc_b200_stats_t.
struct LaunchPlan {
    int family = 0;              // TINYMPC_KERNEL_TPI / GPI / GPS; 0 = this family cannot serve the solve
    int lanes = 0;               // lanes per instance (TPI: 1)
    int group_instances = 0;     // GPS: instances per lane group
    int tmem_cols = 0;           // GPI: tensor-memory columns per CTA (0 = the whole state in shared memory)
    int warps_resident = 0;      // GPI / GPS: warps per CTA the on-chip memory holds
    int instances_per_cta = 0;   // GPI: capacity (warps_resident); GPS: of this launch; TPI: threads per CTA
    int ctas = 0, threads = 0;   // launch geometry for this batch
    size_t smem = 0;             // dynamic shared memory per CTA
    size_t workspace_bytes = 0;  // TPI structure-of-arrays / GPS state records
    size_t scratch_bytes = 0;    // GPI: previous-slack scratch, when state.v / state.z is requested
    int gps_has_b = 0;           // GPS: the records carry region B (previous / family slacks)
};

// per-(nx,nu) entry.  plan: host arithmetic only, no CUDA calls.  launch: 0 on success, TINYMPC_ERR_UNSUPPORTED when
// the planned variant is not compiled, TINYMPC_ERR_CUDA when the launch fails.
struct DimEntry {
    int nx, nu;
    LaunchPlan (*plan)(const LaunchDesc &d, int family);
    int (*launch)(LaunchDesc *d, const LaunchPlan &plan);
    // batched cache precompute on the device (precompute_kernel.cuh): device pointers, one model blob per instance
    int (*precompute_batch)(int dtype, int64_t B, const void *A, const void *Bm, const void *f, const void *Qdiag, const void *Rdiag,
                            const void *rho, void *models_out, int32_t *sweeps_out, int sm_count, cudaStream_t stream);
};

}  // namespace tmpc

// the list of compiled dimension pairs: X(nx, nu)
#define TM_DIMS(X) \
    X(4, 1)        \
    X(6, 3)        \
    X(12, 4)       \
    X(4, 2)        \
    X(4, 4)        \
    X(4, 8)        \
    X(8, 2)        \
    X(8, 4)        \
    X(8, 8)        \
    X(12, 2)       \
    X(12, 8)       \
    X(16, 2)       \
    X(16, 4)       \
    X(16, 8)
