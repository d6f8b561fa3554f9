// gpi_kernel.cuh — lane-group-per-instance (GPI) batched ADMM solve with the whole per-instance state
// resident on chip.  This is the kernel BASELINE.json's north_star describes.
//
//   * L lanes (4, 8 or 16) own one MPC instance, 32/L instances per warp; lane l owns the state rows
//     [l*RX, (l+1)*RX) and the input rows [l*RU, (l+1)*RU)  (RX = ceil(nx/L), RU = ceil(nu/L)) of every vector.
//   * the rows of Kinf / Quu_inv / AmBKt / A / B that a lane needs are loaded ONCE into registers (staged
//     through shared memory by a TMA bulk copy, cp.async.bulk), the p / x recursions run in registers, each
//     mat-vec is RX (or RU) independent ascending-k dot products per lane (bit-identical to the pinned
//     oracle in STRICT mode), and the freshly computed vector is all-gathered inside the lane group through
//     a small shared-memory buffer (STS + 16-byte broadcast LDS);
//   * the N-indexed state lives on chip for the whole solve: the primal pack (vnew rows, znew rows) as one
//     16-byte vector per lane and knot point in shared memory; the dual pack (g rows, y rows) and d either next
//     to it in shared memory, or (TM = true) in TENSOR MEMORY — the thread's own 32-bit TMEM columns, 5 per knot point in
//     fp32 (two per fp64 value), tcgen05.ld/st.32x32b — which halves the shared-memory footprint and doubles the instances
//     (= warps) resident per SM; only the final trajectories / residuals are written back;
//   * fp64: only the rows of the running sweep are in registers (re-read from the resident blob at every sweep start), so
//     that narrower lane groups fit (gpi_per_sweep_rows);
//   * the kernel is persistent: one CTA per SM; every lane group ("slot") pulls its next instance from a
//     global atomic counter as soon as its current one terminates (per-instance termination, admm.cpp:310-328).
// Reference semantics: tiny_solve -> solve (admm.cpp:331-455); per-iteration order as in SURVEY A.2.
// Scope: box constraints (admm.cpp:85-98).  Cones / hyperplanes run on the streamed lane-group kernel (gps_kernel.cuh).
#pragma once
#include <cuda/barrier>

#include "common.cuh"
#include "launch.h"

namespace tmpc {

template <int NX, int NU, int L, int ES>
struct GpiCfg {
    static constexpr int RX = (NX + L - 1) / L;
    static constexpr int RU = (NU + L - 1) / L;
    static constexpr int IPW = 32 / L;      // instances per warp
    static constexpr int W = 16 / ES;       // elements per 16-byte shared-memory vector
    static constexpr int PV = RX + RU;      // values a lane owns per knot point (state rows, then input rows)
    static constexpr int PVP = (PV + W - 1) / W * W;
    static constexpr int NPV = PVP / W;     // vectors per pack
    static constexpr int NXP = (L * RX + W - 1) / W * W;  // gather buffer width (state vectors)
    static constexpr int NUP = (L * RU + W - 1) / W * W;  // gather buffer width (input vectors)
    static constexpr int GBUF1 = IPW * (NXP > NUP ? NXP : NUP);  // one gather buffer
    static constexpr int GBUF = 3 * GBUF1;  // tensor-memory variant: three of them, each hot call site owns one (see gather_x)
    // registers needed for the per-lane matrix rows (in elements of T)
    static constexpr int MAT_REGS = RX * (2 * NX + 2 * NU + 3) + RU * (2 * NX + NU + 2);
    // shared-memory elements per warp for horizon N: primal pack + dual pack per (k, lane), d, gather scratch
    __host__ __device__ static constexpr size_t warp_elems(int N) {
        return (size_t)N * 32 * PVP * 2 + (size_t)(N - 1) * RU * 32 + GBUF1;  // shared memory is the constraint here: one gather buffer
    }
    // per-sweep register needs (elements): backward AmBKt / B^T rows, Kinf^T, Quu_inv, APf, BPf, Qd, Rd; forward A / Kinf rows, B, f
    static constexpr int BWD_REGS = (RX + RU) * NX + RX * NU + RU * NU + 2 * RX + 2 * RU;
    static constexpr int FWD_REGS = (RX + RU) * NX + RX * NU + RX;
    static constexpr int SWEEP_REGS = BWD_REGS > FWD_REGS ? BWD_REGS : FWD_REGS;
    // TMEM variant: the dual pack and d live in tensor memory, CPK 32-bit columns per knot point (two per fp64 value) in
    // the lane of the owning thread; shared memory keeps the primal pack and the gather scratch
    static constexpr int CW = ES / 4;  // 32-bit columns per value
    static constexpr int CPK = (PVP + RU) * CW;
    __host__ __device__ static constexpr size_t warp_elems_tm(int N) { return (size_t)N * 32 * PVP + GBUF; }
    __host__ __device__ static constexpr int tm_cols(int N) { return N * CPK; }
};

// fp64: only the rows of the RUNNING sweep are in registers (re-read from the staged blob in shared memory - or from the
// instance's own blob in a heterogeneous batch - at every sweep start), which halves the register footprint of the matrices
// and lets fp64 problems use narrower lane groups (nx = 12: L = 8 instead of 16, twice the instances per warp)
template <typename T>
__host__ __device__ constexpr bool gpi_per_sweep_rows() {
    return sizeof(T) == 8;
}
template <typename T, int NX, int NU, int L>
__host__ __device__ constexpr bool gpi_feasible() {
    // keep the matrix rows + working set under the 255-register ceiling
    using Cfg = GpiCfg<NX, NU, L, (int)sizeof(T)>;
    if (gpi_per_sweep_rows<T>()) return Cfg::SWEEP_REGS * 2 <= 112;
    return Cfg::MAT_REGS * (int)(sizeof(T) / 4) <= 150;
}

template <typename T, int L>
__device__ __forceinline__ T group_max(T v) {
#pragma unroll
    for (int m = L / 2; m >= 1; m >>= 1) {
        T o = __shfl_xor_sync(0xffffffffu, v, m, L);
        v = (o > v) ? o : v;
    }
    return v;
}

constexpr int GPI_MAX_WARPS = 8;

// Shared-memory accessors on 32-bit shared-window addresses (no generic->shared conversion, no 64-bit
// address arithmetic in the hot loops).  16-byte vector forms move a whole per-lane pack per instruction.
__device__ __forceinline__ float lds(unsigned a, float) {
    float v;
    asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(a));
    return v;
}
__device__ __forceinline__ double lds(unsigned a, double) {
    double v;
    asm volatile("ld.shared.f64 %0, [%1];" : "=d"(v) : "r"(a));
    return v;
}
__device__ __forceinline__ void sts(unsigned a, float v) { asm volatile("st.shared.f32 [%0], %1;" ::"r"(a), "f"(v) : "memory"); }
__device__ __forceinline__ void sts(unsigned a, double v) { asm volatile("st.shared.f64 [%0], %1;" ::"r"(a), "d"(v) : "memory"); }
__device__ __forceinline__ void ldsv(unsigned a, float (&v)[4]) {
    asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(v[0]), "=f"(v[1]), "=f"(v[2]), "=f"(v[3]) : "r"(a));
}
__device__ __forceinline__ void ldsv(unsigned a, double (&v)[2]) {
    asm volatile("ld.shared.v2.f64 {%0,%1}, [%2];" : "=d"(v[0]), "=d"(v[1]) : "r"(a));
}
__device__ __forceinline__ void stsv(unsigned a, const float (&v)[4]) {
    asm volatile("st.shared.v4.f32 [%0], {%1,%2,%3,%4};" ::"r"(a), "f"(v[0]), "f"(v[1]), "f"(v[2]), "f"(v[3]) : "memory");
}
__device__ __forceinline__ void stsv(unsigned a, const double (&v)[2]) {
    asm volatile("st.shared.v2.f64 [%0], {%1,%2};" ::"r"(a), "d"(v[0]), "d"(v[1]) : "memory");
}

// Tensor memory (TMEM, 128 lanes x 512 32-bit columns per SM) used as a per-thread scratchpad: warp w of a CTA owns
// TMEM lanes [32*(w%4), +32), thread t of the warp lane 32*(w%4)+t.  `32x32b` moves n consecutive columns of the
// thread's own lane to / from n registers.  Loads are asynchronous: tm_wait_ld() + tm_tie() before the first use.
__device__ __forceinline__ void tm_ld(unsigned ta, float (&v)[1]) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x1.b32 {%0}, [%1];" : "=f"(v[0]) : "r"(ta));
}
__device__ __forceinline__ void tm_ld(unsigned ta, float (&v)[2]) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x2.b32 {%0,%1}, [%2];" : "=f"(v[0]), "=f"(v[1]) : "r"(ta));
}
__device__ __forceinline__ void tm_ld(unsigned ta, float (&v)[4]) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0,%1,%2,%3}, [%4];" : "=f"(v[0]), "=f"(v[1]), "=f"(v[2]), "=f"(v[3]) : "r"(ta));
}
__device__ __forceinline__ void tm_st(unsigned ta, const float (&v)[1]) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x1.b32 [%0], {%1};" ::"r"(ta), "f"(v[0]) : "memory");
}
__device__ __forceinline__ void tm_st(unsigned ta, const float (&v)[2]) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x2.b32 [%0], {%1,%2};" ::"r"(ta), "f"(v[0]), "f"(v[1]) : "memory");
}
__device__ __forceinline__ void tm_st(unsigned ta, const float (&v)[4]) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x4.b32 [%0], {%1,%2,%3,%4};" ::"r"(ta), "f"(v[0]), "f"(v[1]), "f"(v[2]), "f"(v[3]) : "memory");
}
__device__ __forceinline__ void tm_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tm_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
// makes every later use of v depend on an asm statement that is ordered after tm_wait_ld()
__device__ __forceinline__ void tm_tie(float &v) { asm volatile("" : "+f"(v)); }
// fp64 values occupy two consecutive 32-bit columns (low word first)
__device__ __forceinline__ void tm_tie(double &v) { asm volatile("" : "+d"(v)); }
__device__ __forceinline__ void tm_ld(unsigned ta, double (&v)[1]) {
    unsigned lo, hi;
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x2.b32 {%0,%1}, [%2];" : "=r"(lo), "=r"(hi) : "r"(ta));
    asm volatile("mov.b64 %0, {%1,%2};" : "=d"(v[0]) : "r"(lo), "r"(hi));
}
__device__ __forceinline__ void tm_ld(unsigned ta, double (&v)[2]) {
    unsigned w0, w1, w2, w3;
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0,%1,%2,%3}, [%4];" : "=r"(w0), "=r"(w1), "=r"(w2), "=r"(w3) : "r"(ta));
    asm volatile("mov.b64 %0, {%1,%2};" : "=d"(v[0]) : "r"(w0), "r"(w1));
    asm volatile("mov.b64 %0, {%1,%2};" : "=d"(v[1]) : "r"(w2), "r"(w3));
}
__device__ __forceinline__ void tm_st(unsigned ta, const double (&v)[1]) {
    unsigned lo, hi;
    asm volatile("mov.b64 {%0,%1}, %2;" : "=r"(lo), "=r"(hi) : "d"(v[0]));
    asm volatile("tcgen05.st.sync.aligned.32x32b.x2.b32 [%0], {%1,%2};" ::"r"(ta), "r"(lo), "r"(hi) : "memory");
}
__device__ __forceinline__ void tm_st(unsigned ta, const double (&v)[2]) {
    unsigned w0, w1, w2, w3;
    asm volatile("mov.b64 {%0,%1}, %2;" : "=r"(w0), "=r"(w1) : "d"(v[0]));
    asm volatile("mov.b64 {%0,%1}, %2;" : "=r"(w2), "=r"(w3) : "d"(v[1]));
    asm volatile("tcgen05.st.sync.aligned.32x32b.x4.b32 [%0], {%1,%2,%3,%4};" ::"r"(ta), "r"(w0), "r"(w1), "r"(w2), "r"(w3) : "memory");
}

template <bool B>
struct BoolTag {
    static constexpr bool value = B;
};
template <int J>
struct IntTag {
    static constexpr int value = J;
};

// Box clamp.  STRICT keeps Eigen's compare-select form (differs from fmax/fmin only in the sign of a zero
// result when a bound is a signed zero); FAST uses the single-instruction min/max.
template <bool FAST, typename T>
__device__ __forceinline__ T clamp_box(T v, T lo, T hi) {
    if constexpr (FAST) {
        return fmin(fmax(v, lo), hi);
    } else {
        return clamp_ref(v, lo, hi);
    }
}
// max(m, |d|): identical to the oracle's (|d| > m) ? |d| : m  because m is never NaN and |d| >= +0
__device__ __forceinline__ float absmax(float m, float d) { return fmaxf(m, fabsf(d)); }
// fp64: the oracle's compare-select itself.  fmax(double) has no single instruction: DSETP.MAX + SEL + FSEL + a NaN-quieting
// LOP3 + register moves, 7 instructions per use and 9 % of the streamed fp64 kernel's instruction count (ncu source view).
__device__ __forceinline__ double absmax(double m, double d) {
    const double a = fabs(d);
    return (a > m) ? a : m;
}

// MM (STRICT only): the box clamp as min / max instructions.  Identical to Eigen's compare-select form for every input
// (NaN included: both return the bound) except when a bound is a signed zero - the host sets MM only when no bound is +-0.
template <typename T, int NX, int NU, int L, bool FAST, bool HET, bool TM, bool MM = false>
__global__ void __launch_bounds__(GPI_MAX_WARPS * 32, 1)
    gpi_solve_kernel(const __grid_constant__ KParams<T, NX, NU> P, const T *__restrict__ gmat, unsigned long long *queue) {
    using Cfg = GpiCfg<NX, NU, L, (int)sizeof(T)>;
    constexpr int RX = Cfg::RX, RU = Cfg::RU, IPW = Cfg::IPW, W = Cfg::W, PVP = Cfg::PVP, NPV = Cfg::NPV;
    constexpr int NXP = Cfg::NXP, NUP = Cfg::NUP, CPK = Cfg::CPK;
    constexpr int CW = Cfg::CW;        // 32-bit tensor-memory columns per value
    constexpr bool PS = gpi_per_sweep_rows<T>();  // matrix rows re-read at every sweep start (fp64)
    constexpr bool EXACT = (RX * L == NX) && (RU * L == NU);  // no padding rows: predicates vanish
    constexpr unsigned ES = (unsigned)sizeof(T);
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int N = P.N;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int l = lane % L;     // lane inside the instance group
    const int slot = lane / L;  // which of the warp's instances
    // HET = heterogeneous batch (tinympc_batch_t.models): every instance brings its own model / cache blob and rho;
    // the homogeneous kernel keeps rho a launch constant and its matrix rows immutable registers.
    T rho_m = P.rho;
    auto rho_ = [&]() -> T {
        if constexpr (HET) return rho_m;
        else return P.rho;
    };

    // ---- stage the cache blob (A, B, f, Qd, Rd, Kinf, Pinf, Quu, AmBKt, APf, BPf) into shared memory with
    // one TMA bulk copy per CTA, then pull this lane's rows into registers.  The staging area aliases the
    // first warp's state region and is dead before the solve starts.
    constexpr int OFF_A = 0, OFF_B = OFF_A + NX * NX, OFF_F = OFF_B + NX * NU, OFF_QD = OFF_F + NX, OFF_RD = OFF_QD + NX,
                  OFF_K = OFF_RD + NU, OFF_PINF = OFF_K + NU * NX, OFF_QUU = OFF_PINF + NX * NX,
                  OFF_AMBKT = OFF_QUU + NU * NU, OFF_APF = OFF_AMBKT + NX * NX, OFF_BPF = OFF_APF + NX,
                  BLOB = OFF_BPF + NU;
    constexpr unsigned BLOB_BYTES = (unsigned)(((BLOB * sizeof(T) + 15) / 16) * 16);
    T *stage = reinterpret_cast<T *>(smem_raw);
    __shared__ __align__(8) unsigned long long mbar;
    if (threadIdx.x == 0) {
        const unsigned mb = (unsigned)__cvta_generic_to_shared(&mbar);
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(mb));
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(mb), "r"(BLOB_BYTES) : "memory");
        asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                         (unsigned)__cvta_generic_to_shared(stage)),
                     "l"(gmat), "r"(BLOB_BYTES), "r"(mb)
                     : "memory");
    }
    __syncthreads();
    {
        const unsigned mb = (unsigned)__cvta_generic_to_shared(&mbar);
        unsigned done = 0;
        while (!done) {
            asm volatile(
                "{\n .reg .pred p;\n mbarrier.try_wait.parity.shared::cta.b64 p, [%1], 0;\n selp.u32 %0, 1, 0, p;\n}\n"
                : "=r"(done)
                : "r"(mb)
                : "memory");
        }
    }

    // per-lane matrix rows (registers)
    // stage-1 rows (dot with the gathered nx-vector): backward = [AmBKt rows ; B^T rows], forward = [A rows ; Kinf rows]
    T mS1b[RX + RU][NX], mS1f[RX + RU][NX];
    T mKt[RX][NU], mB[RX][NU], vQd[RX], vAPf[RX], vf[RX];
    T mQuu[RU][NU], vRd[RU], vBPf[RU];
    bool xv[RX], uv[RU];  // row validity (padding rows compute zeros)
#pragma unroll
    for (int a = 0; a < RX; ++a) xv[a] = EXACT || (l * RX + a < NX);
#pragma unroll
    for (int b = 0; b < RU; ++b) uv[b] = EXACT || (l * RU + b < NU);
    // `src` = a cache blob in the layout above (the staged shared-memory copy, or one instance's blob in global memory).
    // Backward-sweep rows (AmBKt, B^T, Kinf^T, Quu_inv, APf, BPf and the cost weights Qd, Rd) and forward-sweep rows (A, Kinf,
    // B, f) load separately: fp64 re-reads the rows of a sweep when it starts (PS), everything else loads both once.
    auto load_bwd_rows = [&](const T *src) {
#pragma unroll
        for (int a = 0; a < RX; ++a) {
            const int ii = xv[a] ? l * RX + a : 0;
#pragma unroll
            for (int m = 0; m < NX; ++m) mS1b[a][m] = xv[a] ? src[OFF_AMBKT + ii + NX * m] : T(0);
#pragma unroll
            for (int j = 0; j < NU; ++j) mKt[a][j] = xv[a] ? src[OFF_K + j + NU * ii] : T(0);  // Kinf^T(i,j) = Kinf(j,i)
            vQd[a] = xv[a] ? src[OFF_QD + ii] : T(0);
            vAPf[a] = xv[a] ? src[OFF_APF + ii] : T(0);
        }
#pragma unroll
        for (int b = 0; b < RU; ++b) {
            const int jj = uv[b] ? l * RU + b : 0;
#pragma unroll
            for (int m = 0; m < NX; ++m) mS1b[RX + b][m] = uv[b] ? src[OFF_B + m + NX * jj] : T(0);  // B^T(j,m) = B(m,j)
#pragma unroll
            for (int m = 0; m < NU; ++m) mQuu[b][m] = uv[b] ? src[OFF_QUU + jj + NU * m] : T(0);
            vRd[b] = uv[b] ? src[OFF_RD + jj] : T(0);
            vBPf[b] = uv[b] ? src[OFF_BPF + jj] : T(0);
        }
    };
    auto load_fwd_rows = [&](const T *src) {
#pragma unroll
        for (int a = 0; a < RX; ++a) {
            const int ii = xv[a] ? l * RX + a : 0;
#pragma unroll
            for (int m = 0; m < NX; ++m) mS1f[a][m] = xv[a] ? src[OFF_A + ii + NX * m] : T(0);
#pragma unroll
            for (int j = 0; j < NU; ++j) mB[a][j] = xv[a] ? src[OFF_B + ii + NX * j] : T(0);
            vf[a] = xv[a] ? src[OFF_F + ii] : T(0);
        }
#pragma unroll
        for (int b = 0; b < RU; ++b) {
            const int jj = uv[b] ? l * RU + b : 0;
#pragma unroll
            for (int m = 0; m < NX; ++m) mS1f[RX + b][m] = uv[b] ? src[OFF_K + jj + NU * m] : T(0);
        }
    };
    auto load_rows = [&](const T *src) {  // both sets at once (everything but fp64), in the order of the blob
#pragma unroll
        for (int a = 0; a < RX; ++a) {
            const int ii = xv[a] ? l * RX + a : 0;
#pragma unroll
            for (int m = 0; m < NX; ++m) {
                mS1b[a][m] = xv[a] ? src[OFF_AMBKT + ii + NX * m] : T(0);
                mS1f[a][m] = xv[a] ? src[OFF_A + ii + NX * m] : T(0);
            }
#pragma unroll
            for (int j = 0; j < NU; ++j) {
                mKt[a][j] = xv[a] ? src[OFF_K + j + NU * ii] : T(0);  // Kinf^T(i,j) = Kinf(j,i)
                mB[a][j] = xv[a] ? src[OFF_B + ii + NX * j] : T(0);
            }
            vQd[a] = xv[a] ? src[OFF_QD + ii] : T(0);
            vAPf[a] = xv[a] ? src[OFF_APF + ii] : T(0);
            vf[a] = xv[a] ? src[OFF_F + ii] : T(0);
        }
#pragma unroll
        for (int b = 0; b < RU; ++b) {
            const int jj = uv[b] ? l * RU + b : 0;
#pragma unroll
            for (int m = 0; m < NX; ++m) {
                mS1b[RX + b][m] = uv[b] ? src[OFF_B + m + NX * jj] : T(0);  // B^T(j,m) = B(m,j)
                mS1f[RX + b][m] = uv[b] ? src[OFF_K + jj + NU * m] : T(0);
            }
#pragma unroll
            for (int m = 0; m < NU; ++m) mQuu[b][m] = uv[b] ? src[OFF_QUU + jj + NU * m] : T(0);
            vRd[b] = uv[b] ? src[OFF_RD + jj] : T(0);
            vBPf[b] = uv[b] ? src[OFF_BPF + jj] : T(0);
        }
    };
    // where this lane's rows come from at a sweep start (PS): the staged blob, or its slot's own blob (heterogeneous batch)
    const T *rowsrc = stage;
    if constexpr (!PS) load_rows(stage);
    // TMEM variant: warp 0 allocates all 512 columns (one CTA per SM); warps w and w+4 share a lane quarter and
    // take the column ranges [0, N*CPK) and [N*CPK, 2*N*CPK)
    unsigned tbase = 0;
    __shared__ unsigned tmem_addr_slot;
    if constexpr (TM) {
        if (warp == 0) {
            asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 512;" ::"r"((unsigned)__cvta_generic_to_shared(&tmem_addr_slot)) : "memory");
            asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
        }
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    }
    __syncthreads();  // staging area is reused as state below
    if constexpr (TM) {
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        tbase = tmem_addr_slot + ((unsigned)((warp & 3) * 32) << 16) + (unsigned)((warp >> 2) * N * CPK);
    }

    // ---- shared-memory state of this warp ----
    //   PA[k][lane][PVP] : primal pack  (vnew rows of this lane, then znew rows)      16-byte vectors,
    //   PB[k][lane][PVP] : dual pack    (g rows, then y rows)                          conflict free
    //   D [k][b][lane]   : d
    //   GB[...]          : gather scratch (one vector of one instance per row)
    //   TMEM variant: PB and D live in tensor memory instead, columns [k*CPK, +PVP) and [k*CPK+PVP, +RU) of the thread's lane
    const int warp_elems = TM ? (int)Cfg::warp_elems_tm(N) : (int)Cfg::warp_elems(N);
    // fp64 (PS): the staged blob stays in shared memory for the whole kernel, the state regions start behind it
    constexpr size_t BLOB_KEEP = PS ? (size_t)BLOB_BYTES : 0;
    T *wbase = reinterpret_cast<T *>(smem_raw + BLOB_KEEP) + (size_t)warp * warp_elems;
    T *gPA = wbase, *gPB = gPA + N * 32 * PVP, *gD = gPB + N * 32 * PVP, *gGB = TM ? gPA + N * 32 * PVP : gD + (N - 1) * RU * 32;
    const unsigned aPA = (unsigned)__cvta_generic_to_shared(gPA) + (unsigned)(lane * PVP) * ES;
    const unsigned aPB = (unsigned)__cvta_generic_to_shared(gPB) + (unsigned)(lane * PVP) * ES;
    const unsigned aD = (unsigned)__cvta_generic_to_shared(gD) + (unsigned)lane * ES;
    const unsigned aGB = (unsigned)__cvta_generic_to_shared(gGB);
    constexpr unsigned KSTR = 32u * PVP * ES;  // bytes per knot point in PA / PB
    constexpr unsigned DSTR = (unsigned)RU * 32u * ES;
    auto load_pack = [&](unsigned base, int k, T (&v)[PVP]) {
#pragma unroll
        for (int c = 0; c < NPV; ++c) {
            T t[W];
            ldsv(base + (unsigned)k * KSTR + (unsigned)(c * W) * ES, t);
#pragma unroll
            for (int e = 0; e < W; ++e) v[c * W + e] = t[e];
        }
    };
    auto store_pack = [&](unsigned base, int k, const T (&v)[PVP]) {
#pragma unroll
        for (int c = 0; c < NPV; ++c) {
            T t[W];
#pragma unroll
            for (int e = 0; e < W; ++e) t[e] = v[c * W + e];
            stsv(base + (unsigned)k * KSTR + (unsigned)(c * W) * ES, t);
        }
    };
    // dual pack / d accessors.  TMEM loads are asynchronous: `pb_ready` / `d_ready` must run before the first use.
    auto load_pb = [&](int k, T (&v)[PVP]) {
        if constexpr (TM) {
#pragma unroll
            for (int c = 0; c < NPV; ++c) {
                T t[W];
                tm_ld(tbase + (unsigned)(k * CPK + c * W * CW), t);
#pragma unroll
                for (int e = 0; e < W; ++e) v[c * W + e] = t[e];
            }
        } else {
            load_pack(aPB, k, v);
        }
    };
    auto pb_ready = [&](T (&v)[PVP]) {
        if constexpr (TM) {
            tm_wait_ld();
#pragma unroll
            for (int e = 0; e < PVP; ++e) tm_tie(v[e]);
        }
    };
    auto store_pb = [&](int k, const T (&v)[PVP]) {  // TMEM: warp-wide, unconditional
        if constexpr (TM) {
#pragma unroll
            for (int c = 0; c < NPV; ++c) {
                T t[W];
#pragma unroll
                for (int e = 0; e < W; ++e) t[e] = v[c * W + e];
                tm_st(tbase + (unsigned)(k * CPK + c * W * CW), t);
            }
        } else {
            store_pack(aPB, k, v);
        }
    };
    auto load_d = [&](int k, T (&d)[RU]) {
        if constexpr (TM) {
#pragma unroll
            for (int b = 0; b < RU; ++b) {
                T t[1];
                tm_ld(tbase + (unsigned)(k * CPK + (PVP + b) * CW), t);
                d[b] = t[0];
            }
        } else {
#pragma unroll
            for (int b = 0; b < RU; ++b) d[b] = lds(aD + (unsigned)k * DSTR + (unsigned)(b * 32) * ES, T());
        }
    };
    auto d_ready = [&](T (&d)[RU]) {
        if constexpr (TM) {
            tm_wait_ld();
#pragma unroll
            for (int b = 0; b < RU; ++b) tm_tie(d[b]);
        }
    };
    auto store_d = [&](int k, const T (&d)[RU], const bool live) {
        if constexpr (TM) {
#pragma unroll
            for (int b = 0; b < RU; ++b) {
                T t[1] = {d[b]};
                tm_st(tbase + (unsigned)(k * CPK + (PVP + b) * CW), t);
            }
        } else {
#pragma unroll
            for (int b = 0; b < RU; ++b)
                if (live && uv[b]) sts(aD + (unsigned)k * DSTR + (unsigned)(b * 32) * ES, d[b]);
        }
    };
    // all-gather inside the lane group through shared memory: every lane stores its R values, then reads the
    // whole vector with 16-byte broadcast loads (absolute row order -> ascending-k dot products as in the oracle).
    // There are three gather buffers; every call site of the sweeps owns one (BUF) such that two consecutive uses of a
    // buffer always have another gather's barrier between them: the barrier that would protect the buffer's previous
    // readers before it is overwritten (LEAD) is then unnecessary, one __syncwarp per gather instead of two.
    // (the all-shared-memory variant has no room for three buffers in its fourth warp: one buffer, both barriers)
    constexpr bool G3 = TM;
    constexpr unsigned GB0 = 0u, GB1 = G3 ? (unsigned)Cfg::GBUF1 * ES : 0u, GB2 = G3 ? 2u * (unsigned)Cfg::GBUF1 * ES : 0u;
    auto gather_x = [&](const unsigned bo, const bool LEAD, const T (&own)[RX], T (&full)[NX]) {  // always inlined with literals
        if (LEAD || !G3) __syncwarp();
#pragma unroll
        for (int a = 0; a < RX; ++a) sts(aGB + bo + (unsigned)(slot * NXP + l * RX + a) * ES, own[a]);
        __syncwarp();
#pragma unroll
        for (int c = 0; c < NXP / W; ++c) {
            T t[W];
            ldsv(aGB + bo + (unsigned)(slot * NXP + c * W) * ES, t);
#pragma unroll
            for (int e = 0; e < W; ++e)
                if (c * W + e < NX) full[c * W + e] = t[e];
        }
    };
    auto gather_u = [&](const unsigned bo, const bool LEAD, const T (&own)[RU], T (&full)[NU]) {
        if (LEAD || !G3) __syncwarp();
#pragma unroll
        for (int b = 0; b < RU; ++b) sts(aGB + bo + (unsigned)(slot * NUP + l * RU + b) * ES, own[b]);
        __syncwarp();
#pragma unroll
        for (int c = 0; c < NUP / W; ++c) {
            T t[W];
            ldsv(aGB + bo + (unsigned)(slot * NUP + c * W) * ES, t);
#pragma unroll
            for (int e = 0; e < W; ++e)
                if (c * W + e < NU) full[c * W + e] = t[e];
        }
    };

    const bool cold = P.cold != 0;
    const bool tvb = P.bounds_tv != 0;
    const bool enx = P.en_state_bound != 0, enu = P.en_input_bound != 0;
    T loX[RX], hiX[RX], loU[RU], hiU[RU];  // bounds of this lane's rows (reloaded per k only if time-varying)
    // a disabled bound (en_*_bound = 0) or a padding row is (-inf, +inf): the clamp is then the identity on every
    // non-NaN value, so it can stay unconditional in the hot loop
    const T kInf = (T)INFINITY;
#pragma unroll
    for (int a = 0; a < RX; ++a) {
        loX[a] = (enx && xv[a]) ? __ldg(P.x_min + l * RX + a) : -kInf;
        hiX[a] = (enx && xv[a]) ? __ldg(P.x_max + l * RX + a) : kInf;
    }
#pragma unroll
    for (int b = 0; b < RU; ++b) {
        loU[b] = (enu && uv[b]) ? __ldg(P.u_min + l * RU + b) : -kInf;
        hiU[b] = (enu && uv[b]) ? __ldg(P.u_max + l * RU + b) : kInf;
    }
    const bool keep_v = (P.s_v != nullptr) || (P.s_z != nullptr);
    // where element (k, row i) of instance-slot s lives inside a pack region
    auto idx_x = [&](int s, int k, int i) { return (k * 32 + s * L + i / RX) * PVP + (i % RX); };
    auto idx_u = [&](int s, int k, int j) { return (k * 32 + s * L + j / RU) * PVP + RX + (j % RU); };

    // ---- per-slot bookkeeping (identical in the L lanes of a slot) ----
    int64_t inst = -1;    // instance held by this lane's slot
    bool busy = false;    // the slot holds an unfinished instance
    bool want = true;     // the slot should try to fetch an instance
    int it = 0, solved = 0;
    T res_px = T(0), res_dx = T(0), res_pu = T(0), res_du = T(0);
    T x0o[RX], pterm[RX];
#pragma unroll
    for (int a = 0; a < RX; ++a) x0o[a] = pterm[a] = T(0);
    const T *xrefp = P.Xref + l * RX;
    const bool has_uref = P.Uref != nullptr;  // warp-uniform: keeps the loops free of divergence bookkeeping
    const T *urefp = has_uref ? P.Uref + l * RU : P.Xref;
    int64_t offx = 0, offu = 0;

    // linear cost of column k for this lane's rows (update_linear_cost, admm.cpp:266-280):
    //   q = -(xref*Qd) - rho*(vnew - g),  r = -(uref*Rd) - rho*(znew - y)
    // split in two so that the global (reference) and shared (state) loads of column k-1 are issued at the top of
    // backward step k and consumed only at its end, behind the dot-product chains: with one warp per scheduler a
    // load consumed right after issue is fully exposed (per-instance references come from L2/HBM)
    auto cost_load = [&](int k, const T *xp, const T *up, T (&xr)[RX], T (&ur)[RU], T (&pa)[PVP], T (&pb)[PVP]) {
#pragma unroll
        for (int a = 0; a < RX; ++a) xr[a] = xv[a] ? __ldg(xp + a) : T(0);
#pragma unroll
        for (int b = 0; b < RU; ++b) ur[b] = (has_uref && uv[b]) ? __ldg(up + b) : T(0);
        load_pack(aPA, k, pa);
        load_pb(k, pb);
    };
    auto cost_eval = [&](const T (&xr)[RX], const T (&ur)[RU], const T (&pa)[PVP], const T (&pb)[PVP], T (&q)[RX], T (&r)[RU]) {
        if constexpr (FAST) {
#pragma unroll
            for (int a = 0; a < RX; ++a) q[a] = nmac<FAST>(-(xr[a] * vQd[a]), rho_(), pa[a] - pb[a]);
#pragma unroll
            for (int b = 0; b < RU; ++b) r[b] = nmac<FAST>(-(ur[b] * vRd[b]), rho_(), pa[RX + b] - pb[RX + b]);
        } else {
            // the same operations on the whole pack (state rows, input rows, padding): (-(ref*W)) - rho*(pa - pb), with the
            // subtractions issued as packed pairs (fp32)
            T m[PVP], df[PVP], t[PVP], o[PVP];
#pragma unroll
            for (int e = 0; e < PVP; ++e) m[e] = T(0);
#pragma unroll
            for (int a = 0; a < RX; ++a) m[a] = -(xr[a] * vQd[a]);
#pragma unroll
            for (int b = 0; b < RU; ++b) m[RX + b] = -(ur[b] * vRd[b]);
            vsub<T, PVP>(pa, pb, df);
#pragma unroll
            for (int e = 0; e < PVP; ++e) t[e] = rho_() * df[e];
            vsub<T, PVP>(m, t, o);
#pragma unroll
            for (int a = 0; a < RX; ++a) q[a] = o[a];
#pragma unroll
            for (int b = 0; b < RU; ++b) r[b] = o[RX + b];
        }
    };

    // forward pass fused with slack / dual update / residuals.  SLOW = some slot is in the first iteration of a
    // warm start (work->v / work->z come from the caller) or work->v / work->z are being persisted.
    auto forward = [&](auto tag, const bool vin, T &rpx, T &rdx, T &rpu, T &rdu) {
        constexpr bool SLOW = decltype(tag)::value;
        if constexpr (PS) load_fwd_rows(rowsrc);
        T xo[RX], Xf[NX];
#pragma unroll
        for (int a = 0; a < RX; ++a) xo[a] = x0o[a];
        gather_x(GB1, false, xo, Xf);
        // one column: slack + dual update of this lane's rows, residual maxima; HASU = the column has inputs
        auto column = [&](int k, const bool HASU, const T (&u)[RU], const T (&vprev)[PVP], const T (&pb)[PVP]) {  // always inlined with a literal HASU
            T pa[PVP], na[PVP], nb[PVP];
            load_pack(aPA, k, pa);
#pragma unroll
            for (int e = 0; e < PVP; ++e) {
                na[e] = pa[e];
                nb[e] = pb[e];
            }
            if (tvb) {
#pragma unroll
                for (int a = 0; a < RX; ++a) {
                    loX[a] = (enx && xv[a]) ? __ldg(P.x_min + (int64_t)k * NX + l * RX + a) : loX[a];
                    hiX[a] = (enx && xv[a]) ? __ldg(P.x_max + (int64_t)k * NX + l * RX + a) : hiX[a];
                }
                if (HASU) {
#pragma unroll
                    for (int b = 0; b < RU; ++b) {
                        loU[b] = (enu && uv[b]) ? __ldg(P.u_min + (int64_t)k * NU + l * RU + b) : loU[b];
                        hiU[b] = (enu && uv[b]) ? __ldg(P.u_max + (int64_t)k * NU + l * RU + b) : hiU[b];
                    }
                }
            }
            if constexpr (FAST) {
    #pragma unroll
                for (int a = 0; a < RX; ++a) {  // vnew = clamp(x + g), g += x - vnew
                    T vo = pa[a];
                    if constexpr (SLOW) {
                        if (vin) vo = vprev[a];
                    }
                    const T v = clamp_box<FAST>(xo[a] + pb[a], loX[a], hiX[a]);
                    na[a] = v;
                    nb[a] = (pb[a] + xo[a]) - v;
                    rpx = absmax(rpx, xo[a] - v);
                    rdx = absmax(rdx, vo - v);
                }
                if (HASU) {
    #pragma unroll
                    for (int b = 0; b < RU; ++b) {
                        T zo = pa[RX + b];
                        if constexpr (SLOW) {
                            if (vin) zo = vprev[RX + b];
                        }
                        const T z = clamp_box<FAST>(u[b] + pb[RX + b], loU[b], hiU[b]);
                        na[RX + b] = z;
                        nb[RX + b] = (pb[RX + b] + u[b]) - z;
                        rpu = absmax(rpu, u[b] - z);
                        rdu = absmax(rdu, zo - z);
                    }
                }
            } else {
                // the same update on the whole pack (state rows, input rows, padding) with the additions / subtractions
                // issued as packed pairs (fp32): vnew = clamp(x + g), g' = (g + x) - vnew, residual differences
                T X[PVP], lo[PVP], hi[PVP], vo[PVP], sum[PVP], v[PVP], dg[PVP], dx[PVP], dv[PVP];
#pragma unroll
                for (int e = 0; e < PVP; ++e) {
                    X[e] = T(0);
                    lo[e] = -kInf;
                    hi[e] = kInf;
                    vo[e] = pa[e];
                    if constexpr (SLOW) {
                        if (vin) vo[e] = vprev[e];
                    }
                }
#pragma unroll
                for (int a = 0; a < RX; ++a) {
                    X[a] = xo[a];
                    lo[a] = loX[a];
                    hi[a] = hiX[a];
                }
#pragma unroll
                for (int b = 0; b < RU; ++b) {
                    X[RX + b] = u[b];
                    lo[RX + b] = loU[b];
                    hi[RX + b] = hiU[b];
                }
                vadd<T, PVP>(X, pb, sum);
#pragma unroll
                for (int e = 0; e < PVP; ++e) v[e] = (e < RX + RU) ? clamp_box<FAST || MM>(sum[e], lo[e], hi[e]) : sum[e];
                vsub<T, PVP>(sum, v, dg);
                vsub<T, PVP>(X, v, dx);
                vsub<T, PVP>(vo, v, dv);
#pragma unroll
                for (int a = 0; a < RX; ++a) {
                    na[a] = v[a];
                    nb[a] = dg[a];
                    rpx = absmax(rpx, dx[a]);
                    rdx = absmax(rdx, dv[a]);
                }
                if (HASU) {
#pragma unroll
                    for (int b = 0; b < RU; ++b) {
                        na[RX + b] = v[RX + b];
                        nb[RX + b] = dg[RX + b];
                        rpu = absmax(rpu, dx[RX + b]);
                        rdu = absmax(rdu, dv[RX + b]);
                    }
                }
            }
            if constexpr (TM) store_pb(k, nb);  // (a slot that is not busy holds no live state)
            if (busy) {
                store_pack(aPA, k, na);
                if constexpr (!TM) store_pb(k, nb);
                if constexpr (SLOW) {
                    // work->v / work->z of this iteration = the primal pack as it was before this column's update
                    // (kept in pack layout in global scratch: one 16-byte store; transposed out only if the solve converges)
                    if (P.gpi_vscratch && !vin) {
                        T *dst = P.gpi_vscratch + ((inst * N + k) * L + l) * PVP;
#pragma unroll
                        for (int c = 0; c < NPV; ++c) {
                            using V16 = typename Vec16<T>::type;
                            V16 v16;
                            T *e16 = reinterpret_cast<T *>(&v16);
#pragma unroll
                            for (int e = 0; e < W; ++e) e16[e] = pa[c * W + e];
                            reinterpret_cast<V16 *>(dst)[c] = v16;
                        }
                    }
                }
            }
        };
        auto load_vprev = [&](int k, T (&vp)[PVP]) {  // caller's work->v / work->z column (first warm iteration only)
#pragma unroll
            for (int e = 0; e < PVP; ++e) vp[e] = T(0);
            if constexpr (SLOW) {
                if (vin && P.gpi_vscratch) {
                    const T *src = P.gpi_vscratch + ((inst * N + k) * L + l) * PVP;
#pragma unroll
                    for (int c = 0; c < NPV; ++c) {
                        using V16 = typename Vec16<T>::type;
                        const V16 v16 = reinterpret_cast<const V16 *>(src)[c];
                        const T *e16 = reinterpret_cast<const T *>(&v16);
#pragma unroll
                        for (int e = 0; e < W; ++e) vp[c * W + e] = e16[e];
                    }
                }
            }
        };
        for (int k = 0; k < N - 1; ++k) {
            T u[RU], Uf[NU], t1[RX + RU], bu[RX], vprev[PVP], pbk[PVP], dk[RU];
            load_vprev(k, vprev);
            load_pb(k, pbk);
            load_d(k, dk);
            dots<FAST>(mS1f, Xf, t1);  // [A x_k ; Kinf x_k]
            d_ready(dk);
            pb_ready(pbk);
#pragma unroll
            for (int b = 0; b < RU; ++b) u[b] = (-t1[RX + b]) - dk[b];  // u_k = -(Kinf x_k) - d_k
            gather_u(GB0, false, u, Uf);
            column(k, true, u, vprev, pbk);
            dots<FAST>(mB, Uf, bu);
            {   // x_{k+1} = (A x_k + B u_k) + f
                T ax[RX], tx[RX];
#pragma unroll
                for (int a = 0; a < RX; ++a) ax[a] = t1[a];
                vadd<T, RX>(ax, bu, tx);
                vadd<T, RX>(tx, vf, xo);
            }
            gather_x(GB1, false, xo, Xf);
        }
        {
            T udummy[RU], vprev[PVP], pbk[PVP];
#pragma unroll
            for (int b = 0; b < RU; ++b) udummy[b] = T(0);
            load_vprev(N - 1, vprev);
            load_pb(N - 1, pbk);
            pb_ready(pbk);
            column(N - 1, false, udummy, vprev, pbk);
            if constexpr (TM) tm_wait_st();  // the dual packs are read back by the next backward pass / the write-back
        }
    };

    // ---- cooperative (all 32 lanes) load of instance `ib` into slot `s`: zero the slot's shared-memory state,
    // read a warm start, and set up the slot's lanes (x0 rows, terminal-cost constant, reference pointers) ----
    auto load_slot = [&](int s, int64_t ib) {
        // the slot owns L consecutive lanes (L*PVP contiguous elements = VPK 16-byte vectors) of every [k][lane][PVP]
        // row of PA and PB; d is always written before it is read and needs no initialisation
        {
            constexpr int VPK = (L * PVP * (int)sizeof(T)) / 16;  // vectors per knot point of one slot
            float4 *a4 = reinterpret_cast<float4 *>(gPA), *b4 = reinterpret_cast<float4 *>(gPB);
            constexpr int ROW4 = (32 * PVP * (int)sizeof(T)) / 16;  // vectors per knot point of the whole warp
            const float4 z4 = make_float4(0.f, 0.f, 0.f, 0.f);
            for (int e = lane; e < N * VPK; e += 32) {
                const int k = e / VPK, w = e - k * VPK;
                a4[k * ROW4 + s * VPK + w] = z4;
                if constexpr (!TM) b4[k * ROW4 + s * VPK + w] = z4;
            }
        }
        __syncwarp();
        if constexpr (TM) {
            // the dual packs live in the lanes' own TMEM columns and TMEM stores are warp-wide: read-modify-write every
            // knot point, replacing the values of slot s's lanes by zeros (cold) or the caller's g / y rows (warm start);
            // the global loads of UNR knot points are issued together, ahead of the dependent TMEM traffic
            const int64_t ox = ib * (int64_t)N * NX, ou = ib * (int64_t)(N - 1) * NU;
            const bool mine = slot == s;
            constexpr int UNR = 5;
            for (int k0 = 0; k0 < N; k0 += UNR) {
                T nv[UNR][PVP];
#pragma unroll
                for (int t = 0; t < UNR; ++t) {
                    const int k = k0 + t;
#pragma unroll
                    for (int e = 0; e < PVP; ++e) nv[t][e] = T(0);
#pragma unroll
                    for (int a = 0; a < RX; ++a)
                        nv[t][a] = (!cold && mine && k < N && xv[a] && P.s_g) ? P.s_g[ox + (int64_t)k * NX + l * RX + a] : T(0);
#pragma unroll
                    for (int b = 0; b < RU; ++b)
                        nv[t][RX + b] = (!cold && mine && k < N - 1 && uv[b] && P.s_y) ? P.s_y[ou + (int64_t)k * NU + l * RU + b] : T(0);
                }
                __syncwarp();
#pragma unroll
                for (int t = 0; t < UNR; ++t) {
                    const int k = k0 + t;
                    if (k < N) {  // warp-uniform
                        T old[PVP];
                        load_pb(k, old);
                        pb_ready(old);
#pragma unroll
                        for (int e = 0; e < PVP; ++e) old[e] = mine ? nv[t][e] : old[e];
                        store_pb(k, old);
                    }
                }
            }
            tm_wait_st();
        }
        if (!cold) {
            // warm start: the instance's vnew/g/znew/y blocks are contiguous in global memory; loads are batched four
            // deep before the dependent shared-memory stores (one warp cannot hide a load-use pair per iteration)
            const int64_t ox = ib * (int64_t)N * NX, ou = ib * (int64_t)(N - 1) * NU;
            constexpr int UNR = 4;
            for (int e0 = lane; e0 < N * NX; e0 += 32 * UNR) {
                T va[UNR], vb[UNR];
#pragma unroll
                for (int t = 0; t < UNR; ++t) {
                    const int e = e0 + 32 * t;
                    const bool ok = e < N * NX;
                    va[t] = (ok && P.s_vnew) ? P.s_vnew[ox + e] : T(0);
                    vb[t] = (!TM && ok && P.s_g) ? P.s_g[ox + e] : T(0);
                }
#pragma unroll
                for (int t = 0; t < UNR; ++t) {
                    const int e = e0 + 32 * t;
                    if (e < N * NX) {
                        const int k = e / NX, i = e - k * NX;
                        const int w = idx_x(s, k, i);
                        gPA[w] = va[t];
                        if constexpr (!TM) gPB[w] = vb[t];
                    }
                }
            }
            for (int e0 = lane; e0 < (N - 1) * NU; e0 += 32 * UNR) {
                T va[UNR], vb[UNR];
#pragma unroll
                for (int t = 0; t < UNR; ++t) {
                    const int e = e0 + 32 * t;
                    const bool ok = e < (N - 1) * NU;
                    va[t] = (ok && P.s_znew) ? P.s_znew[ou + e] : T(0);
                    vb[t] = (!TM && ok && P.s_y) ? P.s_y[ou + e] : T(0);
                }
#pragma unroll
                for (int t = 0; t < UNR; ++t) {
                    const int e = e0 + 32 * t;
                    if (e < (N - 1) * NU) {
                        const int k = e / NU, j = e - k * NU;
                        const int w = idx_u(s, k, j);
                        gPA[w] = va[t];
                        if constexpr (!TM) gPB[w] = vb[t];
                    }
                }
            }
            // work->v / work->z of the caller (only read by the first iteration's dual residual): staged into the global
            // scratch in pack layout, so that the first forward pass fetches them with one 16-byte load per knot point
            if (P.gpi_vscratch) {
                T *sc = P.gpi_vscratch + ib * (int64_t)N * L * PVP;
                for (int e0 = lane; e0 < N * NX; e0 += 32 * UNR) {
                    T va[UNR];
#pragma unroll
                    for (int t = 0; t < UNR; ++t) {
                        const int e = e0 + 32 * t;
                        va[t] = (e < N * NX && P.s_v) ? P.s_v[ox + e] : T(0);
                    }
#pragma unroll
                    for (int t = 0; t < UNR; ++t) {
                        const int e = e0 + 32 * t;
                        if (e < N * NX) {
                            const int k = e / NX, i = e - k * NX;
                            sc[(k * L + i / RX) * PVP + (i % RX)] = va[t];
                        }
                    }
                }
                for (int e0 = lane; e0 < (N - 1) * NU; e0 += 32 * UNR) {
                    T va[UNR];
#pragma unroll
                    for (int t = 0; t < UNR; ++t) {
                        const int e = e0 + 32 * t;
                        va[t] = (e < (N - 1) * NU && P.s_z) ? P.s_z[ou + e] : T(0);
                    }
#pragma unroll
                    for (int t = 0; t < UNR; ++t) {
                        const int e = e0 + 32 * t;
                        if (e < (N - 1) * NU) {
                            const int k = e / NU, j = e - k * NU;
                            sc[(k * L + j / RU) * PVP + RX + (j % RU)] = va[t];
                        }
                    }
                }
            }
            __syncwarp();
        }
        // L2 prefetch, one "generation" of tickets ahead: tickets are handed out in order, so instance ib + PF will be
        // loaded by some warp shortly; touching its per-instance inputs now turns that warp's latency-exposed loads
        // (one warp per scheduler cannot hide them) into L2 hits.  The current instance's references are touched too.
        {
            constexpr int64_t PF = 1024;
            auto touch = [&](const T *base, int64_t elems) {
                const char *pb_ = reinterpret_cast<const char *>(base);
                for (int64_t o = (int64_t)lane * 128; o < elems * (int64_t)sizeof(T); o += 32 * 128) asm volatile("prefetch.global.L2 [%0];" ::"l"(pb_ + o));
            };
            const int64_t nxN = (int64_t)N * NX, nuN = (int64_t)(N - 1) * NU;
            if (P.xref_pi) touch(P.Xref + ib * nxN, nxN);
            if (has_uref && P.uref_pi) touch(P.Uref + ib * nuN, nuN);
            const int64_t ip = ib + PF;
            if (ip < P.B) {
                if (P.xref_pi) touch(P.Xref + ip * nxN, nxN);
                if (has_uref && P.uref_pi) touch(P.Uref + ip * nuN, nuN);
                if (!cold) {
                    if (P.s_vnew) touch(P.s_vnew + ip * nxN, nxN);
                    if (P.s_g) touch(P.s_g + ip * nxN, nxN);
                    if (P.s_znew) touch(P.s_znew + ip * nuN, nuN);
                    if (P.s_y) touch(P.s_y + ip * nuN, nuN);
                    if (P.s_v && P.gpi_vscratch) touch(P.s_v + ip * nxN, nxN);
                    if (P.s_z && P.gpi_vscratch) touch(P.s_z + ip * nuN, nuN);
                }
            }
        }
        if (slot == s) {
            inst = ib;
            busy = true;
            it = 0;
            solved = 0;
            res_px = res_dx = res_pu = res_du = T(0);
            offx = ib * (int64_t)N * NX;
            offu = ib * (int64_t)(N - 1) * NU;
            xrefp = P.Xref + (P.xref_pi ? offx : 0) + l * RX;
            urefp = has_uref ? P.Uref + (P.uref_pi ? offu : 0) + l * RU : P.Xref;
            // heterogeneous batch: this instance has its own model / cache blob (same layout as the shared one, rho appended)
            const T *pinf = P.Pinf_g;
            if constexpr (HET) {
                const T *mb = P.models + ib * (int64_t)(BLOB + 1);
                if constexpr (PS) rowsrc = mb;
                else load_rows(mb);
                rho_m = mb[BLOB];
                pinf = mb + OFF_PINF;
            }
            // x0 (own rows) and the iteration-invariant part of the terminal cost: -(Pinf^T xref_{N-1})
            T xr[NX];
            const T *xl = xrefp - l * RX + (int64_t)(N - 1) * NX;
#pragma unroll
            for (int m = 0; m < NX; ++m) xr[m] = __ldg(xl + m);
#pragma unroll
            for (int a = 0; a < RX; ++a) {
                const int i = l * RX + a, ii = xv[a] ? i : 0;
                x0o[a] = xv[a] ? __ldg(P.x0 + ib * NX + ii) : T(0);
                T sacc = xr[0] * __ldg(pinf + 0 + NX * ii);
#pragma unroll
                for (int m = 1; m < NX; ++m) sacc = mac<FAST>(sacc, xr[m], __ldg(pinf + m + NX * ii));
                pterm[a] = xv[a] ? -sacc : T(0);
            }
        }
        __syncwarp();
    };

    // ---- cooperative write-back of slot `s` (instance `ib`): solution, info, optional state and rollout ----
    auto store_slot = [&](int s, int64_t ib) {
        const int s_solved = __shfl_sync(0xffffffffu, solved, s * L);
        const int s_it = __shfl_sync(0xffffffffu, it, s * L);
        if (slot == s && l == 0) {
            if (P.iter) P.iter[ib] = it;
            if (P.solved) P.solved[ib] = solved;
            if (P.residuals) {
                T *r = P.residuals + 4 * ib;
                r[0] = res_px; r[1] = res_dx; r[2] = res_pu; r[3] = res_du;
            }
        }
        __syncwarp();
        const int64_t ox = ib * (int64_t)N * NX, ou = ib * (int64_t)(N - 1) * NU;
        // solution->x = vnew, solution->u = znew; work->vnew/znew/g/y; coalesced transposing copy
        for (int e = lane; e < N * NX; e += 32) {
            const int k = e / NX, i = e - k * NX;
            const int w = idx_x(s, k, i);
            const T v = gPA[w];
            if (P.sol_x) P.sol_x[ox + e] = v;
            if (P.s_vnew) P.s_vnew[ox + e] = v;
            if constexpr (!TM)
                if (P.s_g) P.s_g[ox + e] = gPB[w];
            // work->v: previous vnew if the solve converged (staged in the scratch during the last forward pass; unchanged
            // if that was the first iteration of a warm start), else = vnew (admm.cpp:445); untouched when no iteration
            // ran on a warm start
            if (P.s_v && !s_solved && s_it > 0) P.s_v[ox + e] = v;
            else if (P.s_v && s_solved && !(s_it == 1 && !cold)) P.s_v[ox + e] = P.gpi_vscratch[((ib * N + k) * L + i / RX) * PVP + (i % RX)];
            else if (P.s_v && cold && s_it == 0) P.s_v[ox + e] = T(0);
        }
        for (int e = lane; e < (N - 1) * NU; e += 32) {
            const int k = e / NU, j = e - k * NU;
            const int w = idx_u(s, k, j);
            const T z = gPA[w];
            if (P.sol_u) P.sol_u[ou + e] = z;
            if (P.s_znew) P.s_znew[ou + e] = z;
            if constexpr (!TM)
                if (P.s_y) P.s_y[ou + e] = gPB[w];
            if (P.s_z && !s_solved && s_it > 0) P.s_z[ou + e] = z;
            else if (P.s_z && s_solved && !(s_it == 1 && !cold)) P.s_z[ou + e] = P.gpi_vscratch[((ib * N + k) * L + j / RU) * PVP + RX + (j % RU)];
            else if (P.s_z && cold && s_it == 0) P.s_z[ou + e] = T(0);
        }
        if constexpr (TM) {
            if (P.s_g || P.s_y) {  // work->g / work->y from the lanes' own TMEM columns
                __syncwarp();
                for (int k = 0; k < N; ++k) {
                    T v[PVP];
                    load_pb(k, v);
                    pb_ready(v);
                    if (slot == s) {
#pragma unroll
                        for (int a = 0; a < RX; ++a)
                            if (xv[a] && P.s_g) P.s_g[ox + (int64_t)k * NX + l * RX + a] = v[a];
                        if (k < N - 1) {
#pragma unroll
                            for (int b = 0; b < RU; ++b)
                                if (uv[b] && P.s_y) P.s_y[ou + (int64_t)k * NU + l * RU + b] = v[RX + b];
                        }
                    }
                    __syncwarp();
                }
            }
        }
        // work->u.col(0): one rollout step from d_0 (every lane computes, the lanes of slot s store)
        if constexpr (PS) {
            if (P.u0 || P.s_x || P.s_u) load_fwd_rows(rowsrc);
        }
        if (P.u0) {
            __syncwarp();
            T xo0[RX], Xf0[NX], t10[RX + RU];
#pragma unroll
            for (int a = 0; a < RX; ++a) xo0[a] = x0o[a];
            gather_x(GB1, true, xo0, Xf0);
            T d0[RU];
            load_d(0, d0);
            dots<FAST>(mS1f, Xf0, t10);
            d_ready(d0);
#pragma unroll
            for (int b = 0; b < RU; ++b) {
                T u0v = (-t10[RX + b]) - d0[b];
                if (s_it == 0) u0v = (!cold && P.s_u) ? P.s_u[ou + l * RU + b] : T(0);
                if (slot == s && uv[b]) P.u0[ib * NU + l * RU + b] = u0v;
            }
            __syncwarp();
        }
        // work->x / work->u: replay the last rollout from d and x0 (bit-identical to the last forward pass), staging it
        // in this slot's (now dead) primal pack so that the write-back is coalesced too.  Every lane executes the
        // arithmetic (the gathers are warp-wide); only the lanes of slot s store.
        if (P.s_x || P.s_u) {
            __syncwarp();
            T xo[RX], Xf[NX];
#pragma unroll
            for (int a = 0; a < RX; ++a) xo[a] = x0o[a];
            gather_x(GB1, false, xo, Xf);
            for (int k = 0; k < N; ++k) {
                T na[PVP];
#pragma unroll
                for (int e = 0; e < PVP; ++e) na[e] = T(0);
#pragma unroll
                for (int a = 0; a < RX; ++a) na[a] = xo[a];
                if (k < N - 1) {
                    T u[RU], Uf[NU], t1[RX + RU], bu[RX], dk[RU];
                    load_d(k, dk);
                    dots<FAST>(mS1f, Xf, t1);
                    d_ready(dk);
#pragma unroll
                    for (int b = 0; b < RU; ++b) {
                        u[b] = (-t1[RX + b]) - dk[b];
                        na[RX + b] = u[b];
                    }
                    gather_u(GB0, false, u, Uf);
                    dots<FAST>(mB, Uf, bu);
#pragma unroll
                    for (int a = 0; a < RX; ++a) xo[a] = (t1[a] + bu[a]) + vf[a];
                }
                if (slot == s) store_pack(aPA, k, na);
                if (k < N - 1) gather_x(GB1, true, xo, Xf);
            }
            __syncwarp();
            if (P.s_x)
                for (int e = lane; e < N * NX; e += 32) {
                    const int k = e / NX, i = e - k * NX;
                    if (s_it > 0 || k == 0) P.s_x[ox + e] = gPA[idx_x(s, k, i)];
                    else if (cold) P.s_x[ox + e] = T(0);
                }
            if (P.s_u)
                for (int e = lane; e < (N - 1) * NU; e += 32) {
                    const int k = e / NU, j = e - k * NU;
                    if (s_it > 0) P.s_u[ou + e] = gPA[idx_u(s, k, j)];
                    else if (cold) P.s_u[ou + e] = T(0);
                }
        }
        __syncwarp();
    };

    // ---- persistent loop: every slot runs its own instance; a slot that terminates (converged or max_iter) is
    // written back and refilled from the global queue immediately, so no lane group waits for the slowest
    // instance of its warp (termination is per instance, admm.cpp:310-328) ----
    for (;;) {
        // 1. retire finished slots / fill empty ones
        const bool fin = busy && (solved || it >= P.max_iter);
        const unsigned todo = __ballot_sync(0xffffffffu, (fin || (!busy && want)) && l == 0);
        for (unsigned m = todo; m; m &= m - 1) {
            const int s = (__ffs(m) - 1) / L;
            const int64_t ib_old = __shfl_sync(0xffffffffu, inst, s * L);
            const int was_busy = __shfl_sync(0xffffffffu, (int)busy, s * L);
            // the queue ticket is requested before the write-back of the finished instance so that the atomic's
            // latency hides behind it.  (Never hold a ticket in advance: measured on B200, a ticket prefetched by every
            // warp kept up to 592 instances hostage until a slot freed up and cost a whole extra wave per launch.)
            unsigned long long nxt = 0;
            if (lane == 0) nxt = atomicAdd(queue, 1ULL);
            if (was_busy) store_slot(s, ib_old);
            nxt = __shfl_sync(0xffffffffu, nxt, 0);
            if ((int64_t)nxt < P.B) {
                load_slot(s, (int64_t)nxt);
            } else if (slot == s) {
                busy = false;
                want = false;
            }
        }
        if (!__any_sync(0xffffffffu, busy)) break;
        if (__any_sync(0xffffffffu, busy && it >= P.max_iter)) continue;  // max_iter <= 0: retire without iterating
        __syncwarp();

        // 2. ADMM iterations for every busy slot until some slot terminates.  This inner loop has warp-uniform
        // control flow only, so the compiler keeps the warp converged (no divergence bookkeeping around the
        // shared-memory gathers).
        do {
        // ---- terminal cost + backward pass (update_linear_cost fused, software-pipelined by one column) ----
        if constexpr (PS) load_bwd_rows(rowsrc);
        T po[RX], Pf[NX];
        {
            T pa[PVP], pb[PVP];
            load_pack(aPA, N - 1, pa);
            load_pb(N - 1, pb);
            pb_ready(pb);
#pragma unroll
            for (int a = 0; a < RX; ++a) po[a] = nmac<FAST>(pterm[a], rho_(), pa[a] - pb[a]);
        }
        gather_x(GB1, false, po, Pf);
        T q[RX], r[RU], Rf[NU];
        const T *xp = xrefp + (int64_t)(N - 2) * NX;
        const T *up = urefp + (has_uref ? (int64_t)(N - 2) * NU : 0);
        {
            T xr[RX], ur[RU], pa[PVP], pb[PVP];
            cost_load(N - 2, xp, up, xr, ur, pa, pb);
            pb_ready(pb);
            cost_eval(xr, ur, pa, pb, q, r);
        }
        gather_u(GB2, false, r, Rf);
        // one backward step; MORE = another column follows (its cost inputs are fetched now and consumed at the end of
        // the step).  The last step (k = 0) is peeled so that the loop body carries no k > 0 predicates.
        auto bwd_step = [&](int k, const bool MORE) {  // always inlined with a literal MORE
            T xr_n[RX], ur_n[RU], pa_n[PVP], pb_n[PVP];
            if (MORE) {
                xp -= NX;
                if (has_uref) up -= NU;
                cost_load(k - 1, xp, up, xr_n, ur_n, pa_n, pb_n);
            }
            // d_k = Quu_inv ((B^T p_{k+1} + r_k) + BPf)
            T s_[RU], Sf[NU], acc1[RX + RU], kr[RX], dq[RU];
            dots<FAST>(mS1b, Pf, acc1);  // [AmBKt p_{k+1} ; B^T p_{k+1}]
#pragma unroll
            for (int b = 0; b < RU; ++b) s_[b] = (acc1[RX + b] + r[b]) + vBPf[b];
            gather_u(GB0, false, s_, Sf);
            // p_k = ((q_k + AmBKt p_{k+1}) - Kinf^T r_k) + APf
            dots<FAST>(mKt, Rf, kr);
            {
                T a1[RX], t1_[RX], t2_[RX];
#pragma unroll
                for (int a = 0; a < RX; ++a) a1[a] = acc1[a];
                vadd<T, RX>(q, a1, t1_);
                vsub<T, RX>(t1_, kr, t2_);
                vadd<T, RX>(t2_, vAPf, po);
            }
            if (MORE) gather_x(GB1, false, po, Pf);  // p_0 itself is never used (the forward pass starts from x_0)
            dots<FAST>(mQuu, Sf, dq);
            store_d(k, dq, busy);
            if (MORE) {
                pb_ready(pb_n);
                cost_eval(xr_n, ur_n, pa_n, pb_n, q, r);
                gather_u(GB2, false, r, Rf);
            }
        };
        for (int k = N - 2; k >= 1; --k) bwd_step(k, true);
        bwd_step(0, false);
        if constexpr (TM) tm_wait_st();  // d is read back by the forward pass
        __syncwarp();

        T rpx = T(0), rdx = T(0), rpu = T(0), rdu = T(0);
        const bool vin = busy && (!cold) && it == 0;  // work->v / work->z come from the caller on the first iteration
        if (keep_v || __any_sync(0xffffffffu, vin)) forward(BoolTag<true>{}, vin, rpx, rdx, rpu, rdu);
        else forward(BoolTag<false>{}, false, rpx, rdx, rpu, rdu);
        __syncwarp();
        // ---- termination_condition (admm.cpp:310-328), per instance ----
        rpx = group_max<T, L>(rpx);
        rdx = group_max<T, L>(rdx);
        rpu = group_max<T, L>(rpu);
        rdu = group_max<T, L>(rdu);
        if (busy) {
            it += 1;
            if (it % P.check_termination == 0) {
                res_px = rpx;
                res_dx = rdx * rho_();
                res_pu = rpu;
                res_du = rdu * rho_();
                if (res_px < P.pri_tol && res_pu < P.pri_tol && res_dx < P.dua_tol && res_du < P.dua_tol) solved = 1;
            }
        }
        } while (!__any_sync(0xffffffffu, busy && (solved || it >= P.max_iter)));
    }
    if constexpr (TM) {
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
        __syncthreads();
        if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 512;" ::"r"(tmem_addr_slot) : "memory");
    }
}

// ---------------------------------------------------------------------------------------------------------
// host side: plan + launch
// ---------------------------------------------------------------------------------------------------------
// TINYMPC_GPI_TMEM=0 keeps everything in shared memory (A/B switch for measurements)
inline bool gpi_allow_tm() {
    const char *e = std::getenv("TINYMPC_GPI_TMEM");
    return !(e && e[0] == '0');
}

// candidate (L, TM): replaces `best` (lanes, warps_resident, smem, tmem_cols) when it holds more; pvp = its GpiCfg::PVP
template <typename T, int NX, int NU, int L, bool TM>
inline void gpi_consider(int N, int max_smem, LaunchPlan &best, int &pvp) {
    if constexpr (gpi_feasible<T, NX, NU, L>()) {
        using Cfg = GpiCfg<NX, NU, L, (int)sizeof(T)>;
        const size_t per_warp = (TM ? Cfg::warp_elems_tm(N) : Cfg::warp_elems(N)) * sizeof(T);
        // fp32: the TMA staging area aliases the start of the state region (the allocation is at least as large as the blob);
        // fp64: the blob stays resident in front of the state regions (matrix rows are re-read at every sweep start)
        const size_t blob = ((size_t)(3 * NX * NX + 2 * NX * NU + NU * NU + 4 * NX + 2 * NU) * sizeof(T) + 15) / 16 * 16 + 64;
        const size_t keep = gpi_per_sweep_rows<T>() ? ((size_t)(3 * NX * NX + 2 * NX * NU + NU * NU + 4 * NX + 2 * NU) * sizeof(T) + 15) / 16 * 16 : 0;
        if ((size_t)max_smem < keep + per_warp) return;
        int w = (int)std::min<size_t>(GPI_MAX_WARPS, ((size_t)max_smem - keep) / per_warp);
        if (TM) {
            // every TMEM lane quarter is shared by the warps w, w+4, ...: 512 columns / (N*CPK columns per warp)
            const int cols = Cfg::tm_cols(N);
            if (cols > 512) return;
            w = std::min(w, 4 * (512 / cols));
        }
        if (w < 1 || blob > (size_t)max_smem) return;
        // score: instances resident per SM, then fewer lanes per instance (less shuffle traffic)
        const int inst = w * Cfg::IPW, binst = best.warps_resident * (best.lanes ? 32 / best.lanes : 0);
        const bool better = best.lanes == 0 || (w >= 4 && best.warps_resident < 4) ||
                            (((w >= 4) == (best.warps_resident >= 4)) && inst > binst);
        if (better) {
            best.lanes = L;
            best.warps_resident = w;
            best.smem = std::max(keep + per_warp * (size_t)w, blob);
            best.tmem_cols = TM ? 512 : 0;  // the kernel allocates all of them
            pvp = Cfg::PVP;
        }
    }
}

template <typename T, int NX, int NU>
inline LaunchPlan gpi_plan(const LaunchDesc &d) {
    LaunchPlan p;
    int pvp = 0;
    const int N = d.N, max_smem = d.smem_budget;
    // L = 16 is only ever needed in fp64 (two registers per matrix entry: L = 4 / 8 exceed the register ceiling from
    // nx = 12 on); for fp32 L = 8 covers every (nx, nu) pair of TM_DIMS, so the fp32 L = 16 kernels are compiled only
    // with -DTM_GPI_L16 (wider states) to keep the build short
    constexpr bool L16 = sizeof(T) == 8
#ifdef TM_GPI_L16
                         || true
#endif
        ;
    // TINYMPC_GPI_LANES=4|8|16 restricts the choice to one group width (A/B switch for measurements)
    const char *e = std::getenv("TINYMPC_GPI_LANES");
    const int only = e ? std::atoi(e) : 0;
    if (!only || only == 4) gpi_consider<T, NX, NU, 4, false>(N, max_smem, p, pvp);
    if (!only || only == 8) gpi_consider<T, NX, NU, 8, false>(N, max_smem, p, pvp);
    if constexpr (L16)
        if (!only || only == 16) gpi_consider<T, NX, NU, 16, false>(N, max_smem, p, pvp);
    if (gpi_allow_tm()) {  // taken only when it holds more instances per SM
        if (!only || only == 4) gpi_consider<T, NX, NU, 4, true>(N, max_smem, p, pvp);
        if (!only || only == 8) gpi_consider<T, NX, NU, 8, true>(N, max_smem, p, pvp);
        if constexpr (L16)
            if (!only || only == 16) gpi_consider<T, NX, NU, 16, true>(N, max_smem, p, pvp);
    }
    if (p.lanes == 0) return p;
    p.family = TINYMPC_KERNEL_GPI;
    p.instances_per_cta = p.warps_resident * (32 / p.lanes);
    const int64_t ngroups = (d.io.B + (32 / p.lanes) - 1) / (32 / p.lanes);
    // ngroups = warps the batch fills.  A batch smaller than one wave is spread over all SMs with fewer warps per CTA
    // (the kernel's carve-up is per warp, any block size up to warps_resident works): the latency of a solve is set by how
    // many warps share a scheduler (C2: 2.08 ms per 100 iterations with 8 warps per SM, 1.34 ms with one).
    int warps = p.warps_resident;
    if ((ngroups + warps - 1) / warps < d.sm_count) warps = (int)std::max<int64_t>(1, (ngroups + d.sm_count - 1) / d.sm_count);
    const int64_t want = (ngroups + warps - 1) / warps;
    p.ctas = (int)std::max<int64_t>(1, std::min<int64_t>(d.sm_count, want));
    p.threads = warps * 32;
    // work->v / work->z persistence: the previous-iteration slacks are staged in pack layout, one 16-byte store per knot point
    if (d.io.state.v || d.io.state.z) p.scratch_bytes = (size_t)d.io.B * N * p.lanes * pvp * sizeof(T) + 256;
    return p;
}

template <typename T, int NX, int NU, int L, bool FAST, bool HET, bool TM, bool MM = false>
int launch_gpi_L(LaunchDesc *d, const LaunchPlan &plan, const KParams<T, NX, NU> &P, const T *gmat) {
    if constexpr (gpi_feasible<T, NX, NU, L>()) {
        auto kern = gpi_solve_kernel<T, NX, NU, L, FAST, HET, TM, MM>;
        if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)plan.smem) != cudaSuccess)
            return TINYMPC_ERR_CUDA;
        kern<<<plan.ctas, plan.threads, plan.smem, d->stream>>>(P, gmat, (unsigned long long *)d->work_queue);
        return cudaGetLastError() == cudaSuccess ? TINYMPC_OK : TINYMPC_ERR_CUDA;
    } else {
        return TINYMPC_ERR_UNSUPPORTED;
    }
}

}  // namespace tmpc
