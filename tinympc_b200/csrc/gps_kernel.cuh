// gps_kernel.cuh — lane-group-per-instance batched ADMM solve with the N-indexed state STREAMED through a per-slot
// workspace in global memory (L2 / HBM) behind a ring of record images in shared memory filled by TMA bulk copies ("GPS").
//
// Same lane mapping as the on-chip kernel (gpi_kernel.cuh): L lanes form a group, lane l owns the state rows
// [l*RX, (l+1)*RX) and the input rows [l*RU, (l+1)*RU); its rows of AmBKt / B^T / A / Kinf / Kinf^T / B / Quu_inv live
// in registers (staged once per CTA by a TMA bulk copy), every mat-vec is RX+RU ascending-k dot products per lane and
// the fresh vector is all-gathered inside the lane group through shared memory.  What differs:
//   * every constraint family of the reference is covered: box (admm.cpp:85-98), second-order cones (project_soc,
//     admm.cpp:39-60,102-135), static and time-varying hyperplanes (admm.cpp:70-73,138-211) with their cost / dual
//     twins (admm.cpp:228-255,268-303), in fp32 and fp64.  FAM (template) = bit mask of the families compiled in
//     (1 cones, 2 static hyperplanes, 4 time-varying hyperplanes);
//   * a lane group runs NI (1 or 2) instances at once on the SAME matrix registers: two independent dependency chains
//     per thread.  The sweeps are recurrences of dependent fp64 / fp32 operations and registers cap the kernel at 8
//     warps per SM, so instruction-level parallelism is what hides the arithmetic latency (ncu, rocket landing fp64 with
//     one instance per group: 1.8 `wait` stalls per issued instruction, issue slots 39 % busy);
//   * the per-instance state does not have to fit on chip (rocket landing, N = 100, fp64: 31 KB per instance): it lives
//     in a workspace indexed by RESIDENT SLOT (not by instance), one record per (warp, knot point) laid out
//     [field][slot of the warp][row].  A sweep step needs one contiguous block of the record, which ONE TMA bulk copy
//     (cp.async.bulk, issued by lane 0, completion on a per-stage mbarrier) brings into a ring of record images several
//     steps ahead of its use (GpsRing); every lane reads its own rows from the image and writes results back with
//     predicated vector stores.  fence.proxy.async.global + __syncwarp at each sweep start order a sweep's stores before
//     the next sweep's bulk copies; within a sweep a stage is only overwritten after a gather barrier that follows its last
//     read.  Reference rows come straight into registers (ld.global.nc) behind an L2 prefetch;
//   * the linear cost of the NEXT iteration (q_k, r_k, p_{N-1}; update_linear_cost, admm.cpp:262-304) is evaluated
//     in the forward sweep, where the fresh slack / dual values are in registers, and stored: the backward sweep
//     reads q, r (nx+nu values per knot point) instead of every slack / dual pair (up to 8 (nx+nu));
//   * the cone projections of a knot point (state and input cones of the NI instances of a group) are work items spread
//     over the lanes of the group — every lane projects a different cone (branch-free project_soc) instead of all L
//     lanes repeating the same one — and are applied one after the other through shared memory, exactly like the
//     reference's in-place loop (admm.cpp:115-121), so overlapping cones are fine.
// The kernel is persistent (one CTA per SM); slots are refilled from a global atomic queue as instances terminate
// (per-instance termination, admm.cpp:310-328).  Reference semantics: tiny_solve -> solve (admm.cpp:331-455).
#pragma once
#include "tpi_kernel.cuh"
#include "gpi_kernel.cuh"

namespace tmpc {

__host__ __device__ constexpr int gps_gcd(int a, int b) { return b == 0 ? a : gps_gcd(b, a % b); }
__host__ __device__ constexpr int gps_popc(int m) { return (m & 1) + ((m >> 1) & 1) + ((m >> 2) & 1); }

template <int NX, int NU, int L, int ES, int NI, int FAM>
struct GpsCfg {
    static constexpr int RX = (NX + L - 1) / L;
    static constexpr int RU = (NU + L - 1) / L;
    static constexpr int IPW = 32 / L;    // lane groups per warp
    static constexpr int SPW = IPW * NI;  // instances (slots) per warp; slot index = j * IPW + group
    static constexpr int W = 16 / ES;
    static constexpr int NXP = (L * RX + W - 1) / W * W;
    static constexpr int NUP = (L * RU + W - 1) / W * W;
    static constexpr int GBX = SPW * NXP, GBU = SPW * NUP;  // gather scratch (elements): state vectors, input vectors
    // chunk sizes (bytes) of a lane's piece: global side (limited by the row pitch of an instance) and shared side
    static constexpr int CX = gps_gcd(16, gps_gcd(NX * ES, RX * ES));
    static constexpr int CU = gps_gcd(16, gps_gcd(NU * ES, RU * ES));
    static constexpr int SX = gps_gcd(16, RX * ES);
    static constexpr int SU = gps_gcd(16, RU * ES);
    static constexpr int NF = gps_popc(FAM);
    // matrix rows a lane holds in registers during one sweep (elements): forward A, Kinf, B, Qd, f, Rd; backward AmBKt,
    // B^T, Kinf^T, Quu_inv, APf, BPf
    static constexpr int FWD_ROWS = (RX + RU) * NX + RX * NU + 2 * RX + RU;
    static constexpr int BWD_ROWS = (RX + RU) * NX + RX * NU + RU * NU + RX + RU;
    static constexpr int SWEEP_REGS = (FWD_ROWS > BWD_ROWS ? FWD_ROWS : BWD_ROWS) * (ES / 4);
    static constexpr bool ok = (NX % RX == 0) && (NU % RU == 0) && SWEEP_REGS <= 112;
    static constexpr int PARK_BYTES = 32 * NI * 2 * RX * ES;  // per-lane x0 rows and terminal-cost rows (kept out of registers)
};

// Record layout: one record per (warp, knot point), every field [slot of the warp][row] padded to 16 bytes.  Region A is
// what the sweeps stream; region B (previous box slacks for work->v / work->z, family slacks) exists only when the caller
// wants those arrays back.  All offsets are compile-time, so that every access is [running pointer + immediate].
template <int NX, int NU, int SPW, int ES, int FAM>
struct GpsRec {
    __host__ __device__ static constexpr int fe(int rows) { return (SPW * rows * ES + 15) / 16 * 16 / ES; }  // elements of one field
    static constexpr int FXE = fe(NX), FUE = fe(NU), NF = gps_popc(FAM);
    __host__ __device__ static constexpr int fslot(int f) { return gps_popc(FAM & ((1 << f) - 1)); }
    static constexpr int d = 0, vnew = d + FUE, g = vnew + FXE, gf0 = g + FXE, znew = gf0 + NF * FXE, y = znew + FUE,
                         yf0 = y + FUE, q = yf0 + NF * FUE, r = q + FXE, recA = r + FUE;
    __host__ __device__ static constexpr int gf(int f) { return gf0 + fslot(f) * FXE; }
    __host__ __device__ static constexpr int yf(int f) { return yf0 + fslot(f) * FUE; }
    static constexpr int vprev = 0, zprev = vprev + FXE, vf0 = zprev + FUE, zf0 = vf0 + NF * FXE, recB = zf0 + NF * FUE;
    __host__ __device__ static constexpr int vf(int f) { return vf0 + fslot(f) * FXE; }
    __host__ __device__ static constexpr int zf(int f) { return zf0 + fslot(f) * FUE; }
};

constexpr int GPS_STAGES = 4;              // forward-sweep ring stages
constexpr int GPS_DIST = GPS_STAGES - 1;   // prefetch distance (sweep steps)

// Ring geometry.  A sweep step of a warp needs ONE contiguous block of its record: the forward sweep everything in front of
// q (d | vnew | g | family duals | znew | y | family duals), the backward sweep q | r.  The block is brought into shared
// memory as an image of the record by a single TMA bulk copy (cp.async.bulk, issued by one lane, completion on an mbarrier):
// no per-lane copy instructions and none of their traffic on the LSU / shared-memory data pipe (the per-lane cp.async
// version spent 41 % of the kernel's shared-memory wavefronts on them, ncu).  The reference columns of a step are not part
// of the record: every lane loads its own rows straight into registers (ld.global.nc) at the top of the step, behind an L2
// prefetch issued D steps earlier (staging them per lane through shared memory cost another 17 % of the wavefronts).
template <int NX, int NU, int L, int ES, int NI, int FAM>
struct GpsRing {
    using Cfg = GpsCfg<NX, NU, L, ES, NI, FAM>;
    using REC = GpsRec<NX, NU, Cfg::SPW, ES, FAM>;
    static constexpr int IMGF = REC::q * ES;                   // forward image (bytes, a multiple of 16)
    static constexpr int IMGB = (REC::recA - REC::q) * ES;     // backward image: q | r
    static constexpr int STAGE = IMGF;
    static constexpr int S = GPS_STAGES, D = GPS_DIST;
    static constexpr int RING = S * STAGE;
    static constexpr int BS = (RING / IMGB) < 8 ? (RING / IMGB) : 8;  // backward stages cut from the same memory
    static constexpr int DB = BS - 1 < 6 ? BS - 1 : 6;                // backward prefetch distance
    static constexpr int NBAR = S > BS ? S : BS;
    static constexpr size_t WARP_BYTES = (size_t)(Cfg::GBX + Cfg::GBU) * ES + (size_t)Cfg::PARK_BYTES + (size_t)RING + (size_t)((NBAR * 8 + 15) / 16 * 16);
    static constexpr size_t ZERO_BYTES = (size_t)IMGF;  // per CTA: what padding lanes read instead of a record image
    static_assert(IMGF % 16 == 0 && IMGB % 16 == 0 && STAGE % 16 == 0, "bulk copies move multiples of 16 bytes");
    static_assert(BS >= 2, "ring too small for the backward sweep");
};

// smallest lane-group width whose matrix rows fit in registers (0 = none)
template <typename T, int NX, int NU>
constexpr int gps_pick_L() {
    if (GpsCfg<NX, NU, 4, (int)sizeof(T), 1, 0>::ok) return 4;
    if (GpsCfg<NX, NU, 8, (int)sizeof(T), 1, 0>::ok) return 8;
    if (GpsCfg<NX, NU, 16, (int)sizeof(T), 1, 0>::ok) return 16;
    return 0;
}
// instances per lane group: two when the matrix rows leave room for a second set of working registers
template <typename T, int NX, int NU, int L>
constexpr int gps_pick_NI() {
    return GpsCfg<NX, NU, L, (int)sizeof(T), 1, 0>::SWEEP_REGS <= 72 ? 2 : 1;
}

// warps per CTA: one instance per lane group leaves room for twice the warps of the two-instance variant (registers)
__host__ __device__ constexpr int gps_max_warps(int NI) { return NI == 1 ? 14 : 8; }

// predicated read-only global loads of a lane's rows into registers (pr == 0: the registers keep their zeros) and L2 prefetch
__device__ __forceinline__ void ldg_chunk(const float *p, float (&v)[1], unsigned pr) {
    asm volatile("{\n .reg .pred q;\n setp.ne.u32 q, %2, 0;\n @q ld.global.nc.f32 %0, [%1];\n}" : "+f"(v[0]) : "l"(p), "r"(pr));
}
__device__ __forceinline__ void ldg_chunk(const float *p, float (&v)[2], unsigned pr) {
    asm volatile("{\n .reg .pred q;\n setp.ne.u32 q, %3, 0;\n @q ld.global.nc.v2.f32 {%0,%1}, [%2];\n}" : "+f"(v[0]), "+f"(v[1]) : "l"(p), "r"(pr));
}
__device__ __forceinline__ void ldg_chunk(const float *p, float (&v)[4], unsigned pr) {
    asm volatile("{\n .reg .pred q;\n setp.ne.u32 q, %5, 0;\n @q ld.global.nc.v4.f32 {%0,%1,%2,%3}, [%4];\n}"
                 : "+f"(v[0]), "+f"(v[1]), "+f"(v[2]), "+f"(v[3])
                 : "l"(p), "r"(pr));
}
__device__ __forceinline__ void ldg_chunk(const double *p, double (&v)[1], unsigned pr) {
    asm volatile("{\n .reg .pred q;\n setp.ne.u32 q, %2, 0;\n @q ld.global.nc.f64 %0, [%1];\n}" : "+d"(v[0]) : "l"(p), "r"(pr));
}
__device__ __forceinline__ void ldg_chunk(const double *p, double (&v)[2], unsigned pr) {
    asm volatile("{\n .reg .pred q;\n setp.ne.u32 q, %3, 0;\n @q ld.global.nc.v2.f64 {%0,%1}, [%2];\n}" : "+d"(v[0]), "+d"(v[1]) : "l"(p), "r"(pr));
}
template <typename T, int R, int CB>
__device__ __forceinline__ void ldg_piece(const T *p, T (&v)[R], unsigned pr) {
    constexpr int E = CB / (int)sizeof(T);
#pragma unroll
    for (int c = 0; c < R / E; ++c) {
        T t[E];
#pragma unroll
        for (int e = 0; e < E; ++e) t[e] = T(0);
        ldg_chunk(p + c * E, t, pr);
#pragma unroll
        for (int e = 0; e < E; ++e) v[c * E + e] = t[e];
    }
}
__device__ __forceinline__ void prefetch_l2(const void *p, unsigned pr) {
    asm volatile("{\n .reg .pred q;\n setp.ne.u32 q, %1, 0;\n @q prefetch.global.L2 [%0];\n}" ::"l"(p), "r"(pr));
}

// ---- chunked piece moves between registers and shared / global memory ----
__device__ __forceinline__ void lds_chunk(unsigned a, float (&v)[1]) { v[0] = lds(a, 0.f); }
__device__ __forceinline__ void lds_chunk(unsigned a, float (&v)[2]) {
    asm volatile("ld.shared.v2.f32 {%0,%1}, [%2];" : "=f"(v[0]), "=f"(v[1]) : "r"(a));
}
__device__ __forceinline__ void lds_chunk(unsigned a, float (&v)[4]) { ldsv(a, v); }
__device__ __forceinline__ void lds_chunk(unsigned a, double (&v)[1]) { v[0] = lds(a, 0.0); }
__device__ __forceinline__ void lds_chunk(unsigned a, double (&v)[2]) { ldsv(a, v); }
__device__ __forceinline__ void sts_chunk(unsigned a, const float (&v)[1]) { sts(a, v[0]); }
__device__ __forceinline__ void sts_chunk(unsigned a, const float (&v)[2]) {
    asm volatile("st.shared.v2.f32 [%0], {%1,%2};" ::"r"(a), "f"(v[0]), "f"(v[1]) : "memory");
}
__device__ __forceinline__ void sts_chunk(unsigned a, const float (&v)[4]) { stsv(a, v); }
__device__ __forceinline__ void sts_chunk(unsigned a, const double (&v)[1]) { sts(a, v[0]); }
__device__ __forceinline__ void sts_chunk(unsigned a, const double (&v)[2]) { stsv(a, v); }
__device__ __forceinline__ void stg_chunk(float *p, const float (&v)[1]) { *p = v[0]; }
__device__ __forceinline__ void stg_chunk(float *p, const float (&v)[2]) { *reinterpret_cast<float2 *>(p) = make_float2(v[0], v[1]); }
__device__ __forceinline__ void stg_chunk(float *p, const float (&v)[4]) { *reinterpret_cast<float4 *>(p) = make_float4(v[0], v[1], v[2], v[3]); }
__device__ __forceinline__ void stg_chunk(double *p, const double (&v)[1]) { *p = v[0]; }
__device__ __forceinline__ void stg_chunk(double *p, const double (&v)[2]) { *reinterpret_cast<double2 *>(p) = make_double2(v[0], v[1]); }
// predicated stores: one PTX predicate instead of a branch around the store (lanes that own only padding rows skip theirs)
__device__ __forceinline__ void stg_chunk(float *p, const float (&v)[1], unsigned pr) {
    asm volatile("{\n .reg .pred q;\n setp.ne.u32 q, %2, 0;\n @q st.global.f32 [%0], %1;\n}" ::"l"(p), "f"(v[0]), "r"(pr) : "memory");
}
__device__ __forceinline__ void stg_chunk(float *p, const float (&v)[2], unsigned pr) {
    asm volatile("{\n .reg .pred q;\n setp.ne.u32 q, %3, 0;\n @q st.global.v2.f32 [%0], {%1,%2};\n}" ::"l"(p), "f"(v[0]), "f"(v[1]), "r"(pr) : "memory");
}
__device__ __forceinline__ void stg_chunk(float *p, const float (&v)[4], unsigned pr) {
    asm volatile("{\n .reg .pred q;\n setp.ne.u32 q, %5, 0;\n @q st.global.v4.f32 [%0], {%1,%2,%3,%4};\n}" ::"l"(p), "f"(v[0]), "f"(v[1]), "f"(v[2]),
                 "f"(v[3]), "r"(pr)
                 : "memory");
}
__device__ __forceinline__ void stg_chunk(double *p, const double (&v)[1], unsigned pr) {
    asm volatile("{\n .reg .pred q;\n setp.ne.u32 q, %2, 0;\n @q st.global.f64 [%0], %1;\n}" ::"l"(p), "d"(v[0]), "r"(pr) : "memory");
}
__device__ __forceinline__ void stg_chunk(double *p, const double (&v)[2], unsigned pr) {
    asm volatile("{\n .reg .pred q;\n setp.ne.u32 q, %3, 0;\n @q st.global.v2.f64 [%0], {%1,%2};\n}" ::"l"(p), "d"(v[0]), "d"(v[1]), "r"(pr) : "memory");
}

template <typename T, int R, int CB>
__device__ __forceinline__ void lds_piece(unsigned a, T (&v)[R]) {
    constexpr int E = CB / (int)sizeof(T);
#pragma unroll
    for (int c = 0; c < R / E; ++c) {
        T t[E];
        lds_chunk(a + (unsigned)(c * CB), t);
#pragma unroll
        for (int e = 0; e < E; ++e) v[c * E + e] = t[e];
    }
}
template <typename T, int R, int CB>
__device__ __forceinline__ void sts_piece(unsigned a, const T (&v)[R]) {
    constexpr int E = CB / (int)sizeof(T);
#pragma unroll
    for (int c = 0; c < R / E; ++c) {
        T t[E];
#pragma unroll
        for (int e = 0; e < E; ++e) t[e] = v[c * E + e];
        sts_chunk(a + (unsigned)(c * CB), t);
    }
}
template <typename T, int R, int CB>
__device__ __forceinline__ void stg_piece(T *p, const T (&v)[R]) {
    constexpr int E = CB / (int)sizeof(T);
#pragma unroll
    for (int c = 0; c < R / E; ++c) {
        T t[E];
#pragma unroll
        for (int e = 0; e < E; ++e) t[e] = v[c * E + e];
        stg_chunk(p + c * E, t);
    }
}
template <typename T, int R, int CB>
__device__ __forceinline__ void stg_piece(T *p, const T (&v)[R], unsigned pr) {
    constexpr int E = CB / (int)sizeof(T);
#pragma unroll
    for (int c = 0; c < R / E; ++c) {
        T t[E];
#pragma unroll
        for (int e = 0; e < E; ++e) t[e] = v[c * E + e];
        stg_chunk(p + c * E, t, pr);
    }
}

// own rows of a vector every lane of the group holds in full: out[a] = full[l*R + a] without dynamic register indexing
template <typename T, int NE, int R, int L>
__device__ __forceinline__ void extract_own(const T (&full)[NE], int l, T (&out)[R]) {
#pragma unroll
    for (int a = 0; a < R; ++a) {
        T v = T(0);
#pragma unroll
        for (int g = 0; g < L; ++g)
            if (g * R + a < NE) v = (l == g) ? full[g * R + a] : v;
        out[a] = v;
    }
}

template <int J>
struct IdxTag {
    static constexpr int value = J;
};

template <typename T, int NX, int NU, int L, int NI, int FAM, bool FAST>
__global__ void __launch_bounds__(gps_max_warps(NI) * 32, 1)
    gps_solve_kernel(const __grid_constant__ KParams<T, NX, NU> P, const T *__restrict__ gmat, unsigned long long *queue) {
    using Cfg = GpsCfg<NX, NU, L, (int)sizeof(T), NI, FAM>;
    using REC = GpsRec<NX, NU, Cfg::SPW, (int)sizeof(T), FAM>;
    constexpr int RX = Cfg::RX, RU = Cfg::RU, IPW = Cfg::IPW, W = Cfg::W, NXP = Cfg::NXP, NUP = Cfg::NUP;
    using RING = GpsRing<NX, NU, L, (int)sizeof(T), NI, FAM>;
    constexpr int D = RING::D, S = RING::S, recA = REC::recA, recB = REC::recB;
    constexpr int JX = IPW * NX, JU = IPW * NU;  // element distance between the two instances of a group inside a field
    constexpr int CX = Cfg::CX, CU = Cfg::CU, SX = Cfg::SX, SU = Cfg::SU;
    constexpr unsigned ES = (unsigned)sizeof(T);
    constexpr unsigned STAGE = RING::STAGE, IMGF = RING::IMGF, IMGB = RING::IMGB;
    constexpr bool EXT = FAM != 0;
    static_assert(Cfg::ok, "lane mapping not available for this shape");
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int N = P.N;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
    const int l = lane % L, grp = lane / L;
    const bool has_b = P.gps.has_b != 0;
    const T rho = P.rho;

    // ---- stage the cache blob into shared memory with one TMA bulk copy per CTA, pull this lane's rows into registers
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
    const bool xvl = l * RX < NX, uvl = l * RU < NU;  // does this lane own real rows (else padding rows: zeros)
    const unsigned pxv = xvl ? 1u : 0u, puv = uvl ? 1u : 0u;  // the same as PTX predicate sources (predicated copies / stores)
    // The staged blob stays in shared memory for the whole kernel.  A sweep only needs half of the matrices (forward:
    // A, Kinf, B; backward: AmBKt, B^T, Kinf^T, Quu_inv), so each sweep pulls this lane's rows of ITS matrices into
    // registers when it starts: about half the register footprint of keeping everything resident, which is what makes
    // room for the second instance per lane group.
    const unsigned aBlob = (unsigned)__cvta_generic_to_shared(stage);
    auto bl = [&](int idx) { return lds(aBlob + (unsigned)idx * ES, T()); };
    auto load_fwd_rows = [&](T (&mS1f)[RX + RU][NX], T (&mB)[RX][NU], T (&vQd)[RX], T (&vf)[RX], T (&vRd)[RU]) {
#pragma unroll
        for (int a = 0; a < RX; ++a) {
            const int ii = xvl ? l * RX + a : 0;
#pragma unroll
            for (int m = 0; m < NX; ++m) mS1f[a][m] = xvl ? bl(OFF_A + ii + NX * m) : T(0);
#pragma unroll
            for (int j = 0; j < NU; ++j) mB[a][j] = xvl ? bl(OFF_B + ii + NX * j) : T(0);
            vQd[a] = xvl ? bl(OFF_QD + ii) : T(0);
            vf[a] = xvl ? bl(OFF_F + ii) : T(0);
        }
#pragma unroll
        for (int b = 0; b < RU; ++b) {
            const int jj = uvl ? l * RU + b : 0;
#pragma unroll
            for (int m = 0; m < NX; ++m) mS1f[RX + b][m] = uvl ? bl(OFF_K + jj + NU * m) : T(0);
            vRd[b] = uvl ? bl(OFF_RD + jj) : T(0);
        }
    };
    auto load_bwd_rows = [&](T (&mS1b)[RX + RU][NX], T (&mKt)[RX][NU], T (&mQuu)[RU][NU], T (&vAPf)[RX], T (&vBPf)[RU]) {
#pragma unroll
        for (int a = 0; a < RX; ++a) {
            const int ii = xvl ? l * RX + a : 0;
#pragma unroll
            for (int m = 0; m < NX; ++m) mS1b[a][m] = xvl ? bl(OFF_AMBKT + ii + NX * m) : T(0);
#pragma unroll
            for (int j = 0; j < NU; ++j) mKt[a][j] = xvl ? bl(OFF_K + j + NU * ii) : T(0);  // Kinf^T(i,j) = Kinf(j,i)
            vAPf[a] = xvl ? bl(OFF_APF + ii) : T(0);
        }
#pragma unroll
        for (int b = 0; b < RU; ++b) {
            const int jj = uvl ? l * RU + b : 0;
#pragma unroll
            for (int m = 0; m < NX; ++m) mS1b[RX + b][m] = uvl ? bl(OFF_B + m + NX * jj) : T(0);  // B^T(j,m) = B(m,j)
#pragma unroll
            for (int m = 0; m < NU; ++m) mQuu[b][m] = uvl ? bl(OFF_QUU + jj + NU * m) : T(0);
            vBPf[b] = uvl ? bl(OFF_BPF + jj) : T(0);
        }
    };

    // ---- shared memory of this warp: gather scratch (state vectors | input vectors) + parked rows + ring of record images + mbarriers ----
    constexpr unsigned wbytes = (unsigned)RING::WARP_BYTES;
    const unsigned aZero = aBlob + BLOB_BYTES;  // IMGF bytes of zeros (per CTA)
    const unsigned aGX = aZero + (unsigned)RING::ZERO_BYTES + (unsigned)warp * wbytes;
    const unsigned aGU = aGX + (unsigned)Cfg::GBX * ES;
    const unsigned aPark = aGU + (unsigned)Cfg::GBU * ES + (unsigned)lane * (NI * 2 * RX) * ES;  // [j][x0 rows | pterm rows]
    const unsigned aRing = aGU + (unsigned)Cfg::GBU * ES + (unsigned)Cfg::PARK_BYTES;
    const unsigned aBar = aRing + (unsigned)RING::RING;  // NBAR mbarriers of this warp
    // this lane's rows inside a state-shaped / input-shaped field of a record image (first instance of the group)
    const unsigned lxo = (unsigned)(grp * NX + l * RX) * ES, luo = (unsigned)(grp * NU + l * RU) * ES;
    // the CTA's zero image: what padding lanes read instead of a record image, so that their arithmetic stays finite and
    // never reaches a residual
    for (unsigned o = (unsigned)threadIdx.x * 16u; o < (unsigned)RING::ZERO_BYTES; o += (unsigned)blockDim.x * 16u)
        asm volatile("st.shared.v4.f32 [%0], {%1,%1,%1,%1};" ::"r"(aZero + o), "f"(0.f) : "memory");
    if (lane == 0) {
#pragma unroll
        for (int b = 0; b < RING::NBAR; ++b) asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(aBar + 8u * b));
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    unsigned phase = 0;  // bit b = parity the next wait on barrier b expects (warp-uniform)
    // one bulk copy of `bytes` from `src` (global) to `dst` (shared), completion on barrier b; lane 0 issues
    auto bulk_load = [&](unsigned dst, const T *src, unsigned bytes, int b) {
        if (lane == 0) {
            const unsigned mb = aBar + 8u * (unsigned)b;
            asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(mb), "r"(bytes) : "memory");
            asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst), "l"(src),
                         "r"(bytes), "r"(mb)
                         : "memory");
        }
    };
    auto bulk_wait = [&](int b) {
        const unsigned mb = aBar + 8u * (unsigned)b, par = (phase >> b) & 1u;
        unsigned done = 0;
        while (!done) {
            asm volatile("{\n .reg .pred p;\n mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n selp.u32 %0, 1, 0, p;\n}\n"
                         : "=r"(done)
                         : "r"(mb), "r"(par)
                         : "memory");
        }
        phase ^= 1u << b;
    };
    // the records are written with ordinary stores (all lanes) and read back by bulk copies (async proxy): every lane orders
    // its stores before later async-proxy operations, the warp converges, then lane 0 may issue copies
    auto sweep_fence = [&]() {
        asm volatile("fence.proxy.async.global;" ::: "memory");
        __syncwarp();
    };
    // gather scratch of instance j of this lane's group (slot j*IPW + grp): own rows / whole vector
    const unsigned gxf0 = aGX + (unsigned)(grp * NXP) * ES, gxo0 = gxf0 + (unsigned)(l * RX) * ES;
    const unsigned guf0 = aGU + (unsigned)(grp * NUP) * ES, guo0 = guf0 + (unsigned)(l * RU) * ES;
    auto gxo = [&](int j) { return gxo0 + (unsigned)(j * IPW * NXP) * ES; };
    auto gxf = [&](int j) { return gxf0 + (unsigned)(j * IPW * NXP) * ES; };
    auto guo = [&](int j) { return guo0 + (unsigned)(j * IPW * NUP) * ES; };
    auto guf = [&](int j) { return guf0 + (unsigned)(j * IPW * NUP) * ES; };

    auto gather_x = [&](const T (&own)[NI][RX], T (&full)[NI][NX]) {
        __syncwarp();
#pragma unroll
        for (int j = 0; j < NI; ++j) sts_piece<T, RX, SX>(gxo(j), own[j]);
        __syncwarp();
#pragma unroll
        for (int j = 0; j < NI; ++j) {
#pragma unroll
            for (int c = 0; c < NXP / W; ++c) {
                T t[W];
                ldsv(gxf(j) + (unsigned)(c * W) * ES, t);
#pragma unroll
                for (int e = 0; e < W; ++e)
                    if (c * W + e < NX) full[j][c * W + e] = t[e];
            }
        }
    };
    auto gather_u = [&](const T (&own)[NI][RU], T (&full)[NI][NU]) {
        __syncwarp();
#pragma unroll
        for (int j = 0; j < NI; ++j) sts_piece<T, RU, SU>(guo(j), own[j]);
        __syncwarp();
#pragma unroll
        for (int j = 0; j < NI; ++j) {
#pragma unroll
            for (int c = 0; c < NUP / W; ++c) {
                T t[W];
                ldsv(guf(j) + (unsigned)(c * W) * ES, t);
#pragma unroll
                for (int e = 0; e < W; ++e)
                    if (c * W + e < NU) full[j][c * W + e] = t[e];
            }
        }
    };

    // ---- streamed state of this warp: records [k][field][slot of the warp][row] ----
    // region A records first (N * recA), then, when maintained, the region B records (N * recB)
    T *const wsw = P.gps_ws + (int64_t)(blockIdx.x * nwarps + warp) * N * (recA + (has_b ? recB : 0));
    T *const wsb = wsw + (int64_t)N * recA;
    // this lane's rows of the group's first instance inside a state-shaped / input-shaped field of record 0; the second
    // instance of the group sits JX / JU elements further
    T *const px0 = wsw + grp * NX + l * RX;
    T *const pu0 = wsw + grp * NU + l * RU;

    const bool cold = P.cold != 0;
    const bool tvb = P.bounds_tv != 0;
    const bool enx = P.en_state_bound != 0, enu = P.en_input_bound != 0;
    const T kInf = (T)INFINITY;
    T loX[RX], hiX[RX], loU[RU], hiU[RU];
#pragma unroll
    for (int a = 0; a < RX; ++a) {
        loX[a] = (enx && xvl) ? __ldg(P.x_min + l * RX + a) : -kInf;
        hiX[a] = (enx && xvl) ? __ldg(P.x_max + l * RX + a) : kInf;
    }
#pragma unroll
    for (int b = 0; b < RU; ++b) {
        loU[b] = (enu && uvl) ? __ldg(P.u_min + l * RU + b) : -kInf;
        hiU[b] = (enu && uvl) ? __ldg(P.u_max + l * RU + b) : kInf;
    }
    const bool keep_v = has_b && (P.s_v != nullptr || P.s_z != nullptr);
    // family slacks are kept (region B) when the caller wants them back
    const bool keep_f[3] = {has_b && (P.s_vcnew || P.s_zcnew), has_b && (P.s_vlnew || P.s_zlnew), has_b && (P.s_vlnew_tv || P.s_zlnew_tv)};
    // a family takes part when it is compiled in AND enabled (warp-uniform)
    const bool fx[3] = {(FAM & 1) && P.soc_x != 0, (FAM & 2) && P.lin_x != 0, (FAM & 4) && P.tvl_x != 0};
    const bool fu[3] = {(FAM & 1) && P.soc_u != 0, (FAM & 2) && P.lin_u != 0, (FAM & 4) && P.tvl_u != 0};
    const bool has_uref = P.Uref != nullptr;

    // ---- per-slot bookkeeping (identical in the L lanes of a group) ----
    int64_t inst[NI];
    bool busy[NI], want[NI];
    int it[NI], solved[NI];
#pragma unroll
    for (int j = 0; j < NI; ++j) {
        inst[j] = -1;
        busy[j] = false;
        want[j] = true;
        it[j] = solved[j] = 0;
        const T z[RX] = {};
        sts_piece<T, RX, SX>(aPark + (unsigned)((2 * j) * RX) * ES, z);
        sts_piece<T, RX, SX>(aPark + (unsigned)((2 * j + 1) * RX) * ES, z);
    }
    // x0 rows / terminal-cost rows of instance j of this lane's group: parked in shared memory, fetched where used
    auto load_x0 = [&](int j, T (&v)[RX]) { lds_piece<T, RX, SX>(aPark + (unsigned)((2 * j) * RX) * ES, v); };
    auto load_pterm = [&](int j, T (&v)[RX]) { lds_piece<T, RX, SX>(aPark + (unsigned)((2 * j + 1) * RX) * ES, v); };
    // reference columns of instance j (this lane's rows of column 0); instances outside the batch read instance 0's
    auto xref_of = [&](int j) {
        const int64_t ib = inst[j] < 0 ? 0 : inst[j];
        return P.Xref + (P.xref_pi ? ib * (int64_t)N * NX : 0) + l * RX;
    };
    auto uref_of = [&](int j) {
        const int64_t ib = inst[j] < 0 ? 0 : inst[j];
        return has_uref ? P.Uref + (P.uref_pi ? ib * (int64_t)(N - 1) * NU : 0) + l * RU : P.Xref;
    };

    // ---- cone projections of one knot point (admm.cpp:102-135).  The candidate slacks (x + gc, u + yc; own rows) of the
    // group's NI instances go to the gather scratch; the 2*NI (instance, side) vectors are work items dealt to the
    // lanes of the group; cone c of every item is projected in place (project_soc, admm.cpp:39-60), cone after cone as
    // the reference's loop does; finally every lane reads its own rows back ----
    auto cones_xu = [&](T (&sx)[NI][RX], T (&su)[NI][RU], const bool HASU) {
        __syncwarp();
#pragma unroll
        for (int j = 0; j < NI; ++j) {
            if (fx[0]) sts_piece<T, RX, SX>(gxo(j), sx[j]);
            if (fu[0] && HASU) sts_piece<T, RU, SU>(guo(j), su[j]);
        }
        __syncwarp();
        const int ncx = fx[0] ? P.ncx : 0, ncu = (fu[0] && HASU) ? P.ncu : 0;
        const int nc = ncx > ncu ? ncx : ncu;
        constexpr int ROUNDS = (2 * NI + L - 1) / L;
        for (int c = 0; c < nc; ++c) {
#pragma unroll
            for (int r = 0; r < ROUNDS; ++r) {
                const int item = r * L + l, side = item & 1;
                const int j_ = (item >> 1) < NI ? (item >> 1) : NI - 1;
                const bool ok = item < 2 * NI && (side ? c < ncu : c < ncx);
                const int st0 = ok ? (side ? P.cone_u_start[c] : P.cone_x_start[c]) : 0;
                const T mu = side ? P.cone_u_mu[c] : P.cone_x_mu[c];
                const unsigned base = (side ? guf(j_) : gxf(j_)) + (unsigned)st0 * ES;
                T s0 = lds(base, T()), s1 = lds(base + ES, T()), s2 = lds(base + 2 * ES, T());
                project_soc3_sel(s0, s1, s2, mu);
                if (ok) {
                    sts(base, s0);
                    sts(base + ES, s1);
                    sts(base + 2 * ES, s2);
                }
            }
            __syncwarp();
        }
#pragma unroll
        for (int j = 0; j < NI; ++j) {
            if (fx[0] && xvl) lds_piece<T, RX, SX>(gxo(j), sx[j]);
            if (fu[0] && HASU && uvl) lds_piece<T, RU, SU>(guo(j), su[j]);
        }
    };
    // hyperplanes (admm.cpp:138-211): the rows are applied one after the other to the whole column, so every lane of
    // the group carries the full vector through the sequence (same arithmetic on every lane) and keeps its own rows
    auto planes_x = [&](T (&own)[NI][RX], const T *A, int ld, int row0, int n, const T *bvec) {
        T full[NI][NX];
        gather_x(own, full);
#pragma unroll
        for (int j = 0; j < NI; ++j) {
            project_rows<FAST, T, NX>(full[j], A, ld, row0, n, bvec);
            T o[RX];
            extract_own<T, NX, RX, L>(full[j], l, o);
#pragma unroll
            for (int a = 0; a < RX; ++a) own[j][a] = xvl ? o[a] : own[j][a];
        }
    };
    auto planes_u = [&](T (&own)[NI][RU], const T *A, int ld, int row0, int n, const T *bvec) {
        T full[NI][NU];
        gather_u(own, full);
#pragma unroll
        for (int j = 0; j < NI; ++j) {
            project_rows<FAST, T, NU>(full[j], A, ld, row0, n, bvec);
            T o[RU];
            extract_own<T, NU, RU, L>(full[j], l, o);
#pragma unroll
            for (int b = 0; b < RU; ++b) own[j][b] = uvl ? o[b] : own[j][b];
        }
    };

    // ---- ring producers: one bulk copy per sweep step (record block of knot point k -> stage image) ----
    // forward step k into stage si: the record block of knot point k (one bulk copy); this lane's reference columns of
    // that step are pulled into L2 (per-instance references come from HBM)
    auto issue_fwd = [&](int k, int si, const T *(&xr)[NI], const T *(&ur)[NI]) {
        if (k < N) {
            bulk_load(aRing + (unsigned)si * STAGE, wsw + (int64_t)k * recA, IMGF, si);
            const unsigned pu_ = (k < N - 1 && has_uref) ? puv : 0u;
#pragma unroll
            for (int j = 0; j < NI; ++j) {
                prefetch_l2(xr[j], pxv);
                prefetch_l2(ur[j], pu_);
            }
        }
    };
    // The backward sweep fetches only q_k | r_k and does a third of the forward sweep's arithmetic per step, so it cuts the
    // same ring memory into smaller stages (BS images of IMGB bytes) and runs DB steps ahead.
    constexpr int BS = RING::BS, DB = RING::DB;
    auto issue_bwd = [&](int k, int t) {
        if (k >= 0) bulk_load(aRing + (unsigned)t * IMGB, wsw + (int64_t)k * recA + REC::q, IMGB, t);
    };

    // hyperplane family F (1 static, 2 time-varying) of column k, state side then input side: slack = project(x + dual),
    // dual += x - slack, cost -= rho (slack - dual)                  (admm.cpp:138-211, 240-255, 271-276, 284-289)
    auto planes_family = [&](auto ftag, int k, const bool HASU, unsigned bx, unsigned bu, T *cx, T *cu, const T (&xo)[NI][RX],
                             const T (&u)[NI][RU], T (&q)[NI][RX], T (&r)[NI][RU]) {
        constexpr int F = decltype(ftag)::value;
        constexpr int FSEL_ = F;
        if (fx[F]) {
            T gf[NI][RX], sf[NI][RX];
#pragma unroll
            for (int j = 0; j < NI; ++j) {
                lds_piece<T, RX, CX>(bx + (unsigned)(REC::gf(FSEL_) + j * JX) * ES, gf[j]);
#pragma unroll
                for (int a = 0; a < RX; ++a) sf[j][a] = xo[j][a] + gf[j][a];
            }
            if (F == 1) planes_x(sf, P.Alin_x, P.nlx, 0, P.nlx, P.blin_x);
            else planes_x(sf, P.tv_Alin_x, P.ntvx * N, P.ntvx * k, P.ntvx, P.tv_blin_x + (int64_t)k * P.ntvx);
#pragma unroll
            for (int j = 0; j < NI; ++j) {
                T gfn[RX];
#pragma unroll
                for (int a = 0; a < RX; ++a) {
                    gfn[a] = (gf[j][a] + xo[j][a]) - sf[j][a];
                    q[j][a] = nmac<FAST>(q[j][a], rho, sf[j][a] - gfn[a]);
                }
                stg_piece<T, RX, CX>(cx + REC::gf(F) + j * JX, gfn, pxv);
                if (keep_f[F]) stg_piece<T, RX, CX>(wsb + (int64_t)k * recB + REC::vf(F) + (j * IPW + grp) * NX + l * RX, sf[j], pxv);
            }
        }
        if (fu[F] && HASU) {
            T yf[NI][RU], sf[NI][RU];
#pragma unroll
            for (int j = 0; j < NI; ++j) {
                lds_piece<T, RU, CU>(bu + (unsigned)(REC::yf(FSEL_) + j * JU) * ES, yf[j]);
#pragma unroll
                for (int b = 0; b < RU; ++b) sf[j][b] = u[j][b] + yf[j][b];
            }
            if (F == 1) planes_u(sf, P.Alin_u, P.nlu, 0, P.nlu, P.blin_u);
            else planes_u(sf, P.tv_Alin_u, P.ntvu * (N - 1), P.ntvu * k, P.ntvu, P.tv_blin_u + (int64_t)k * P.ntvu);
#pragma unroll
            for (int j = 0; j < NI; ++j) {
                T yfn[RU];
#pragma unroll
                for (int b = 0; b < RU; ++b) {
                    yfn[b] = (yf[j][b] + u[j][b]) - sf[j][b];
                    r[j][b] = nmac<FAST>(r[j][b], rho, sf[j][b] - yfn[b]);
                }
                stg_piece<T, RU, CU>(cu + REC::yf(F) + j * JU, yfn, puv);
                if (keep_f[F]) stg_piece<T, RU, CU>(wsb + (int64_t)k * recB + REC::zf(F) + (j * IPW + grp) * NU + l * RU, sf[j], puv);
            }
        }
    };

    // ---- forward sweep: rollout (admm.cpp:25-32) fused with update_slack (:81-213), update_dual (:219-256), the
    // residual maxima of termination_condition (:310-328) and the NEXT iteration's update_linear_cost (:262-304) ----
    auto forward = [&](T (&rpx)[NI], T (&rdx)[NI], T (&rpu)[NI], T (&rdu)[NI]) {
        T mS1f[RX + RU][NX], mB[RX][NU], vQd[RX], vf[RX], vRd[RU];
        load_fwd_rows(mS1f, mB, vQd, vf, vRd);
        T xo[NI][RX], Xf[NI][NX];
        const T *xr[NI], *ur[NI];  // reference columns of the knot point D steps ahead (what the next issue fetches)
#pragma unroll
        for (int j = 0; j < NI; ++j) {
            load_x0(j, xo[j]);
            xr[j] = xref_of(j);
            ur[j] = uref_of(j);
        }
        T *cx = px0, *cu = pu0;  // this lane's rows in the record of the CURRENT knot point
        sweep_fence();
#pragma unroll
        for (int t = 0; t < D; ++t) {
            issue_fwd(t, t, xr, ur);
#pragma unroll
            for (int j = 0; j < NI; ++j) {
                xr[j] += NX;
                ur[j] += NU;
            }
        }
        gather_x(xo, Xf);
        int sc = 0, si = D % S;  // ring stage of the current step / of the step being fetched
        auto column = [&](int k, const bool HASU) {  // always inlined with a literal HASU
            issue_fwd(k + D, si, xr, ur);
            // this step's reference columns (this lane's rows): issued first, used after the first mat-vec
            T xrfs[NI][RX], urfs[NI][RU];
#pragma unroll
            for (int j = 0; j < NI; ++j) {
                ldg_piece<T, RX, CX>(xr[j] - D * NX, xrfs[j], pxv);
                ldg_piece<T, RU, CU>(ur[j] - D * NU, urfs[j], (HASU && has_uref) ? puv : 0u);
            }
            bulk_wait(sc);
            const unsigned sb = (unsigned)sc * STAGE;
            // record image of this step as seen by this lane (padding lanes: the zero image)
            const unsigned bx = xvl ? aRing + sb + lxo : aZero, bu = uvl ? aRing + sb + luo : aZero;
            T t1[NI][RX + RU], u[NI][RU], Uf[NI][NU];
#pragma unroll
            for (int j = 0; j < NI; ++j)
#pragma unroll
                for (int b = 0; b < RU; ++b) u[j][b] = T(0);
            if (HASU) {
                T dk[NI][RU];
#pragma unroll
                for (int j = 0; j < NI; ++j) lds_piece<T, RU, CU>(bu + (unsigned)(REC::d + j * JU) * ES, dk[j]);
#pragma unroll
                for (int j = 0; j < NI; ++j) dots<FAST>(mS1f, Xf[j], t1[j]);  // [A x_k ; Kinf x_k]
#pragma unroll
                for (int j = 0; j < NI; ++j)
#pragma unroll
                    for (int b = 0; b < RU; ++b) u[j][b] = (-t1[j][RX + b]) - dk[j][b];  // u_k = -(Kinf x_k) - d_k
                gather_u(u, Uf);
            }
            if (tvb) {
#pragma unroll
                for (int a = 0; a < RX; ++a) {
                    loX[a] = (enx && xvl) ? __ldg(P.x_min + (int64_t)k * NX + l * RX + a) : loX[a];
                    hiX[a] = (enx && xvl) ? __ldg(P.x_max + (int64_t)k * NX + l * RX + a) : hiX[a];
                }
                if (HASU) {
#pragma unroll
                    for (int b = 0; b < RU; ++b) {
                        loU[b] = (enu && uvl) ? __ldg(P.u_min + (int64_t)k * NU + l * RU + b) : loU[b];
                        hiU[b] = (enu && uvl) ? __ldg(P.u_max + (int64_t)k * NU + l * RU + b) : hiU[b];
                    }
                }
            }
            // ---- box constraints: state column k and input column k ----
            T q[NI][RX], r[NI][RU];
#pragma unroll
            for (int j = 0; j < NI; ++j) {
                T vo[RX], g[RX], xrf[RX], vn[RX], gn[RX], pt[RX];
                lds_piece<T, RX, CX>(bx + (unsigned)(REC::vnew + j * JX) * ES, vo);
                lds_piece<T, RX, CX>(bx + (unsigned)(REC::g + j * JX) * ES, g);
#pragma unroll
                for (int a = 0; a < RX; ++a) xrf[a] = xrfs[j][a];
                if (!HASU) load_pterm(j, pt);
#pragma unroll
                for (int a = 0; a < RX; ++a) {
                    const T v = clamp_box<FAST>(xo[j][a] + g[a], loX[a], hiX[a]);  // vnew = clamp(x + g)
                    vn[a] = v;
                    gn[a] = (g[a] + xo[j][a]) - v;                                  // g += x - vnew
                    rpx[j] = absmax(rpx[j], xo[j][a] - v);
                    rdx[j] = absmax(rdx[j], vo[a] - v);
                    // k < N-1: q_k = -(xref*Q) - rho (vnew - g);  k = N-1: p_{N-1} = -(Pinf^T xref) - rho (vnew - g)
                    const T base = HASU ? -(xrf[a] * vQd[a]) : pt[a];
                    q[j][a] = nmac<FAST>(base, rho, v - gn[a]);
                }
                stg_piece<T, RX, CX>(cx + REC::vnew + j * JX, vn, pxv);
                stg_piece<T, RX, CX>(cx + REC::g + j * JX, gn, pxv);
                if (keep_v) stg_piece<T, RX, CX>(wsb + (int64_t)k * recB + REC::vprev + (j * IPW + grp) * NX + l * RX, vo, pxv);
#pragma unroll
                for (int b = 0; b < RU; ++b) r[j][b] = T(0);
                if (HASU) {
                    T zo[RU], y[RU], urf[RU], zn[RU], yn[RU];
                    lds_piece<T, RU, CU>(bu + (unsigned)(REC::znew + j * JU) * ES, zo);
                    lds_piece<T, RU, CU>(bu + (unsigned)(REC::y + j * JU) * ES, y);
#pragma unroll
                    for (int b = 0; b < RU; ++b) urf[b] = urfs[j][b];
#pragma unroll
                    for (int b = 0; b < RU; ++b) {
                        const T z = clamp_box<FAST>(u[j][b] + y[b], loU[b], hiU[b]);
                        zn[b] = z;
                        yn[b] = (y[b] + u[j][b]) - z;
                        rpu[j] = absmax(rpu[j], u[j][b] - z);
                        rdu[j] = absmax(rdu[j], zo[b] - z);
                        const T urb = has_uref ? urf[b] : T(0);
                        r[j][b] = nmac<FAST>(-(urb * vRd[b]), rho, z - yn[b]);
                    }
                    stg_piece<T, RU, CU>(cu + REC::znew + j * JU, zn, puv);
                    stg_piece<T, RU, CU>(cu + REC::y + j * JU, yn, puv);
                    if (keep_v) stg_piece<T, RU, CU>(wsb + (int64_t)k * recB + REC::zprev + (j * IPW + grp) * NU + l * RU, zo, puv);
                }
            }
            // ---- cones (family 0): state and input side together ----
            if constexpr ((FAM & 1) != 0) {
                if (fx[0] || (fu[0] && HASU)) {  // warp-uniform
                    constexpr int FSEL_ = 0;
                    T gf[NI][RX], sx[NI][RX], yf[NI][RU], su[NI][RU];
#pragma unroll
                    for (int j = 0; j < NI; ++j) {
                        lds_piece<T, RX, CX>(bx + (unsigned)(REC::gf(FSEL_) + j * JX) * ES, gf[j]);
                        lds_piece<T, RU, CU>(bu + (unsigned)(REC::yf(FSEL_) + j * JU) * ES, yf[j]);
#pragma unroll
                        for (int a = 0; a < RX; ++a) sx[j][a] = xo[j][a] + gf[j][a];
#pragma unroll
                        for (int b = 0; b < RU; ++b) su[j][b] = u[j][b] + yf[j][b];
                    }
                    cones_xu(sx, su, HASU);
#pragma unroll
                    for (int j = 0; j < NI; ++j) {
                        if (fx[0]) {
                            T gfn[RX];
#pragma unroll
                            for (int a = 0; a < RX; ++a) {
                                gfn[a] = (gf[j][a] + xo[j][a]) - sx[j][a];
                                q[j][a] = nmac<FAST>(q[j][a], rho, sx[j][a] - gfn[a]);
                            }
                            stg_piece<T, RX, CX>(cx + REC::gf(0) + j * JX, gfn, pxv);
                            if (keep_f[0]) stg_piece<T, RX, CX>(wsb + (int64_t)k * recB + REC::vf(0) + (j * IPW + grp) * NX + l * RX, sx[j], pxv);
                        }
                        if (fu[0] && HASU) {
                            T yfn[RU];
#pragma unroll
                            for (int b = 0; b < RU; ++b) {
                                yfn[b] = (yf[j][b] + u[j][b]) - su[j][b];
                                r[j][b] = nmac<FAST>(r[j][b], rho, su[j][b] - yfn[b]);
                            }
                            stg_piece<T, RU, CU>(cu + REC::yf(0) + j * JU, yfn, puv);
                            if (keep_f[0]) stg_piece<T, RU, CU>(wsb + (int64_t)k * recB + REC::zf(0) + (j * IPW + grp) * NU + l * RU, su[j], puv);
                        }
                    }
                }
            }
            // ---- hyperplanes (families 1, 2) ----
            if constexpr ((FAM & 2) != 0) planes_family(IdxTag<1>{}, k, HASU, bx, bu, cx, cu, xo, u, q, r);
            if constexpr ((FAM & 4) != 0) planes_family(IdxTag<2>{}, k, HASU, bx, bu, cx, cu, xo, u, q, r);
#pragma unroll
            for (int j = 0; j < NI; ++j) {
                stg_piece<T, RX, CX>(cx + REC::q + j * JX, q[j], pxv);
                if (HASU) stg_piece<T, RU, CU>(cu + REC::r + j * JU, r[j], puv);
            }
            if (HASU) {  // x_{k+1} = (A x_k + B u_k) + f                                  (admm.cpp:30)
#pragma unroll
                for (int j = 0; j < NI; ++j) {
                    T bu_[RX];
                    dots<FAST>(mB, Uf[j], bu_);
#pragma unroll
                    for (int a = 0; a < RX; ++a) xo[j][a] = (t1[j][a] + bu_[a]) + vf[a];
                }
                gather_x(xo, Xf);
            }
            cx += recA;
            cu += recA;
#pragma unroll
            for (int j = 0; j < NI; ++j) {
                xr[j] += NX;
                ur[j] += NU;
            }
            sc = (sc + 1 == S) ? 0 : sc + 1;
            si = (si + 1 == S) ? 0 : si + 1;
        };
        for (int k = 0; k < N - 1; ++k) column(k, true);
        column(N - 1, false);
    };

    // ---- backward sweep (admm.cpp:13-20) on the stored linear cost ----
    auto backward = [&]() {
        T mS1b[RX + RU][NX], mKt[RX][NU], mQuu[RU][NU], vAPf[RX], vBPf[RU];
        load_bwd_rows(mS1b, mKt, mQuu, vAPf, vBPf);
        T *cu = pu0 + (int64_t)(N - 1) * recA;  // this lane's input rows in the record of the current knot point
        sweep_fence();
#pragma unroll
        for (int t = 0; t < DB; ++t) issue_bwd(N - 1 - t, t);
        int tc = 0, ti = DB % BS;  // ring stage of the current step / of the step being fetched
        T po[NI][RX], Pf[NI][NX];
        {   // terminal cost p_{N-1}
            issue_bwd(N - 1 - DB, ti);
            bulk_wait(tc);
            const unsigned ox = xvl ? aRing + (unsigned)tc * IMGB + lxo : aZero;
#pragma unroll
            for (int j = 0; j < NI; ++j) lds_piece<T, RX, CX>(ox + (unsigned)(j * JX) * ES, po[j]);
            gather_x(po, Pf);
            cu -= recA;
            tc = (tc + 1 == BS) ? 0 : tc + 1;
            ti = (ti + 1 == BS) ? 0 : ti + 1;
        }
        for (int k = N - 2; k >= 0; --k) {
            issue_bwd(k - DB, ti);
            bulk_wait(tc);
            T q[NI][RX], r[NI][RU], Rf[NI][NU];
            const unsigned ox = xvl ? aRing + (unsigned)tc * IMGB + lxo : aZero;
            const unsigned ou = uvl ? aRing + (unsigned)tc * IMGB + luo : aZero;
#pragma unroll
            for (int j = 0; j < NI; ++j) {
                lds_piece<T, RX, CX>(ox + (unsigned)(j * JX) * ES, q[j]);
                lds_piece<T, RU, CU>(ou + (unsigned)(REC::r - REC::q + j * JU) * ES, r[j]);
            }
            gather_u(r, Rf);
            // d_k = Quu_inv ((B^T p_{k+1} + r_k) + BPf)
            T s_[NI][RU], Sf[NI][NU], acc1[NI][RX + RU];
#pragma unroll
            for (int j = 0; j < NI; ++j) {
                dots<FAST>(mS1b, Pf[j], acc1[j]);  // [AmBKt p_{k+1} ; B^T p_{k+1}]
#pragma unroll
                for (int b = 0; b < RU; ++b) s_[j][b] = (acc1[j][RX + b] + r[j][b]) + vBPf[b];
            }
            gather_u(s_, Sf);
            // p_k = ((q_k + AmBKt p_{k+1}) - Kinf^T r_k) + APf
#pragma unroll
            for (int j = 0; j < NI; ++j) {
                T kr[RX];
                dots<FAST>(mKt, Rf[j], kr);
#pragma unroll
                for (int a = 0; a < RX; ++a) po[j][a] = ((q[j][a] + acc1[j][a]) - kr[a]) + vAPf[a];
            }
            if (k > 0) gather_x(po, Pf);  // p_0 itself is never used
#pragma unroll
            for (int j = 0; j < NI; ++j) {
                T dq[RU];
                dots<FAST>(mQuu, Sf[j], dq);
                stg_piece<T, RU, CU>(cu + REC::d + j * JU, dq, puv);
            }
            cu -= recA;
            tc = (tc + 1 == BS) ? 0 : tc + 1;
            ti = (ti + 1 == BS) ? 0 : ti + 1;
        }
    };

    // ---- cooperative (all 32 lanes) load of instance `ib` into slot (group s, instance J of the group): the slot's
    // records are initialised from the warm-start state (zeros when cold), including the first iteration's linear cost
    // (admm.cpp:262-304 on the state as solve() finds it; cone / hyperplane slacks = previous rollout, admm.cpp:352-376) ----
    auto load_slot = [&](auto jtag, int s, int64_t ib) {
        constexpr int J = decltype(jtag)::value;
        const int sidx = J * IPW + s;
        const int64_t ox = ib * (int64_t)N * NX, ou = ib * (int64_t)(N - 1) * NU;
        const T *xrefb = P.Xref + (P.xref_pi ? ox : 0);
        const T *urefb = has_uref ? P.Uref + (P.uref_pi ? ou : 0) : nullptr;
        const T *const sgf[3] = {P.s_gc, P.s_gl, P.s_gl_tv};
        const T *const syf[3] = {P.s_yc, P.s_yl, P.s_yl_tv};
        for (int e = lane; e < N * NX; e += 32) {
            const int k = e / NX, i = e - k * NX;
            const T vnew_in = (!cold && P.s_vnew) ? P.s_vnew[ox + e] : T(0);
            const T g_in = (!cold && P.s_g) ? P.s_g[ox + e] : T(0);
            const T v_in = (!cold && P.s_v) ? P.s_v[ox + e] : T(0);
            T acc;
            if (k < N - 1) {
                acc = -(__ldg(xrefb + e) * __ldg(gmat + OFF_QD + i));
            } else {  // -(Pinf^T xref_{N-1})(i), m ascending
                const T *xl = xrefb + (int64_t)(N - 1) * NX;
                T sacc = __ldg(xl) * __ldg(gmat + OFF_PINF + NX * i);
                for (int m = 1; m < NX; ++m) sacc = mac<FAST>(sacc, __ldg(xl + m), __ldg(gmat + OFF_PINF + m + NX * i));
                acc = -sacc;
            }
            acc = nmac<FAST>(acc, rho, vnew_in - g_in);
            T *r_ = wsw + (int64_t)k * recA + sidx * NX + i;
            T *rb_ = wsb + (int64_t)k * recB + sidx * NX + i;
            r_[REC::vnew] = v_in;  // the slot of the box slack holds work->v until the first forward sweep rewrites it
            r_[REC::g] = g_in;
            if constexpr (EXT) {
                const T xin = (k == 0) ? __ldg(P.x0 + ib * NX + i) : ((!cold && P.s_x) ? P.s_x[ox + e] : T(0));
#pragma unroll
                for (int f = 0; f < 3; ++f) {
                    if (((FAM >> f) & 1) && fx[f]) {
                        const T gf_in = (!cold && sgf[f]) ? sgf[f][ox + e] : T(0);
                        acc = nmac<FAST>(acc, rho, xin - gf_in);
                        r_[REC::gf(f)] = gf_in;
                        if (keep_f[f]) rb_[REC::vf(f)] = xin;
                    }
                }
            }
            r_[REC::q] = acc;
        }
        for (int e = lane; e < (N - 1) * NU; e += 32) {
            const int k = e / NU, j = e - k * NU;
            const T znew_in = (!cold && P.s_znew) ? P.s_znew[ou + e] : T(0);
            const T y_in = (!cold && P.s_y) ? P.s_y[ou + e] : T(0);
            const T z_in = (!cold && P.s_z) ? P.s_z[ou + e] : T(0);
            const T ur = has_uref ? __ldg(urefb + e) : T(0);
            T acc = nmac<FAST>(-(ur * __ldg(gmat + OFF_RD + j)), rho, znew_in - y_in);
            T *r_ = wsw + (int64_t)k * recA + sidx * NU + j;
            T *rb_ = wsb + (int64_t)k * recB + sidx * NU + j;
            r_[REC::znew] = z_in;
            r_[REC::y] = y_in;
            if constexpr (EXT) {
                const T uin = (!cold && P.s_u) ? P.s_u[ou + e] : T(0);
#pragma unroll
                for (int f = 0; f < 3; ++f) {
                    if (((FAM >> f) & 1) && fu[f]) {
                        const T yf_in = (!cold && syf[f]) ? syf[f][ou + e] : T(0);
                        acc = nmac<FAST>(acc, rho, uin - yf_in);
                        r_[REC::yf(f)] = yf_in;
                        if (keep_f[f]) rb_[REC::zf(f)] = uin;
                    }
                }
            }
            r_[REC::r] = acc;
        }
        if (grp == s) {
            inst[J] = ib;
            busy[J] = true;
            it[J] = 0;
            solved[J] = 0;
            const T *xl = xrefb + (int64_t)(N - 1) * NX;
            T x0v[RX], ptv[RX];
#pragma unroll
            for (int a = 0; a < RX; ++a) {
                const int ii = xvl ? l * RX + a : 0;
                x0v[a] = xvl ? __ldg(P.x0 + ib * NX + ii) : T(0);
                T sacc = __ldg(xl) * __ldg(gmat + OFF_PINF + NX * ii);
                for (int m = 1; m < NX; ++m) sacc = mac<FAST>(sacc, __ldg(xl + m), __ldg(gmat + OFF_PINF + m + NX * ii));
                ptv[a] = xvl ? -sacc : T(0);
            }
            sts_piece<T, RX, SX>(aPark + (unsigned)((2 * J) * RX) * ES, x0v);
            sts_piece<T, RX, SX>(aPark + (unsigned)((2 * J + 1) * RX) * ES, ptv);
            // the four residuals keep their last checked value (types.hpp:202-205); none checked yet
            if (l == 0 && P.residuals) {
                T *r4 = P.residuals + 4 * ib;
                r4[0] = r4[1] = r4[2] = r4[3] = T(0);
            }
        }
        __syncwarp();  // the records were written by all lanes; their owners read them from here on
    };

    // ---- cooperative write-back of slot (group s, instance J of the group) holding instance `ib` ----
    auto store_slot = [&](auto jtag, int s, int64_t ib) {
        constexpr int J = decltype(jtag)::value;
        const int sidx = J * IPW + s;
        const int s_solved = __shfl_sync(0xffffffffu, solved[J], s * L);
        const int s_it = __shfl_sync(0xffffffffu, it[J], s * L);
        if (grp == s && l == 0) {
            if (P.iter) P.iter[ib] = it[J];
            if (P.solved) P.solved[ib] = solved[J];
        }
        __syncwarp();  // owner lanes wrote the records; every lane reads them below
        const int64_t ox = ib * (int64_t)N * NX, ou = ib * (int64_t)(N - 1) * NU;
        const bool ran = s_it > 0;
        T *const ovf[3] = {P.s_vcnew, P.s_vlnew, P.s_vlnew_tv};
        T *const ogf[3] = {P.s_gc, P.s_gl, P.s_gl_tv};
        T *const ozf[3] = {P.s_zcnew, P.s_zlnew, P.s_zlnew_tv};
        T *const oyf[3] = {P.s_yc, P.s_yl, P.s_yl_tv};
        for (int e = lane; e < N * NX; e += 32) {
            const int k = e / NX, i = e - k * NX;
            const T *r_ = wsw + (int64_t)k * recA + sidx * NX + i;
            const T *rb_ = wsb + (int64_t)k * recB + sidx * NX + i;
            // solution->x = vnew (admm.cpp:436,452); no iteration (max_iter <= 0): the state as it came in
            const T v = ran ? r_[REC::vnew] : ((!cold && P.s_vnew) ? P.s_vnew[ox + e] : T(0));
            if (P.sol_x) P.sol_x[ox + e] = v;
            if (P.s_vnew) P.s_vnew[ox + e] = v;
            if (P.s_g) P.s_g[ox + e] = r_[REC::g];
            // work->v: previous vnew when the solve converged (the return at admm.cpp:441 precedes :445), else = vnew
            if (P.s_v && ran) P.s_v[ox + e] = s_solved ? rb_[REC::vprev] : v;
            else if (P.s_v && cold) P.s_v[ox + e] = T(0);
            if constexpr (EXT) {
#pragma unroll
                for (int f = 0; f < 3; ++f) {
                    if (((FAM >> f) & 1) && fx[f]) {
                        if (ovf[f]) ovf[f][ox + e] = rb_[REC::vf(f)];
                        if (ogf[f]) ogf[f][ox + e] = r_[REC::gf(f)];
                    }
                }
            }
        }
        for (int e = lane; e < (N - 1) * NU; e += 32) {
            const int k = e / NU, j = e - k * NU;
            const T *r_ = wsw + (int64_t)k * recA + sidx * NU + j;
            const T *rb_ = wsb + (int64_t)k * recB + sidx * NU + j;
            const T z = ran ? r_[REC::znew] : ((!cold && P.s_znew) ? P.s_znew[ou + e] : T(0));
            if (P.sol_u) P.sol_u[ou + e] = z;
            if (P.s_znew) P.s_znew[ou + e] = z;
            if (P.s_y) P.s_y[ou + e] = r_[REC::y];
            if (P.s_z && ran) P.s_z[ou + e] = s_solved ? rb_[REC::zprev] : z;
            else if (P.s_z && cold) P.s_z[ou + e] = T(0);
            if constexpr (EXT) {
#pragma unroll
                for (int f = 0; f < 3; ++f) {
                    if (((FAM >> f) & 1) && fu[f]) {
                        if (ozf[f]) ozf[f][ou + e] = rb_[REC::zf(f)];
                        if (oyf[f]) oyf[f][ou + e] = r_[REC::yf(f)];
                    }
                }
            }
        }
        // work->x / work->u (and u0 = work->u.col(0)): replay of the last rollout from d and x0, bit-identical to the last
        // forward sweep.  Every lane executes the arithmetic (the gathers are warp-wide); the lanes of group s store.
        if (P.s_x || P.s_u || P.u0) {
            __syncwarp();
            const bool mine = grp == s;
            T mS1f[RX + RU][NX], mB[RX][NU], vQd[RX], vf[RX], vRd[RU];
            load_fwd_rows(mS1f, mB, vQd, vf, vRd);
            T xo[NI][RX], Xf[NI][NX];
#pragma unroll
            for (int j = 0; j < NI; ++j) load_x0(j, xo[j]);
            gather_x(xo, Xf);
            const int kend = (P.s_x || P.s_u) ? N : 1;
            for (int k = 0; k < kend; ++k) {
                if (P.s_x && mine && xvl) {
#pragma unroll
                    for (int a = 0; a < RX; ++a) {
                        if (ran || k == 0) P.s_x[ox + (int64_t)k * NX + l * RX + a] = xo[J][a];
                        else if (cold) P.s_x[ox + (int64_t)k * NX + l * RX + a] = T(0);
                    }
                }
                if (k < N - 1) {
                    T u[NI][RU], Uf[NI][NU], t1[NI][RX + RU];
#pragma unroll
                    for (int j = 0; j < NI; ++j) {
                        T dk[RU];
#pragma unroll
                        for (int b = 0; b < RU; ++b) dk[b] = (ran && uvl) ? pu0[(int64_t)k * recA + REC::d + j * JU + b] : T(0);
                        dots<FAST>(mS1f, Xf[j], t1[j]);
#pragma unroll
                        for (int b = 0; b < RU; ++b) u[j][b] = (-t1[j][RX + b]) - dk[b];
                    }
                    if (mine && uvl) {
#pragma unroll
                        for (int b = 0; b < RU; ++b) {
                            const int64_t o = ou + (int64_t)k * NU + l * RU + b;
                            if (P.s_u) {
                                if (ran) P.s_u[o] = u[J][b];
                                else if (cold) P.s_u[o] = T(0);
                            }
                            if (P.u0 && k == 0) P.u0[ib * NU + l * RU + b] = ran ? u[J][b] : ((!cold && P.s_u) ? P.s_u[o] : T(0));
                        }
                    }
                    if (k + 1 < kend) {
                        gather_u(u, Uf);
#pragma unroll
                        for (int j = 0; j < NI; ++j) {
                            T bu_[RX];
                            dots<FAST>(mB, Uf[j], bu_);
#pragma unroll
                            for (int a = 0; a < RX; ++a) xo[j][a] = (t1[j][a] + bu_[a]) + vf[a];
                        }
                        gather_x(xo, Xf);
                    }
                }
            }
        }
        __syncwarp();
    };

    // retire / refill the J-th instance of every group that needs it
    auto service = [&](auto jtag) {
        constexpr int J = decltype(jtag)::value;
        const bool fin = busy[J] && (solved[J] || it[J] >= P.max_iter);
        const unsigned todo = __ballot_sync(0xffffffffu, (fin || (!busy[J] && want[J])) && l == 0);
        for (unsigned m = todo; m; m &= m - 1) {
            const int s = (__ffs(m) - 1) / L;
            const int64_t ib_old = __shfl_sync(0xffffffffu, inst[J], s * L);
            const int was_busy = __shfl_sync(0xffffffffu, (int)busy[J], s * L);
            unsigned long long nxt = 0;
            if (lane == 0) nxt = atomicAdd(queue, 1ULL);
            if (was_busy) store_slot(jtag, s, ib_old);
            nxt = __shfl_sync(0xffffffffu, nxt, 0);
            if ((int64_t)nxt < P.B) {
                load_slot(jtag, s, (int64_t)nxt);
            } else if (grp == s) {
                busy[J] = false;
                want[J] = false;
            }
        }
    };

    // ---- persistent loop (same protocol as the on-chip kernel): retire / refill slots, then iterate until some
    // slot terminates; the iteration loop has warp-uniform control flow only ----
    for (;;) {
        service(IdxTag<0>{});
        if constexpr (NI > 1) service(IdxTag<1>{});
        bool anyb = false, over = false;
#pragma unroll
        for (int j = 0; j < NI; ++j) {
            anyb = anyb || busy[j];
            over = over || (busy[j] && it[j] >= P.max_iter);
        }
        if (!__any_sync(0xffffffffu, anyb)) break;
        if (__any_sync(0xffffffffu, over)) continue;  // max_iter <= 0: retire without iterating
        __syncwarp();
        bool stop;
        do {
            backward();
            __syncwarp();
            T rpx[NI], rdx[NI], rpu[NI], rdu[NI];
#pragma unroll
            for (int j = 0; j < NI; ++j) rpx[j] = rdx[j] = rpu[j] = rdu[j] = T(0);
            forward(rpx, rdx, rpu, rdu);
            __syncwarp();
            // termination_condition (admm.cpp:310-328), per instance
            stop = false;
#pragma unroll
            for (int j = 0; j < NI; ++j) {
                const T a = group_max<T, L>(rpx[j]), b = group_max<T, L>(rdx[j]), c = group_max<T, L>(rpu[j]), d = group_max<T, L>(rdu[j]);
                if (busy[j]) {
                    it[j] += 1;
                    if (it[j] % P.check_termination == 0) {
                        const T r_px = a, r_dx = b * rho, r_pu = c, r_du = d * rho;
                        if (l == 0 && P.residuals) {
                            T *r4 = P.residuals + 4 * inst[j];
                            r4[0] = r_px; r4[1] = r_dx; r4[2] = r_pu; r4[3] = r_du;
                        }
                        if (r_px < P.pri_tol && r_pu < P.pri_tol && r_dx < P.dua_tol && r_du < P.dua_tol) solved[j] = 1;
                    }
                }
                stop = stop || (busy[j] && (solved[j] || it[j] >= P.max_iter));
            }
        } while (!__any_sync(0xffffffffu, stop));
    }
}

// ---------------------------------------------------------------------------------------------------------
// host side: resident-slot plan, variant dispatch, launch
// ---------------------------------------------------------------------------------------------------------
inline int gps_env_int(const char *name, int dflt) {
    const char *e = std::getenv(name);
    return e ? std::atoi(e) : dflt;
}

template <typename T, int NX, int NU, int L, int NI, int FAM>
inline LaunchPlan gps_plan_L(const LaunchDesc &d) {
    using Cfg = GpsCfg<NX, NU, L, (int)sizeof(T), NI, FAM>;
    using REC = GpsRec<NX, NU, Cfg::SPW, (int)sizeof(T), FAM>;
    LaunchPlan p;
    const int SPW = Cfg::SPW;
    const tinympc_state_t &s = d.io.state;
    const size_t blob = ((size_t)(3 * NX * NX + 2 * NX * NU + NU * NU + 4 * NX + 2 * NU) * sizeof(T) + 15) / 16 * 16;
    using RINGH = GpsRing<NX, NU, L, (int)sizeof(T), NI, FAM>;
    const size_t per_warp = RINGH::WARP_BYTES, fixed = blob + RINGH::ZERO_BYTES;
    if (fixed + per_warp > (size_t)d.smem_budget) return p;
    int maxw = (int)std::min<size_t>(gps_max_warps(NI), ((size_t)d.smem_budget - fixed) / per_warp);
    maxw = std::max(1, std::min(maxw, std::max(1, gps_env_int("TINYMPC_GPS_WARPS", gps_max_warps(NI)))));
    // balance the waves: with `waves` passes over the resident slots, use just enough warps per SM to hold B / waves
    const int64_t groups = (d.io.B + SPW - 1) / SPW;  // warps' worth of instances
    const int64_t cap = (int64_t)d.sm_count * maxw;
    const int64_t waves = std::max<int64_t>(1, (groups + cap - 1) / cap);
    const int warps = (int)std::min<int64_t>(maxw, std::max<int64_t>(1, (groups + waves * d.sm_count - 1) / (waves * d.sm_count)));
    p.family = TINYMPC_KERNEL_GPS;
    p.lanes = L;
    p.group_instances = NI;
    p.warps_resident = maxw;
    p.instances_per_cta = warps * (32 / L) * NI;
    p.threads = warps * 32;
    p.ctas = (int)std::max<int64_t>(1, std::min<int64_t>(d.sm_count, (groups + warps - 1) / warps));
    p.smem = fixed + per_warp * (size_t)warps;
    // region B: previous box slacks (work->v / work->z) and family slacks, only when the caller wants them back
    p.gps_has_b = (s.v || s.z || s.vcnew || s.zcnew || s.vlnew || s.zlnew || s.vlnew_tv || s.zlnew_tv) ? 1 : 0;
    p.workspace_bytes = (size_t)p.ctas * warps * d.N * (REC::recA + (p.gps_has_b ? REC::recB : 0)) * sizeof(T);
    return p;
}

template <typename T, int NX, int NU, int L, int NI, int FAM, bool FAST>
int launch_gps_cfg(LaunchDesc *d, const LaunchPlan &plan, const KParams<T, NX, NU> &P0) {
    KParams<T, NX, NU> P = P0;
    P.gps.has_b = plan.gps_has_b;
    P.gps_ws = (T *)d->workspace;
    auto kern = gps_solve_kernel<T, NX, NU, L, NI, FAM, FAST>;
    if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)plan.smem) != cudaSuccess) return TINYMPC_ERR_CUDA;
    kern<<<plan.ctas, plan.threads, plan.smem, d->stream>>>(P, (const T *)d->gmat, (unsigned long long *)d->work_queue);
    return cudaGetLastError() == cudaSuccess ? TINYMPC_OK : TINYMPC_ERR_CUDA;
}

// family mask of the kernel that serves a feature set: 0 box only, 1 cones only, 6 hyperplanes only, 7 anything else
inline int gps_family_mask(const LaunchDesc &d) {
    const bool soc = d.soc_x || d.soc_u, lin = d.lin_x || d.lin_u || d.tvl_x || d.tvl_u;
    return !soc && !lin ? 0 : (soc && !lin ? 1 : (!soc ? 6 : 7));
}

// The compiled variant that serves d, for the planner and the launcher alike: f(IdxTag<L>, IdxTag<NI>, IdxTag<FAM>) with
// the shape's lane width L, the family mask FAM of d and NI instances per lane group; `none` when the shape has no
// variant.  Only the planner's NI is compiled; -DTM_GPS_TUNE also builds the one-instance variant of the shapes that
// default to two, which ni = 1 selects (developer sweeps).
template <typename T, int NX, int NU, typename R, typename F>
R gps_variant(const LaunchDesc &d, int ni, R none, F &&f) {
    constexpr int L = gps_pick_L<T, NX, NU>();
    if constexpr (L == 0) {
        return none;
    } else {
        constexpr int NIP = gps_pick_NI<T, NX, NU, L>();
        const int fam = gps_family_mask(d);
        (void)ni;
#ifdef TM_GPS_TUNE
#define TM_GPS_CASE(FF)                                                  \
    if (fam == FF) {                                                     \
        if constexpr (NIP == 2) {                                        \
            if (ni == 1) return f(IdxTag<L>{}, IdxTag<1>{}, IdxTag<FF>{}); \
        }                                                                \
        return f(IdxTag<L>{}, IdxTag<NIP>{}, IdxTag<FF>{});              \
    }
#else
#define TM_GPS_CASE(FF) \
    if (fam == FF) return f(IdxTag<L>{}, IdxTag<NIP>{}, IdxTag<FF>{});
#endif
        TM_GPS_CASE(0)
        TM_GPS_CASE(1)
        TM_GPS_CASE(6)
        TM_GPS_CASE(7)
#undef TM_GPS_CASE
        return none;
    }
}

}  // namespace tmpc
