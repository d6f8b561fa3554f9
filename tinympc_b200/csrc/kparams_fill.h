// kparams_fill.h — LaunchDesc (type-erased, host) -> KParams<T,NX,NU> (the kernels' parameter block).
#pragma once
#include <cstring>
#include <limits>

#include "common.cuh"
#include "launch.h"

namespace tmpc {

template <typename T, int NX, int NU>
inline void fill_params(KParams<T, NX, NU> &P, const LaunchDesc &d) {
    std::memset(&P, 0, sizeof(P));
    std::memcpy(P.A, d.A, sizeof(T) * NX * NX);
    std::memcpy(P.Bm, d.Bm, sizeof(T) * NX * NU);
    std::memcpy(P.f, d.f, sizeof(T) * NX);
    std::memcpy(P.Qd, d.Qd, sizeof(T) * NX);
    std::memcpy(P.Rd, d.Rd, sizeof(T) * NU);
    std::memcpy(P.Kinf, d.Kinf, sizeof(T) * NU * NX);
    std::memcpy(P.Pinf, d.Pinf, sizeof(T) * NX * NX);
    std::memcpy(P.Quu, d.Quu, sizeof(T) * NU * NU);
    std::memcpy(P.AmBKt, d.AmBKt, sizeof(T) * NX * NX);
    std::memcpy(P.APf, d.APf, sizeof(T) * NX);
    std::memcpy(P.BPf, d.BPf, sizeof(T) * NU);
    P.rho = (T)d.rho;
    P.pri_tol = (T)d.pri_tol;
    P.dua_tol = (T)d.dua_tol;
    P.N = d.N;
    P.max_iter = d.max_iter;
    P.check_termination = d.check_termination;
    P.en_state_bound = d.en_state_bound;
    P.en_input_bound = d.en_input_bound;
    P.soc_x = d.soc_x; P.soc_u = d.soc_u; P.ncx = d.ncx; P.ncu = d.ncu;
    P.lin_x = d.lin_x; P.lin_u = d.lin_u; P.nlx = d.nlx; P.nlu = d.nlu;
    P.tvl_x = d.tvl_x; P.tvl_u = d.tvl_u; P.ntvx = d.ntvx; P.ntvu = d.ntvu;
    for (int c = 0; c < MAX_CONES; ++c) {
        P.cone_x_start[c] = d.cone_x_start[c];
        P.cone_u_start[c] = d.cone_u_start[c];
        P.cone_x_mu[c] = (T)d.cone_x_mu[c];
        P.cone_u_mu[c] = (T)d.cone_u_mu[c];
    }
    const tinympc_batch_t &io = d.io;
    P.B = io.B;
    P.Bpad = d.Bpad;
    P.cold = io.cold_start;
    P.bounds_tv = d.bounds_tv;
    {
        const T inf = std::numeric_limits<T>::infinity();
        for (int i = 0; i < NX; ++i) {
            P.xlo[i] = (d.en_state_bound && d.h_xlo) ? ((const T *)d.h_xlo)[i] : -inf;
            P.xhi[i] = (d.en_state_bound && d.h_xhi) ? ((const T *)d.h_xhi)[i] : inf;
        }
        for (int j = 0; j < NU; ++j) {
            P.ulo[j] = (d.en_input_bound && d.h_ulo) ? ((const T *)d.h_ulo)[j] : -inf;
            P.uhi[j] = (d.en_input_bound && d.h_uhi) ? ((const T *)d.h_uhi)[j] : inf;
        }
    }
    P.Pinf_g = d.gmat ? (const T *)d.gmat + (NX * NX + NX * NU + NX + NX + NU + NU * NX) : nullptr;
    P.xref_pi = io.xref_per_instance;
    P.uref_pi = io.uref_per_instance;
    P.x0 = (const T *)io.x0; P.Xref = (const T *)io.Xref; P.Uref = (const T *)io.Uref;
    P.x_min = (const T *)d.x_min; P.x_max = (const T *)d.x_max; P.u_min = (const T *)d.u_min; P.u_max = (const T *)d.u_max;
    P.Alin_x = (const T *)d.Alin_x; P.blin_x = (const T *)d.blin_x; P.Alin_u = (const T *)d.Alin_u; P.blin_u = (const T *)d.blin_u;
    P.tv_Alin_x = (const T *)d.tv_Alin_x; P.tv_blin_x = (const T *)d.tv_blin_x;
    P.tv_Alin_u = (const T *)d.tv_Alin_u; P.tv_blin_u = (const T *)d.tv_blin_u;
    const tinympc_state_t &s = io.state;
    P.s_x = (T *)s.x; P.s_u = (T *)s.u; P.s_v = (T *)s.v; P.s_z = (T *)s.z;
    P.s_vnew = (T *)s.vnew; P.s_znew = (T *)s.znew; P.s_g = (T *)s.g; P.s_y = (T *)s.y;
    P.s_vcnew = (T *)s.vcnew; P.s_zcnew = (T *)s.zcnew; P.s_gc = (T *)s.gc; P.s_yc = (T *)s.yc;
    P.s_vlnew = (T *)s.vlnew; P.s_zlnew = (T *)s.zlnew; P.s_gl = (T *)s.gl; P.s_yl = (T *)s.yl;
    P.s_vlnew_tv = (T *)s.vlnew_tv; P.s_zlnew_tv = (T *)s.zlnew_tv; P.s_gl_tv = (T *)s.gl_tv; P.s_yl_tv = (T *)s.yl_tv;
    P.sol_x = (T *)io.sol_x; P.sol_u = (T *)io.sol_u;
    P.iter = io.iter; P.solved = io.solved; P.residuals = (T *)io.residuals;
    P.u0 = (T *)io.u0;
    P.models = (const T *)io.models;
    P.gpi_vscratch = (T *)d.scratch;
}

}  // namespace tmpc
