// hbv_adj.cu — K3: implicit (backward-Euler) HBV with a per-lane Newton solve and its adjoint.
//
// Replaces, for `HbvAdj` (paths relative to /root/reference/src/hydrodl2):
//   models/hbv/hbv_adj.py:341-498  HBV.forward   — rhs f(y, theta, t) as 12 simultaneous fluxes
//   models/hbv/hbv_adj.py:669-687  MOL.forward   — residual G(x) = (x - xt)/dt - f(x)
//   models/hbv/hbv_adj.py:504-615  NewtonSolve.forward (batchJacobian + linalg.solve per iteration,
//                                  three host syncs per iteration)
//   models/hbv/hbv_adj.py:620-633  the intended adjoint: lambda = (dG/dx)^-T dL/dx,
//                                  dL/dp = -lambda^T dG/dp, dL/dxt = -lambda^T dG/dxt
//   models/hbv/hbv_adj.py:689-712  MOL.nsteps_pDyn time loop, :309-317 flux at the end-of-step
//                                  state and the nmul mean
//   core/calc/fdj.py:46-92         float64 forward-difference dG/dp  -> analytic here
//   core/calc/batch_jacobian.pye   (ciphertext) batched autograd Jacobian -> analytic here
//
// One thread per (basin, component) lane.  The Jacobian of the residual is block lower
// triangular — {SNOWPACK, MELTWATER} 2x2, then SM, SUZ, SLZ — so the 5x5 solve is a 2x2 Cramer
// step plus three substitutions, all in registers (no batched LU, no host round trip).
// Stopping rule (per lane; the reference's whole-batch rule cannot be evaluated by independent
// threads and makes a basin's result depend on its batch mates): update while ||G||_inf > tol,
// then one polishing update, at most `max_updates` updates.  The forward stores every
// end-of-step state ([T, 5, B, nmul]); the adjoint kernel walks them backwards, rebuilds the
// Jacobian at the converged state (exact implicit-function gradient), solves the transposed
// block system and accumulates lambda^T df/dp with PyTorch's sub-gradient conventions
// (clamp inclusive, min ties 1/2 : 1/2, mask casts carry no gradient).
#include "hbv_common.cuh"

namespace hbv {

#ifndef HBV_ADJ_BWD_MINB
#define HBV_ADJ_BWD_MINB 5     // resident CTAs per SM the adjoint kernel's registers are sized for
#endif
constexpr int ADJ_NPAR = 13;
constexpr int ADJ_TC = 8;       // time steps per output staging chunk

struct AdjFwdPtrs {
    const float* forcing; const float* dyn; const uint8_t* drop; const float* state_in;
    float* state_out; float* qsim; float* ysol; int* stats;
};
struct AdjBwdPtrs {
    const float* forcing; const float* dyn; const uint8_t* drop; const float* ysol;
    const float* gqsim; const float* gstate_out;
    float* gdyn; float* gstate_in;
    int zero_fill;
    float* gforcing;
};
// adjoint kernel forms (compile-time): ADJ_GFORCING also produces dL/d(P, T, Ep) into `gforcing`;
// ADJ_NO_PLANE makes no parameter-gradient stores (gdyn == NULL: forcing / initial-state gradient only)
constexpr int ADJ_GFORCING = 1, ADJ_NO_PLANE = 2;

// Everything one evaluation of the right-hand side produces.
struct AdjEval {
    float SP, MW, SM, SUZ, SLZ;       // clamped stores (hbv_adj.py:385-391)
    float m0, m1, m2, m3, m4;         // clamp pass-through masks
    float dT;                         // T - TT
    float wm, pm;                     // melt = min(max(CFMAX dT, 0), SP): weight on the potential, its relu mask
    float wr, pr;                     // refreeze, same
    float a;                          // Isnow = max(MW - CWH SP, 0) mask
    float r, sw0, sw, bsw, W;         // soil wetness, PEFF = W sw
    float e;                          // excess mask
    float ef0, ef1, be, we, Ep;       // evap: et = min(SM, Ep clamp(ef0^BETAET)), we = weight on SM
    float wp;                         // perc = min(SUZ, PERC): weight on SUZ
    float u, q0a;                     // interflow mask / argument
    float f[5];                       // dS
    float Q;                          // q0 + q1 + q2
    // dense pieces of -d f/d y (before the 1/dt diagonal)
    float dP, dEt;                    // d PEFF/d SM, d et/d SM
};

template <bool BETAET>
__device__ __forceinline__ void adj_eval(const float (&y)[5], const float (&p)[ADJ_NPAR], float P, float T,
                                         float Ep, AdjEval& E) {
    E.SP = fmaxf(y[0], 0.f); E.MW = fmaxf(y[1], 0.f); E.SM = fmaxf(y[2], 1e-8f);
    E.SUZ = fmaxf(y[3], 0.f); E.SLZ = fmaxf(y[4], 0.f);
    E.m0 = (y[0] >= 0.f) ? 1.f : 0.f; E.m1 = (y[1] >= 0.f) ? 1.f : 0.f; E.m2 = (y[2] >= 1e-8f) ? 1.f : 0.f;
    E.m3 = (y[3] >= 0.f) ? 1.f : 0.f; E.m4 = (y[4] >= 0.f) ? 1.f : 0.f;
    const float TT = p[HBV_P_TT];
    E.dT = T - TT;
    const float sf = (T < TT) ? P : 0.f;
    const float rf = (T >= TT) ? P : 0.f;
    // refreeze (hbv_adj.py:448-452)
    const float rp0 = p[HBV_P_CFR] * p[HBV_P_CFMAX] * (TT - T);
    const float rp = fmaxf(rp0, 0.f);
    E.pr = (rp0 >= 0.f) ? 1.f : 0.f;
    const float refr = fminf(rp, E.MW);
    E.wr = min_w(rp, E.MW);
    // melt (:454-458)
    const float mp0 = p[HBV_P_CFMAX] * E.dT;
    const float mp = fmaxf(mp0, 0.f);
    E.pm = (mp0 >= 0.f) ? 1.f : 0.f;
    const float melt = fminf(mp, E.SP);
    E.wm = min_w(mp, E.SP);
    // Isnow (:464-468)
    const float is0 = E.MW - p[HBV_P_CWH] * E.SP;
    const float Isnow = fmaxf(is0, 0.f);
    E.a = (is0 >= 0.f) ? 1.f : 0.f;
    // Peff (:470-474)
    E.r = fdiv(E.SM, p[HBV_P_FC]);
    E.sw0 = pow_pos(E.r, p[HBV_P_BETA]);
    E.sw = fminf(fmaxf(E.sw0, 0.f), 1.f);
    E.bsw = (E.sw0 >= 0.f && E.sw0 <= 1.f) ? 1.f : 0.f;
    E.W = rf + Isnow;
    const float PEFF = E.W * E.sw;
    // excess (:476-479)
    const float ex0 = E.SM - p[HBV_P_FC];
    const float ex = fmaxf(ex0, 0.f);
    E.e = (ex0 >= 0.f) ? 1.f : 0.f;
    // evap (:481-486)
    E.ef0 = fdiv(E.SM, p[HBV_P_LP] * p[HBV_P_FC]);
    E.ef1 = BETAET ? pow_pos(E.ef0, p[HBV_P_BETAET]) : E.ef0;
    const float ef = fminf(fmaxf(E.ef1, 0.f), 1.f);
    E.be = (E.ef1 >= 0.f && E.ef1 <= 1.f) ? 1.f : 0.f;
    const float ETact = Ep * ef;
    const float et = fminf(E.SM, ETact);
    E.we = min_w(E.SM, ETact);
    E.Ep = Ep;
    // percolation, interflow, baseflows (:488-498)
    const float perc = fminf(E.SUZ, p[HBV_P_PERC]);
    E.wp = min_w(E.SUZ, p[HBV_P_PERC]);
    E.q0a = E.SUZ - p[HBV_P_UZL];
    E.u = (E.q0a >= 0.f) ? 1.f : 0.f;
    const float q0 = p[HBV_P_K0] * fmaxf(E.q0a, 0.f);
    const float q1 = p[HBV_P_K1] * E.SUZ;
    const float q2 = p[HBV_P_K2] * E.SLZ;
    // store ODEs (:425-429)
    E.f[0] = sf + refr - melt;
    E.f[1] = melt - refr - Isnow;
    E.f[2] = Isnow + rf - PEFF - ex - et;
    E.f[3] = PEFF + ex - perc - q0 - q1;
    E.f[4] = perc - q2;
    E.Q = q0 + q1 + q2;
    // derivatives w.r.t. SM used by the Jacobian
    const float inv_SM = rcp_approx(E.SM);
    E.dP = E.W * E.bsw * p[HBV_P_BETA] * E.sw0 * inv_SM;
    const float bexp = BETAET ? p[HBV_P_BETAET] : 1.0f;
    E.dEt = E.we + (1.f - E.we) * Ep * E.be * bexp * E.ef1 * inv_SM;
}

// 1/d to ~0.5 ulp without the IEEE-division slow path (MUFU.RCP + one Newton-Raphson step); the
// Jacobian diagonals are >= 1/dt > 0 and the 2x2 determinant is >= 1/dt^2
__device__ __forceinline__ float rcp_nr(float d) {
    float r = rcp_approx(d);
    return fmaf(r, fmaf(-d, r, 1.0f), r);
}

// J = I/dt - d f/d y, block lower triangular (rows: SP, MW | SM | SUZ | SLZ).
struct AdjJac { float j00, j01, j10, j11, j20, j21, j22, j30, j31, j32, j33, j43, j44; };

__device__ __forceinline__ void adj_jac(const AdjEval& E, const float (&p)[ADJ_NPAR], float inv_dt, AdjJac& J) {
    const float ac = E.a * p[HBV_P_CWH];
    J.j00 = inv_dt + E.m0 * (1.f - E.wm);
    J.j01 = -E.m1 * (1.f - E.wr);
    J.j10 = -E.m0 * ((1.f - E.wm) + ac);
    J.j11 = inv_dt + E.m1 * ((1.f - E.wr) + E.a);
    J.j20 = E.m0 * ac * (1.f - E.sw);
    J.j21 = -E.m1 * E.a * (1.f - E.sw);
    J.j22 = inv_dt + E.m2 * (E.dP + E.e + E.dEt);
    J.j30 = E.m0 * ac * E.sw;
    J.j31 = -E.m1 * E.a * E.sw;
    J.j32 = -E.m2 * (E.dP + E.e);
    J.j33 = inv_dt + E.m3 * (E.wp + p[HBV_P_K0] * E.u + p[HBV_P_K1]);
    J.j43 = -E.m3 * E.wp;
    J.j44 = inv_dt + E.m4 * p[HBV_P_K2];
}

// One implicit step: x (in: xt, out: x^{t+1}).  Returns the number of updates; `conv` reports
// whether the stopping rule was met.
template <bool BETAET>
__device__ __forceinline__ int adj_newton(float (&x)[5], const float (&p)[ADJ_NPAR], float P, float T, float Ep,
                                          float inv_dt, float tol, int maxu, bool& conv, float& Qout) {
    float xt[5];
#pragma unroll
    for (int s = 0; s < 5; ++s) xt[s] = x[s];
    AdjEval E;
    conv = false;
    int n = 0;
#pragma unroll 1
    for (int it = 0; it < maxu; ++it) {
        adj_eval<BETAET>(x, p, P, T, Ep, E);
        float G[5];
        float res = 0.f;
#pragma unroll
        for (int s = 0; s < 5; ++s) { G[s] = (x[s] - xt[s]) * inv_dt - E.f[s]; res = fmaxf(res, fabsf(G[s])); }
        AdjJac J;
        adj_jac(E, p, inv_dt, J);
        const float idet = rcp_nr(J.j00 * J.j11 - J.j01 * J.j10);
        const float d0 = (G[0] * J.j11 - J.j01 * G[1]) * idet;
        const float d1 = (J.j00 * G[1] - J.j10 * G[0]) * idet;
        const float d2 = (G[2] - J.j20 * d0 - J.j21 * d1) * rcp_nr(J.j22);
        const float d3 = (G[3] - J.j30 * d0 - J.j31 * d1 - J.j32 * d2) * rcp_nr(J.j33);
        const float d4 = (G[4] - J.j43 * d3) * rcp_nr(J.j44);
        x[0] -= d0; x[1] -= d1; x[2] -= d2; x[3] -= d3; x[4] -= d4;
        ++n;
        if (res <= tol) { conv = true; break; }
    }
    // flux at the end-of-step state (hbv_adj.py:309-313)
    adj_eval<BETAET>(x, p, P, T, Ep, E);
    Qout = E.Q;
    return n;
}

template <bool BETAET, int DM>
__global__ void __launch_bounds__(128)
hbv_adj_fwd_kernel(const KDesc d, const AdjFwdPtrs io, const float tol, const int maxu) {
    constexpr int NPAR = ADJ_NPAR;
    using DS = DynSet<NPAR, DM>;
    extern __shared__ __align__(16) float qtile[];   // [ADJ_TC][NT]
    const int tid = threadIdx.x, NT = blockDim.x, nmul = d.nmul;
    const int bl = tid / nmul, j = tid - bl * nmul;
    const int b_raw = blockIdx.x * d.BPB + bl;
    const bool valid = b_raw < d.B;
    const int b = valid ? b_raw : d.B - 1;
    const int64_t lane = (int64_t)b * nmul + j;
    const int64_t nlane = (int64_t)d.B * nmul;

    float p[NPAR];
    const uint32_t dynmask = resolve_params<NPAR, DM>(d, io.dyn, nullptr, io.drop, b, j, p, nullptr, nullptr);
    const float* dyn_lane = io.dyn + (int64_t)b * d.dyn_ncol + j;
    const int64_t dyn_tstride = (int64_t)d.B * d.dyn_ncol;
    const float* fptr = io.forcing + (int64_t)b * d.nvar;
    const int64_t f_tstride = (int64_t)d.B * d.nvar;

    float x[5];
#pragma unroll
    for (int s = 0; s < 5; ++s) x[s] = __ldg(io.state_in + s * nlane + lane);

    const float inv_nmul = 1.0f / (float)nmul;
    int max_updates = 0, n_unconv = 0;
    StepIn<DS::NS> nxt;
    load_step<NPAR, DM>(d, fptr, f_tstride, dyn_lane, dyn_tstride, dynmask, 0, nxt);
    for (int t0 = 0; t0 < d.T; t0 += ADJ_TC) {
        const int tcn = min(ADJ_TC, d.T - t0);
        // not unrolled: the Newton body is ~700 SASS instructions; ptxas unrolled this loop x4 and
        // the 44 KB loop body ran out of the instruction cache (ncu: 2.9 `no_instruction` stall
        // cycles per issued instruction, the largest stall reason of the kernel)
#pragma unroll 1
        for (int tc = 0; tc < tcn; ++tc) {
            const int t = t0 + tc;
            const StepIn<DS::NS> cur = nxt;
            load_step<NPAR, DM>(d, fptr, f_tstride, dyn_lane, dyn_tstride, dynmask, min(t + 1, d.T - 1), nxt);
            apply_dyn<NPAR, DM>(d, dynmask, cur, p, nullptr);
            bool conv; float Q;
            const int n = adj_newton<BETAET>(x, p, cur.P, cur.T, cur.PET, d.inv_dt, tol, maxu, conv, Q);
            max_updates = max(max_updates, n);
            n_unconv += conv ? 0 : 1;
            if (io.ysol != nullptr && valid) {
                float* ys = io.ysol + (int64_t)t * 5 * nlane + lane;
#pragma unroll
                for (int s = 0; s < 5; ++s) ys[s * nlane] = x[s];
            }
            if (io.qsim != nullptr) qtile[tc * NT + tid] = Q * d.dt;   // simulation = flux * delta_t (:313)
        }
        if (io.qsim != nullptr) {
            __syncthreads();
            for (int it = tid; it < tcn * d.BPB; it += NT) {
                const int tc = it / d.BPB, bl2 = it - tc * d.BPB;
                const int bb = blockIdx.x * d.BPB + bl2;
                if (bb < d.B) {
                    float acc = 0.f;
                    for (int jj = 0; jj < nmul; ++jj) acc += qtile[tc * NT + bl2 * nmul + jj];
                    io.qsim[(int64_t)(t0 + tc) * d.B + bb] = acc * inv_nmul;
                }
            }
            __syncthreads();
        }
    }
    if (valid && io.state_out != nullptr) {
#pragma unroll
        for (int s = 0; s < 5; ++s) io.state_out[s * nlane + lane] = x[s];
    }
    if (io.stats != nullptr && valid) {
        atomicMax(io.stats + 0, max_updates);
        if (n_unconv) atomicAdd(io.stats + 1, n_unconv);
    }
}

// One step of the adjoint sweep at the converged end-of-step state y: adds the flux cotangent to
// gx (= dL/dx_t on entry), solves J^T lambda = gx, returns dL/dp of the step in gp,
// dL/dx_{t-1} = lambda / dt in gx and, with GF, dL/d(P, T, Ep) = lambda^T df/d(P, T, Ep) in gf.
template <bool BETAET, bool GF>
__device__ __forceinline__ void adj_bwd_step(const float (&y)[5], const float (&p)[ADJ_NPAR], float P, float T,
                                             float PET, float gQ, float inv_dt, float (&gx)[5],
                                             float (&gp)[ADJ_NPAR], float (&gf)[3]) {
    AdjEval E;
    adj_eval<BETAET>(y, p, P, T, PET, E);
    AdjJac J;
    adj_jac(E, p, inv_dt, J);
    // flux Q(x_t, p_t) = q0 + q1 + q2 read at the end-of-step state
    gx[3] += gQ * E.m3 * (p[HBV_P_K0] * E.u + p[HBV_P_K1]);
    gx[4] += gQ * E.m4 * p[HBV_P_K2];
    // J^T lambda = gx (upper block triangular)
    const float l4 = gx[4] * rcp_nr(J.j44);
    const float l3 = (gx[3] - J.j43 * l4) * rcp_nr(J.j33);
    const float l2 = (gx[2] - J.j32 * l3) * rcp_nr(J.j22);
    const float r0 = gx[0] - J.j20 * l2 - J.j30 * l3;
    const float r1 = gx[1] - J.j21 * l2 - J.j31 * l3;
    const float idet = rcp_nr(J.j00 * J.j11 - J.j01 * J.j10);
    const float l0 = (r0 * J.j11 - J.j10 * r1) * idet;
    const float l1 = (J.j00 * r1 - J.j01 * r0) * idet;
    // dL/dp = lambda^T df/dp + gQ dQ/dp, flux by flux
#pragma unroll
    for (int i = 0; i < ADJ_NPAR; ++i) gp[i] = 0.f;
    const float c_melt = (l1 - l0) * E.wm * E.pm;
    const float c_refr = (l0 - l1) * E.wr * E.pr;
    gp[HBV_P_CFMAX] = c_melt * E.dT - c_refr * p[HBV_P_CFR] * E.dT;
    gp[HBV_P_CFR] = -c_refr * p[HBV_P_CFMAX] * E.dT;
    gp[HBV_P_TT] = -c_melt * p[HBV_P_CFMAX] + c_refr * p[HBV_P_CFR] * p[HBV_P_CFMAX];
    const float c_pe = l3 - l2;
    const float c_is = (l2 - l1) + c_pe * E.sw;
    gp[HBV_P_CWH] = -c_is * E.a * E.SP;
    const float t_pe = c_pe * E.W * E.bsw * E.sw0;
    gp[HBV_P_BETA] = t_pe * flog(E.r);
    float gFC = -fdiv(t_pe * p[HBV_P_BETA], p[HBV_P_FC]) - c_pe * E.e;
    const float c_et = -l2 * (1.f - E.we) * E.Ep * E.be * E.ef1;
    const float bexp = BETAET ? p[HBV_P_BETAET] : 1.0f;
    gp[HBV_P_LP] = -fdiv(c_et * bexp, p[HBV_P_LP]);
    gFC -= fdiv(c_et * bexp, p[HBV_P_FC]);
    if constexpr (BETAET) gp[HBV_P_BETAET] = c_et * flog(E.ef0);
    gp[HBV_P_FC] = gFC;
    gp[HBV_P_PERC] = (l4 - l3) * (1.f - E.wp);
    const float c_q01 = gQ - l3;
    gp[HBV_P_K0] = c_q01 * fmaxf(E.q0a, 0.f);
    gp[HBV_P_UZL] = -c_q01 * p[HBV_P_K0] * E.u;
    gp[HBV_P_K1] = c_q01 * E.SUZ;
    gp[HBV_P_K2] = (gQ - l4) * E.SLZ;
    if constexpr (GF) {
        // P: snowfall feeds SNOWPACK; rainfall feeds SM and, through PEFF = (rf + Isnow) sw, SUZ
        // (the rain/snow mask carries no gradient).  T enters through T - TT only (melt,
        // refreeze); Ep through et = min(SM, Ep ef).  Q does not depend on the forcings.
        gf[0] = (T < p[HBV_P_TT]) ? l0 : l2 + c_pe * E.sw;
        gf[1] = -gp[HBV_P_TT];
        // (the clamped evaporation factor is recomputed, not kept in AdjEval: one more field there
        // changes the register allocation of the forward kernel K3)
        gf[2] = -l2 * (1.f - E.we) * fminf(fmaxf(E.ef1, 0.f), 1.f);
    }
    // dL/dxt = -lambda^T dG/dxt = lambda / dt
    gx[0] = l0 * inv_dt; gx[1] = l1 * inv_dt; gx[2] = l2 * inv_dt; gx[3] = l3 * inv_dt; gx[4] = l4 * inv_dt;

}

// dL/d(P, T, Ep) of step t summed over the nmul components of basin b, stored by the basin's first
// lane (deterministic, no atomics): butterfly shuffles when the lanes of a basin are an aligned
// power-of-two group of one warp (`mask`: the warp's lanes), else a sum in component order through
// the shared-memory slab [NT][3] — the sweep is uniform over the CTA, so its barriers are too.
__device__ __forceinline__ void adj_store_gforcing(const KDesc& d, float* gforcing, int t, int b, int j, int nmul,
                                                   bool valid, bool shfl, unsigned mask, float* slab, int tid,
                                                   float (&g)[3]) {
    if (shfl) {
        for (int o = nmul >> 1; o > 0; o >>= 1) {
            g[0] += __shfl_xor_sync(mask, g[0], o);
            g[1] += __shfl_xor_sync(mask, g[1], o);
            g[2] += __shfl_xor_sync(mask, g[2], o);
        }
    } else {
        slab[tid * 3 + 0] = g[0]; slab[tid * 3 + 1] = g[1]; slab[tid * 3 + 2] = g[2];
        __syncthreads();
        if (j == 0) {
            float a0 = 0.f, a1 = 0.f, a2 = 0.f;
            for (int q = 0; q < nmul; ++q) {
                a0 += slab[(tid + q) * 3 + 0]; a1 += slab[(tid + q) * 3 + 1]; a2 += slab[(tid + q) * 3 + 2];
            }
            g[0] = a0; g[1] = a1; g[2] = a2;
        }
        __syncthreads();
    }
    if (valid && j == 0) {
        float* gx = gforcing + ((int64_t)t * d.B + b) * d.nvar;
        gx[d.i_prcp] = g[0]; gx[d.i_tmean] = g[1]; gx[d.i_pet] = g[2];
    }
}

// (the forcing-gradient forms are sized for one CTA per SM fewer: at the 96 registers of
// HBV_ADJ_BWD_MINB the any-dynamic-set form spills; at 128 none does)
template <bool BETAET, int DM, int MODE>
__global__ void __launch_bounds__(128, (MODE & ADJ_GFORCING) ? HBV_ADJ_BWD_MINB - 1 : HBV_ADJ_BWD_MINB)
hbv_adj_bwd_kernel(const KDesc d, const AdjBwdPtrs io) {
    constexpr int NPAR = ADJ_NPAR;
    constexpr bool GF = (MODE & ADJ_GFORCING) != 0, PLANE = (MODE & ADJ_NO_PLANE) == 0;
    using DS = DynSet<NPAR, DM>;
    extern __shared__ __align__(16) float fx_slab[];   // GF, nmul not a power of two: [NT][3]
    const int tid = threadIdx.x, nmul = d.nmul;
    const int bl = tid / nmul, j = tid - bl * nmul;
    const int b_raw = blockIdx.x * d.BPB + bl;
    const bool valid = b_raw < d.B;
    const int b = valid ? b_raw : d.B - 1;
    const int64_t lane = (int64_t)b * nmul + j;
    const int64_t nlane = (int64_t)d.B * nmul;

    float p[NPAR], dpd[NPAR], gacc[NPAR];
    uint32_t lastmask = 0;
    const uint32_t dynmask = resolve_params<NPAR, DM>(d, io.dyn, nullptr, io.drop, b, j, p, nullptr, nullptr);
#pragma unroll
    for (int i = 0; i < NPAR; ++i) { dpd[i] = 0.f; gacc[i] = 0.f; }
    const float* dyn_lane = io.dyn + (int64_t)b * d.dyn_ncol + j;
    const int64_t dyn_tstride = (int64_t)d.B * d.dyn_ncol;
    const float* fptr = io.forcing + (int64_t)b * d.nvar;
    const int64_t f_tstride = (int64_t)d.B * d.nvar;
    float* gdyn_lane = io.gdyn + (int64_t)b * d.dyn_ncol + j;
    const float inv_nmul = 1.0f / (float)nmul;
    const float inv_dt = d.inv_dt;
    const bool shfl = (nmul & (nmul - 1)) == 0 && nmul <= 32;     // then NT is a power of two as well
    const unsigned shfl_mask = blockDim.x >= 32 ? 0xffffffffu : (1u << blockDim.x) - 1u;

    float gx[5];
#pragma unroll
    for (int s = 0; s < 5; ++s) gx[s] = io.gstate_out ? __ldg(io.gstate_out + s * nlane + lane) : 0.f;

    StepIn<DS::NS> nxt;
    float ynx[5];
    float gqn = 0.f;
    auto load_all = [&](int t) {
        const int tt = min(max(t, 0), d.T - 1);
        load_step<NPAR, DM>(d, fptr, f_tstride, dyn_lane, dyn_tstride, dynmask, tt, nxt);
        const float* ys = io.ysol + (int64_t)tt * 5 * nlane + lane;
#pragma unroll
        for (int s = 0; s < 5; ++s) ynx[s] = __ldg(ys + s * nlane);
        gqn = io.gqsim ? __ldg(io.gqsim + (int64_t)tt * d.B + b) : 0.f;
    };
    load_all(d.T - 1);
#pragma unroll 1
    for (int t = d.T - 1; t >= 0; --t) {
        const StepIn<DS::NS> cur = nxt;
        float y[5];
#pragma unroll
        for (int s = 0; s < 5; ++s) y[s] = ynx[s];
        if (PLANE && io.zero_fill) {
            // fused zero fill (nmul 16): a warp owns two basins, whose gradient rows of step t are
            // one contiguous, 8 B-aligned run; zero it with 8 B stores, then the lanes store their
            // gradients on top.  Row T-1 also receives the static-parameter and routing gradients.
            if (t < d.T - 1) {
                const int wb0 = blockIdx.x * d.BPB + (tid >> 5) * 2;
                const int nb = min(2, d.B - wb0);
                if (nb > 0) {
                    float2* z = reinterpret_cast<float2*>(io.gdyn + ((int64_t)t * d.B + wb0) * d.dyn_ncol);
                    const int n2 = (nb * d.dyn_ncol) >> 1;
                    for (int e = tid & 31; e < n2; e += 32) z[e] = make_float2(0.f, 0.f);
                }
            }
            __syncwarp();
        }
        const float gQ = gqn * inv_nmul * d.dt;
        load_all(t - 1);
        apply_dyn<NPAR, DM>(d, dynmask, cur, p, dpd);
        float gp[NPAR], gf[3];
        adj_bwd_step<BETAET, GF>(y, p, cur.P, cur.T, cur.PET, gQ, inv_dt, gx, gp, gf);

        if constexpr (PLANE) {
            float* gr = gdyn_lane + (int64_t)t * dyn_tstride;
#pragma unroll
            for (int i = 0; i < NPAR; ++i) {
                if (i < d.n_par) {
                    if (DS::is_dyn(i, dynmask)) { if (valid) gr[d.col[i]] = gp[i] * dpd[i]; }
                    else gacc[i] += gp[i];
                }
            }
        }
        // (after the parameter gradient: the reduction's branches must not split the step's
        // arithmetic from the accumulation above, or its mul-add pairs are no longer fused and
        // the parameter gradient changes in the last bits)
        if constexpr (GF) adj_store_gforcing(d, io.gforcing, t, b, j, nmul, valid, shfl, shfl_mask, fx_slab, tid, gf);
    }
    if constexpr (PLANE) resolve_params<NPAR, DM>(d, io.dyn, nullptr, io.drop, b, j, p, dpd, &lastmask);
    if (valid) {
        if constexpr (PLANE) {
            float* glast = gdyn_lane + (int64_t)(d.T - 1) * dyn_tstride;
#pragma unroll
            for (int i = 0; i < NPAR; ++i)
                if (i < d.n_par && !DS::is_dyn(i, dynmask) && (lastmask & (1u << i))) glast[d.col[i]] = gacc[i] * dpd[i];
        }
        if (io.gstate_in != nullptr) {
#pragma unroll
            for (int s = 0; s < 5; ++s) io.gstate_in[s * nlane + lane] = gx[s];
        }
    }
}

// K3^T, ring form: the same sweep for the standard case (nmul 16, forcing columns prcp / tmean /
// pet = 0 / 1 / 2 of a 3-wide x_phy, the shipped dynamic set [parBETA, parBETAET], no dropout mask)
// as one-warp CTAs whose inputs arrive through the cp.async ring of K2s (hbv_lean.cu): a step is
// staged by FOUR wide copies — 4 B x 8 lanes (P, T, PET, dL/dQ of the warp's two basins), 8 B x 32
// (the two 64 B parameter runs of each basin), 16 B x 32 + 16 B x 8 (the five 128 B rows of the
// stored solution) — ARD steps ahead, and read back with one LDS.128 + 7 LDS.  The register form
// above prefetches ONE step ahead and ncu showed 3.1 long-scoreboard stall cycles per issued
// instruction at 64 % issue-slot utilisation (profiles/r02_ncu_c5_adj.md).
constexpr int ARD = 8;
constexpr int ASLOT = 8 + 32 * (2 + 5);

// (forcing-gradient forms: at least 16 CTAs per SM, i.e. <= 128 registers — left to itself ptxas
// capped them at 96 registers and spilled)
template <bool BETAET, int MODE>
__global__ void __launch_bounds__(32, (MODE & ADJ_GFORCING) ? 16 : 0)
hbv_adj_bwd_ring_kernel(const KDesc d, const AdjBwdPtrs io) {
    constexpr int NPAR = ADJ_NPAR;
    constexpr int DM = DM_D2;
    constexpr bool GF = (MODE & ADJ_GFORCING) != 0, PLANE = (MODE & ADJ_NO_PLANE) == 0;
    using DS = DynSet<NPAR, DM>;
    extern __shared__ __align__(16) float ringmem[];
    const int tid = threadIdx.x;
    const int bl = tid >> 4, j = tid & 15;
    const int b0w = blockIdx.x * 2;
    const int b_raw = b0w + bl;
    const bool valid = b_raw < d.B;
    const int b = valid ? b_raw : d.B - 1;
    const int64_t lane = (int64_t)b * 16 + j;
    const int64_t nlane = (int64_t)d.B * 16;

    float p[NPAR], dpd[NPAR], gacc[NPAR];
    uint32_t lastmask = 0;
    const uint32_t dynmask = resolve_params<NPAR, DM>(d, io.dyn, nullptr, nullptr, b, j, p, nullptr, nullptr);
#pragma unroll
    for (int i = 0; i < NPAR; ++i) { dpd[i] = 0.f; gacc[i] = 0.f; }
    const int64_t dyn_tstride = (int64_t)d.B * d.dyn_ncol;
    float* gdyn_lane = io.gdyn + (int64_t)b * d.dyn_ncol + j;
    constexpr float inv_nmul = 1.0f / 16.0f;
    const float inv_dt = d.inv_dt;

    float gx[5];
#pragma unroll
    for (int s = 0; s < 5; ++s) gx[s] = io.gstate_out ? __ldg(io.gstate_out + s * nlane + lane) : 0.f;

    // ---- ring staging (sources positioned on step T-1, walked backwards)
    constexpr int PARB = 8, STB = 8 + 32 * 2;
    float* const ring_end = ringmem + ARD * ASLOT;
    float* wp = ringmem;
    const float* rp = ringmem;
    const int nbw = min(2, d.B - b0w);
    const int kA = tid & 15, bbA = tid >> 4;
    const bool actA = kA < 3 || (kA == 3 && io.gqsim != nullptr);
    const int64_t rowA = (int64_t)(d.T - 1) * d.B + min(b0w + bbA, d.B - 1);
    const float* srcA = (kA < 3) ? io.forcing + rowA * 3 + kA : (io.gqsim ? io.gqsim + rowA : io.forcing);
    const int64_t strA = (kA < 3) ? (int64_t)d.B * 3 : (int64_t)d.B;
    const int dstA = 4 * bbA + kA;
    // B: run r = tid >> 3 of the warp's four (basin, parameter) runs, 8 B piece q = tid & 7
    const int rB = tid >> 3, qB = tid & 7;
    const int bbB = rB >> 1, kB = rB & 1;
    const int colB = kB == 0 ? d.col[HBV_P_BETA] : d.col[HBV_P_BETAET];
    const float* srcB = io.dyn + ((int64_t)(d.T - 1) * d.B + min(b0w + bbB, d.B - 1)) * d.dyn_ncol + colB + 2 * qB;
    const int dstB = PARB + kB * 32 + bbB * 16 + 2 * qB;
    const int sC = tid >> 3, qC = tid & 7;
    const bool actC = 4 * qC < 16 * nbw;
    const float* srcC = io.ysol + ((int64_t)(d.T - 1) * 5 + sC) * nlane + (int64_t)b0w * 16 + 4 * qC;
    const float* srcD = io.ysol + ((int64_t)(d.T - 1) * 5 + 4) * nlane + (int64_t)b0w * 16 + 4 * qC;
    const bool actD = actC && tid < 8;
    const int dstC = STB + sC * 32 + 4 * qC, dstD = STB + 4 * 32 + 4 * qC;
    const int64_t strC = 5 * nlane;
    int t_stage = d.T - 1;
    auto issue = [&]() {             // stage the inputs of the next step of the sweep (if any)
        if (t_stage >= 0) {
            if (actA) cp_async4(wp + dstA, srcA);
            cp_async8(wp + dstB, srcB);
            if (actC) cp_async16(wp + dstC, srcC);
            if (actD) cp_async16(wp + dstD, srcD);
            srcA -= strA; srcB -= dyn_tstride; srcC -= strC; srcD -= strC;
        }
        --t_stage;
        cp_async_commit();
        wp += ASLOT;
        if (wp == ring_end) wp = ringmem;
    };
#pragma unroll 1
    for (int q = 0; q < ARD - 1; ++q) issue();

    const bool has_gq = io.gqsim != nullptr;
#pragma unroll 1
    for (int t = d.T - 1; t >= 0; --t) {
        cp_async_wait<ARD - 2>();
        __syncwarp();                // the oldest step has landed for every lane; the slot refilled
        issue();                     // now was read by every lane one iteration ago
        const float4 f = *reinterpret_cast<const float4*>(rp + 4 * bl);
        StepIn<DS::NS> cur;
        cur.P = f.x; cur.T = f.y; cur.PET = f.z;
        cur.raw[0] = rp[PARB + tid];
        cur.raw[1] = rp[PARB + 32 + tid];
        float y[5];
#pragma unroll
        for (int s = 0; s < 5; ++s) y[s] = rp[STB + s * 32 + tid];
        rp += ASLOT;
        if (rp == ring_end) rp = ringmem;
        if (PLANE && io.zero_fill) { // (see the register form)
            if (t < d.T - 1 && nbw > 0) {
                float2* z = reinterpret_cast<float2*>(io.gdyn + ((int64_t)t * d.B + b0w) * d.dyn_ncol);
                const int n2 = (nbw * d.dyn_ncol) >> 1;
                for (int e = tid; e < n2; e += 32) z[e] = make_float2(0.f, 0.f);
            }
            __syncwarp();
        }
        const float gQ = has_gq ? f.w * inv_nmul * d.dt : 0.f;
        apply_dyn<NPAR, DM>(d, dynmask, cur, p, dpd);
        float gp[NPAR], gf[3];
        adj_bwd_step<BETAET, GF>(y, p, cur.P, cur.T, cur.PET, gQ, inv_dt, gx, gp, gf);
        if constexpr (PLANE) {
            float* gr = gdyn_lane + (int64_t)t * dyn_tstride;
#pragma unroll
            for (int i = 0; i < NPAR; ++i) {
                if (i < d.n_par) {
                    if (DS::is_dyn(i, dynmask)) { if (valid) gr[d.col[i]] = gp[i] * dpd[i]; }
                    else gacc[i] += gp[i];
                }
            }
        }
        // (a warp is two basins of 16 lanes: two aligned shuffle groups; placed as in the register form)
        if constexpr (GF) adj_store_gforcing(d, io.gforcing, t, b, j, 16, valid, true, 0xffffffffu, nullptr, tid, gf);
    }
    cp_async_wait<0>();
    if constexpr (PLANE) resolve_params<NPAR, DM>(d, io.dyn, nullptr, nullptr, b, j, p, dpd, &lastmask);
    if (valid) {
        if constexpr (PLANE) {
            float* glast = gdyn_lane + (int64_t)(d.T - 1) * dyn_tstride;
#pragma unroll
            for (int i = 0; i < NPAR; ++i)
                if (i < d.n_par && !DS::is_dyn(i, dynmask) && (lastmask & (1u << i))) glast[d.col[i]] = gacc[i] * dpd[i];
        }
        if (io.gstate_in != nullptr) {
#pragma unroll
            for (int s = 0; s < 5; ++s) io.gstate_in[s * nlane + lane] = gx[s];
        }
    }
}

int make_kdesc(const hbv_desc_t* desc, KDesc& d);

template <bool BETAET, int DM>
static int launch_adj_fwd(const KDesc& d, const AdjFwdPtrs& io, float tol, int maxu, cudaStream_t st) {
    const int NT = d.BPB * d.nmul;
    const int grid = (d.B + d.BPB - 1) / d.BPB;
    const size_t smem = io.qsim ? (size_t)ADJ_TC * NT * sizeof(float) : 0;
    hbv_adj_fwd_kernel<BETAET, DM><<<grid, NT, smem, st>>>(d, io, tol, maxu);
    count_launch();
    const cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) set_error(cudaGetErrorString(e));
    return (int)e;
}

template <bool BETAET, int DM, int MODE>
static int launch_adj_bwd(const KDesc& d, const AdjBwdPtrs& io, cudaStream_t st) {
    const int NT = d.BPB * d.nmul;
    const int grid = (d.B + d.BPB - 1) / d.BPB;
    const bool pow2 = (d.nmul & (d.nmul - 1)) == 0 && d.nmul <= 32;   // (the kernel's shuffle test)
    const size_t smem = ((MODE & ADJ_GFORCING) && !pow2) ? (size_t)3 * NT * sizeof(float) : 0;
    hbv_adj_bwd_kernel<BETAET, DM, MODE><<<grid, NT, smem, st>>>(d, io);
    count_launch();
    const cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) set_error(cudaGetErrorString(e));
    return (int)e;
}

template <bool BETAET, int DM>
static int launch_adj_bwd(const KDesc& d, const AdjBwdPtrs& io, int mode, cudaStream_t st) {
    switch (mode) {
        case 0: return launch_adj_bwd<BETAET, DM, 0>(d, io, st);
        case ADJ_GFORCING: return launch_adj_bwd<BETAET, DM, ADJ_GFORCING>(d, io, st);
        case ADJ_NO_PLANE: return launch_adj_bwd<BETAET, DM, ADJ_NO_PLANE>(d, io, st);
        default: return launch_adj_bwd<BETAET, DM, ADJ_GFORCING | ADJ_NO_PLANE>(d, io, st);
    }
}

template <bool BETAET, int MODE>
static int launch_adj_bwd_ring(const KDesc& d, const AdjBwdPtrs& io, cudaStream_t st) {
    const int grid = (d.B + 1) / 2;
    const size_t smem = (size_t)ARD * ASLOT * sizeof(float);
    hbv_adj_bwd_ring_kernel<BETAET, MODE><<<grid, 32, smem, st>>>(d, io);
    count_launch();
    const cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) set_error(cudaGetErrorString(e));
    return (int)e;
}

template <bool BETAET>
static int launch_adj_bwd_ring(const KDesc& d, const AdjBwdPtrs& io, int mode, cudaStream_t st) {
    switch (mode) {
        case 0: return launch_adj_bwd_ring<BETAET, 0>(d, io, st);
        case ADJ_GFORCING: return launch_adj_bwd_ring<BETAET, ADJ_GFORCING>(d, io, st);
        case ADJ_NO_PLANE: return launch_adj_bwd_ring<BETAET, ADJ_NO_PLANE>(d, io, st);
        default: return launch_adj_bwd_ring<BETAET, ADJ_GFORCING | ADJ_NO_PLANE>(d, io, st);
    }
}

static int adj_prepare(const hbv_desc_t* desc, KDesc& d) {
    int rc = make_kdesc(desc, d);
    if (rc) return rc;
    while (d.BPB > 1 && d.BPB * d.nmul > 128) d.BPB >>= 1;
    if (d.BPB * d.nmul > 128) { set_error("nmul > 128 unsupported by the implicit solver"); return HBV_E_NMUL; }
    for (int i = 0; i < d.n_par; ++i)
        if (d.src[i] == HBV_SRC_STA) { set_error("hbv_adj reads packed parameters only"); return HBV_E_SHAPE; }
    return 0;
}

int adj_fwd_dispatch(const hbv_desc_t* desc, const hbv_adj_fwd_io_t* io, cudaStream_t st) {
    KDesc d;
    int rc = adj_prepare(desc, d);
    if (rc) return rc;
    // one-warp CTAs at nmul 16: the chunk barrier of the flow staging then couples no warps whose
    // Newton counts differ (10,000 basins x 730 days, forward alone: 2.79 / 2.82 / 2.84 ms with 2 / 4 / 8
    // basins per CTA)
    if (opt(OPT_ADJ_BPB) > 0 && opt(OPT_ADJ_BPB) * d.nmul <= 128) d.BPB = (int)opt(OPT_ADJ_BPB);
    else if (d.nmul == 16) d.BPB = 2;
    AdjFwdPtrs p{io->forcing, io->dyn, io->drop, io->state_in, io->state_out, io->qsim, io->ysol, io->stats};
    const float tol = desc->adj_tol > 0.f ? desc->adj_tol : 1e-3f;
    const int maxu = desc->adj_max_updates > 0 ? desc->adj_max_updates : 8;
    const int dm = static_dynmask(d, io->drop != nullptr);
    if (desc->betaet) {
        if (dm == 0) return launch_adj_fwd<true, 0>(d, p, tol, maxu, st);
        if (dm == DM_D2) return launch_adj_fwd<true, DM_D2>(d, p, tol, maxu, st);
        return launch_adj_fwd<true, -1>(d, p, tol, maxu, st);
    }
    if (dm == 0) return launch_adj_fwd<false, 0>(d, p, tol, maxu, st);
    return launch_adj_fwd<false, -1>(d, p, tol, maxu, st);
}

int adj_bwd_dispatch(const hbv_desc_t* desc, const hbv_adj_bwd_io_t* io, cudaStream_t st) {
    KDesc d;
    int rc = adj_prepare(desc, d);
    if (rc) return rc;
    AdjBwdPtrs p{io->forcing, io->dyn, io->drop, io->ysol, io->gqsim, io->gstate_out, io->gdyn, io->gstate_in, 0,
                 io->gforcing};
    if (io->gdyn_zero_fill) {
        if (d.nmul != 16 || d.dyn_ncol % 2 != 0 || io->gdyn == nullptr || reinterpret_cast<uintptr_t>(io->gdyn) % 8 != 0) {
            set_error("adj_bwd: gdyn_zero_fill needs nmul 16, an even row width and an 8 B-aligned gdyn");
            return HBV_E_SHAPE;
        }
        p.zero_fill = 1;
    }
    const int mode = (io->gforcing != nullptr ? ADJ_GFORCING : 0) | (io->gdyn == nullptr ? ADJ_NO_PLANE : 0);
    const int dm = static_dynmask(d, io->drop != nullptr);
    // standard case: the ring form (wide cp.async copies: even rows, 8 / 16 B-aligned bases)
    if (dm == DM_D2 && d.nmul == 16 && d.nvar == 3 && d.i_prcp == 0 && d.i_tmean == 1 && d.i_pet == 2 &&
        d.dyn_ncol % 2 == 0 && d.col[HBV_P_BETA] % 2 == 0 && d.col[HBV_P_BETAET] % 2 == 0 &&
        reinterpret_cast<uintptr_t>(io->dyn) % 8 == 0 && reinterpret_cast<uintptr_t>(io->ysol) % 16 == 0 &&
        reinterpret_cast<uintptr_t>(io->gdyn) % 8 == 0 && opt(OPT_RING) != 0) {   // (gdyn may be NULL)
        return desc->betaet ? launch_adj_bwd_ring<true>(d, p, mode, st) : launch_adj_bwd_ring<false>(d, p, mode, st);
    }
    if (desc->betaet) {
        if (dm == 0) return launch_adj_bwd<true, 0>(d, p, mode, st);
        if (dm == DM_D2) return launch_adj_bwd<true, DM_D2>(d, p, mode, st);
        return launch_adj_bwd<true, -1>(d, p, mode, st);
    }
    if (dm == 0) return launch_adj_bwd<false, 0>(d, p, mode, st);
    return launch_adj_bwd<false, -1>(d, p, mode, st);
}

}  // namespace hbv
