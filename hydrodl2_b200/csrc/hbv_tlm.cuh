// hbv_tlm.cuh — tangent-linear HBV step (forward-mode derivative) for one (basin, component) lane.
//
// Each stage evaluates the primal with the very same code as the forward kernels (snow_fwd /
// soil_fwd / resp_fwd of hbv_step.cuh, with the tape on) and then pushes the tangents of its
// states, parameters and forcings through the recorded intermediates.  The sub-gradient
// conventions are PyTorch's, as in the adjoint of hbv_step.cuh (which is the transpose of what is
// written here):
//   min(a, b): the tangent of the smaller operand, the mean of both on a tie;
//   clamp(x, lo, hi) / max(x, c): the tangent passes where lo <= x <= hi (bounds inclusive);
//   relu(0) = 0 (routing only); a**b at a = 0: 0 for both the base and the exponent tangent;
//   mask conditions (rain / snow, the parTT elevation switch, the Ac branch) carry no tangent.
#pragma once
#include "hbv_common.cuh"

namespace hbv {

// snow routine.  In: dSP, dMW (tangents of the state before the step), dP, dT (forcing tangents
// as the step uses them), dp (parameter tangents).  Out: the same states after the step, the
// tangents of RAIN and tosoil.
template <int VAR>
__device__ __forceinline__ void snow_tlm(float& SP, float& MW, float& dSP, float& dMW,
                                         const float (&p)[Traits<VAR>::NPAR], const float (&dp)[Traits<VAR>::NPAR],
                                         float P, float T, float dP, float dT, const LaneConst& c,
                                         float& RAIN, float& tosoil, float& dRAIN, float& dtosoil, Tape& tp) {
    using TR = Traits<VAR>;
    const float dt = c.dt, inv_dt = c.inv_dt;
    auto D = [&](float x) { return TR::HOURLY ? x * dt : x; };
    auto ID = [&](float x) { return TR::HOURLY ? x * inv_dt : x; };
    snow_fwd<VAR, true>(SP, MW, p, P, T, c, RAIN, tosoil, tp);
    float sp = dSP, mw = dMW;
    if constexpr (TR::HOURLY) {   // guard rails: clamp(x, min=0) passes where x >= 0
        sp = (tp.SPg >= 0.f) ? sp : 0.f;
        mw = (tp.MWg >= 0.f) ? mw : 0.f;
    }
    float dTTe = dp[HBV_P_TT];
    if constexpr (TR::LAT) dTTe = (c.Elev >= 2000.f) ? 0.f : dp[HBV_P_TT];
    const bool israin = (T >= tp.TTe);
    dRAIN = israin ? dP : 0.f;
    const float dSNOW = (T < tp.TTe) ? dP : 0.f;
    const float ddT = dT - dTTe;
    const float dSP1 = sp + D(dSNOW);
    const float dmelt0 = dp[HBV_P_CFMAX] * tp.dT + p[HBV_P_CFMAX] * ddT;
    const float dmelt2 = (tp.melt0 >= 0.f) ? D(dmelt0) : 0.f;
    const float wM = min_w(tp.melt2, tp.SP1);
    const float dmelt = wM * dmelt2 + (1.f - wM) * dSP1;
    const float dMW1 = mw + dmelt;
    const float dSP2 = dSP1 - dmelt;
    // rf0 = CFR * CFMAX * (TTe - T)
    const float drf0 = (dp[HBV_P_CFR] * p[HBV_P_CFMAX] + p[HBV_P_CFR] * dp[HBV_P_CFMAX]) * (-tp.dT)
                     - p[HBV_P_CFR] * p[HBV_P_CFMAX] * ddT;
    const float drf2 = (tp.rf0 >= 0.f) ? D(drf0) : 0.f;
    const float wR = min_w(tp.rf2, tp.MW1);
    const float drf = wR * drf2 + (1.f - wR) * dMW1;
    const float dSP3 = dSP2 + drf;
    const float dMW2 = dMW1 - drf;
    const float dts0 = ID(dMW2 - dp[HBV_P_CWH] * tp.SP3 - p[HBV_P_CWH] * dSP3);
    dtosoil = (tp.ts0 >= 0.f) ? dts0 : 0.f;
    dSP = dSP3;
    dMW = dMW2 - D(dtosoil);
}

// soil routine + capillary rise.  dSLZ: tangent of the lower zone before the step; on exit the
// tangent after capillary rise (the response stage's input), as soil_fwd does with SLZ.
struct SoilTan { float recharge, excess, ET, ef, capillary, IE; };

template <int VAR, bool BETAET>
__device__ __forceinline__ void soil_tlm(float& SM, float& SLZ, float& dSM, float& dSLZ,
                                         const float (&p)[Traits<VAR>::NPAR], const float (&dp)[Traits<VAR>::NPAR],
                                         float RAIN, float tosoil, float PET, float dRAIN, float dtosoil, float dPET,
                                         const LaneConst& c, SoilOut& o, SoilTan& od, Tape& tp) {
    using TR = Traits<VAR>;
    const float dt = c.dt, inv_dt = c.inv_dt, nz = c.nearzero;
    auto D = [&](float x) { return TR::HOURLY ? x * dt : x; };
    auto ID = [&](float x) { return TR::HOURLY ? x * inv_dt : x; };
    soil_fwd<VAR, BETAET, true>(SM, SLZ, p, RAIN, tosoil, PET, c, o, tp);
    float sm = dSM, slz = dSLZ;
    if constexpr (TR::HOURLY) {
        sm = (tp.SMg >= nz) ? sm : 0.f;
        slz = (tp.SLZg >= nz) ? slz : 0.f;
    }
    const float FC = p[HBV_P_FC], dFC = dp[HBV_P_FC];
    // r = SM / FC ; sw0 = r^BETA ; sw = clamp(sw0, 0, 1)
    const float dr = fdiv(sm - tp.r * dFC, FC);
    float dsw0 = 0.f;
    if (tp.r > 0.f)
        dsw0 = fdiv(p[HBV_P_BETA] * tp.sw0, tp.r) * dr + tp.sw0 * flog(tp.r) * dp[HBV_P_BETA];
    const float dsw = (tp.sw0 >= 0.f && tp.sw0 <= 1.f) ? dsw0 : 0.f;
    const float dW = dRAIN + dtosoil;
    float drech, dSM1, dIE = 0.f;
    if constexpr (TR::HOURLY) {
        // s = clamp(r, 0, 0.99) ; fmin = FMIN*F0 ; pw = (1 - s)^ALPHA ; fcap = fmin + (F0 - fmin)*pw
        const float ds = (tp.r >= 0.f && tp.r <= 0.99f) ? dr : 0.f;
        const float dfmin = dp[HBV_P_FMIN] * p[HBV_P_F0] + p[HBV_P_FMIN] * dp[HBV_P_F0];
        const float dpw = -fdiv(p[HBV_P_ALPHA] * tp.pw, tp.s_base) * ds + tp.pw * flog(tp.s_base) * dp[HBV_P_ALPHA];
        const float dfcap = dfmin + (dp[HBV_P_F0] - dfmin) * tp.pw + (p[HBV_P_F0] - tp.fmin) * dpw;
        // infil = min(W, fcap) ; IE = max(W - fcap, 0)
        const float wW = min_w(tp.W, tp.fcap);
        const float dinfil = wW * dW + (1.f - wW) * dfcap;
        dIE = (tp.W - tp.fcap >= 0.f) ? dW - dfcap : 0.f;
        drech = dinfil * tp.sw + tp.infil * dsw;
        dSM1 = sm + (dinfil - drech) * dt;
    } else {
        drech = dW * tp.sw + tp.W * dsw;
        dSM1 = sm + dW - drech;
    }
    // excess = max((SM1 - FC)/dt, 0) ; SM2 = SM1 - excess*dt
    const float dexc = (tp.ex0 >= 0.f) ? ID(dSM1 - dFC) : 0.f;
    const float dSM2 = dSM1 - D(dexc);
    // ef0 = SM2 / (LP*FC) ; ef1 = ef0^BETAET ; ef = clamp(ef1, 0, 1)
    const float dden = dp[HBV_P_LP] * FC + p[HBV_P_LP] * dFC;
    const float def0 = fdiv(dSM2 - tp.ef0 * dden, tp.den);
    float def1 = def0;
    if constexpr (BETAET) {
        def1 = 0.f;
        if (tp.ef0 > 0.f)
            def1 = fdiv(p[HBV_P_BETAET] * tp.ef1, tp.ef0) * def0 + tp.ef1 * flog(tp.ef0) * dp[HBV_P_BETAET];
    }
    const float def = (tp.ef1 >= 0.f && tp.ef1 <= 1.f) ? def1 : 0.f;
    // et1 = PET*ef*dt ; et2 = min(SM2, et1) ; ET = et2/dt ; SMd = SM2 - ET*dt ; SM3 = max(SMd, nz)
    const float det1 = D(dPET * tp.ef + PET * def);
    const float wE = min_w(tp.SM2, tp.et1);
    const float det2 = wE * dSM2 + (1.f - wE) * det1;
    const float dET = ID(det2);
    const float dSMd = dSM2 - D(dET);
    const float dSM3 = (tp.SMd >= nz) ? dSMd : 0.f;
    float dSMf = dSM3, dSLZa = slz, dcap = 0.f;
    if constexpr (TR::CAP) {
        // r2 = SM3/FC ; capf = 1 - min(r2, 1) ; c1 = C*SLZ*capf*dt ; c2 = min(SLZ, c1) ; cap = c2/dt
        const float dr2 = fdiv(dSM3 - tp.r2 * dFC, FC);
        const float dcapf = (tp.r2 <= 1.0f) ? -dr2 : 0.f;
        const float dc1 = D(dp[HBV_P_C] * tp.SLZin * tp.capf + p[HBV_P_C] * slz * tp.capf
                            + p[HBV_P_C] * tp.SLZin * dcapf);
        const float wL = min_w(tp.SLZin, tp.c1);
        const float dc2 = wL * slz + (1.f - wL) * dc1;
        dcap = ID(dc2);
        const float dSMc = dSM3 + D(dcap);
        const float dSLZc = slz - D(dcap);
        dSMf = (tp.SMc >= nz) ? dSMc : 0.f;
        dSLZa = (tp.SLZc >= nz) ? dSLZc : 0.f;
    }
    dSM = dSMf;
    dSLZ = dSLZa;
    od.recharge = drech; od.excess = dexc; od.ET = dET; od.ef = def; od.capillary = dcap; od.IE = dIE;
}

// response boxes.  dSLZ enters as the tangent after capillary rise.
struct RespTan { float Q0, Q1, Q2, PERC; };

template <int VAR>
__device__ __forceinline__ void resp_tlm(float& SUZ, float& SLZ, float& dSUZ, float& dSLZ,
                                         const float (&p)[Traits<VAR>::NPAR], const float (&dp)[Traits<VAR>::NPAR],
                                         float recharge, float excess, float drech, float dexc,
                                         const LaneConst& c, RespOut& o, RespTan& od, Tape& tp) {
    using TR = Traits<VAR>;
    const float dt = c.dt, inv_dt = c.inv_dt, nz = c.nearzero;
    auto D = [&](float x) { return TR::HOURLY ? x * dt : x; };
    auto ID = [&](float x) { return TR::HOURLY ? x * inv_dt : x; };
    resp_fwd<VAR, true>(SUZ, SLZ, p, recharge, excess, c, o, tp);
    float suz = dSUZ;
    if constexpr (TR::HOURLY) suz = (tp.SUZg >= nz) ? suz : 0.f;
    const float dSUZ1 = suz + D(drech + dexc);
    const float dpc = D(dp[HBV_P_PERC]);
    const float wS = min_w(tp.SUZ1, tp.pc);
    const float dPERC = ID(wS * dSUZ1 + (1.f - wS) * dpc);
    const float dSUZ2 = dSUZ1 - D(dPERC);
    const float dq0a = dSUZ2 - dp[HBV_P_UZL];
    const float dQ0 = dp[HBV_P_K0] * fmaxf(tp.q0a, 0.f) + ((tp.q0a >= 0.f) ? p[HBV_P_K0] * dq0a : 0.f);
    const float dSUZ3 = dSUZ2 - D(dQ0);
    const float dQ1 = dp[HBV_P_K1] * tp.SUZ3 + p[HBV_P_K1] * dSUZ3;
    const float dSUZ4 = dSUZ3 - D(dQ1);
    const float dSLZ1 = dSLZ + D(dPERC);
    float dSLZ2 = dSLZ1;
    float SLZ2c = tp.SLZ2;
    if constexpr (TR::LAT) {
        float dlf = 0.f;
        if (c.Ac < 2500.f) {
            const bool inside = (tp.lfarg >= -1.f) && (tp.lfarg <= 1.f);
            dlf = inside ? -dp[HBV_P_AC] * (1.0f / 1000.f) : 0.f;
        }
        const float dLF = D(dlf * p[HBV_P_RT] + tp.lfval * dp[HBV_P_RT]);
        dSLZ2 = (tp.SLZ2 >= 0.f) ? dSLZ1 + dLF : 0.f;
        SLZ2c = fmaxf(tp.SLZ2, 0.f);
    }
    const float dQ2 = dp[HBV_P_K2] * SLZ2c + p[HBV_P_K2] * dSLZ2;
    dSUZ = dSUZ4;
    dSLZ = dSLZ2 - D(dQ2);
    od.Q0 = dQ0; od.Q1 = dQ1; od.Q2 = dQ2; od.PERC = dPERC;
}

// Tangent of one step: S = this evaluation's own copy of the states (updated in place), dS their
// tangents, dF the per-lane flux tangents in HBV_F_* order.  P, PET (and dP, dPET) as the step uses
// them (hourly: / dt).
template <int VAR, bool BETAET>
__device__ __forceinline__ void tangent_step(float (&S)[5], float (&dS)[5],
                                             const float (&p)[Traits<VAR>::NPAR], const float (&dp)[Traits<VAR>::NPAR],
                                             float P, float T, float PET, float dP, float dT, float dPET,
                                             const LaneConst& c, float (&dF)[HBV_MAX_FLUX]) {
    using TR = Traits<VAR>;
    Tape tp;
    float RAIN, tosoil, dRAIN, dtosoil;
    SoilOut so; SoilTan sd;
    RespOut ro; RespTan rd;
    snow_tlm<VAR>(S[0], S[1], dS[0], dS[1], p, dp, P, T, dP, dT, c, RAIN, tosoil, dRAIN, dtosoil, tp);
    soil_tlm<VAR, BETAET>(S[2], S[4], dS[2], dS[4], p, dp, RAIN, tosoil, PET, dRAIN, dtosoil, dPET, c, so, sd, tp);
    resp_tlm<VAR>(S[3], S[4], dS[3], dS[4], p, dp, so.recharge, so.excess, sd.recharge, sd.excess, c, ro, rd, tp);
    float dQsim = rd.Q0 + rd.Q1 + rd.Q2;
    if constexpr (TR::HOURLY) dQsim = dQsim + sd.IE;
    dF[HBV_F_QSIM] = dQsim; dF[HBV_F_Q0] = rd.Q0; dF[HBV_F_Q1] = rd.Q1; dF[HBV_F_Q2] = rd.Q2;
    dF[HBV_F_AET] = sd.ET; dF[HBV_F_SWE] = dS[0]; dF[HBV_F_RECHARGE] = sd.recharge; dF[HBV_F_EXCS] = sd.excess;
    dF[HBV_F_EVAPFACTOR] = sd.ef; dF[HBV_F_TOSOIL] = dtosoil; dF[HBV_F_PERC] = rd.PERC;
    dF[HBV_F_CAPILLARY] = sd.capillary;
}

// An opaque copy: the compiler cannot see that it equals its input, so nothing computed from it is
// merged with the same expression computed from the input.
__device__ __forceinline__ float opaque(float x) { asm volatile("" : "+f"(x)); return x; }

// Tangent-linear step: S / dS = states and their tangents (in place), F / dF = the per-lane fluxes
// and their tangents.  The primal is step_fwd exactly as the forward kernels run it: none of its
// intermediates gains a use that could change how the compiler contracts it into FMAs, so the
// primal states and fluxes equal K1's bit for bit.  The tangent stages re-evaluate the step from
// opaque copies of its inputs (the tape run) and push the tangents through.
template <int VAR, bool BETAET>
__device__ __forceinline__ void step_tlm(float (&S)[5], float (&dS)[5],
                                         const float (&p)[Traits<VAR>::NPAR], const float (&dp)[Traits<VAR>::NPAR],
                                         float P, float T, float PET, float dP, float dT, float dPET,
                                         const LaneConst& c, float (&F)[HBV_MAX_FLUX], float (&dF)[HBV_MAX_FLUX]) {
    constexpr int NPAR = Traits<VAR>::NPAR;
    float Sc[5], pc[NPAR];
#pragma unroll
    for (int s = 0; s < 5; ++s) Sc[s] = opaque(S[s]);
#pragma unroll
    for (int i = 0; i < NPAR; ++i) pc[i] = opaque(p[i]);
    const float Pc = opaque(P), Tc = opaque(T), PETc = opaque(PET);
    Tape tp0;
    step_fwd<VAR, BETAET, false>(S, p, P, T, PET, c, F, tp0);
    tangent_step<VAR, BETAET>(Sc, dS, pc, dp, Pc, Tc, PETc, dP, dT, dPET, c, dF);
}

}  // namespace hbv
