// hbv_tlm.cu — K1t: tangent-linear (forward-mode) HBV recurrence, the JVP of K1.
//
// One thread per (basin, component) lane, as in the generic K1 (hbv_fwd.cu): the 5 states and
// their 5 tangents stay in registers for all T steps, parameters are resolved per lane (sigmoid +
// descale, tangent through s (1 - s) (hi - lo)), dropped dynamic parameters read row T-1 for the
// primal and the tangent alike, and the nmul aggregation of the primal and tangent flux series is
// the shared-memory transpose-reduce of K1 (a chunk of TC steps per pass; with muwts the tangent
// of the weighted streamflow is sum_j (mu_dot Q + mu Q_dot)).  Inputs of step t + 1 are loaded
// while step t computes (a register double buffer; the tangents double the bytes of K1's).
// The primal is evaluated with K1's own step code (step_tlm, hbv_tlm.cuh), so the optional primal
// outputs equal the generic K1's.  Without flux outputs (states-only mode) the kernel skips the tile entirely.
#include <atomic>
#include "hbv_tlm.cuh"

namespace hbv {

constexpr int TLM_TC = 4;        // time steps per output chunk
constexpr int TLM_NFP = 24;      // floats per lane per step in the staging tile: 12 primal + 12 tangent
__host__ __device__ inline int tlm_bstride(int nmul) { return nmul * TLM_NFP + 4; }

struct TlmPtrs {
    const float* forcing; const float* dyn; const float* sta; const uint8_t* drop;
    const float* attrs; const float* muwts; const float* state_in;
    const float* forcing_t; const float* dyn_t; const float* sta_t; const float* muwts_t;
    const float* state_in_t;
    float* flux_t[HBV_MAX_FLUX]; float* state_out_t; float* series_t;
    float* flux[HBV_MAX_FLUX]; float* state_out;
};

// inputs of one step: forcings, the raw values of the dynamic parameters, and their tangents
template <int NPAR>
struct TlmIn { float P, T, PET, dP, dT, dPET; float raw[NPAR], draw[NPAR]; };

template <int NPAR>
__device__ __forceinline__ void tlm_load(const KDesc& d, const TlmPtrs& io, int t, int b, int j,
                                         uint32_t dynmask, TlmIn<NPAR>& in) {
    const int64_t fo = ((int64_t)t * d.B + b) * d.nvar;
    in.P = __ldg(io.forcing + fo + d.i_prcp);
    in.T = __ldg(io.forcing + fo + d.i_tmean);
    in.PET = __ldg(io.forcing + fo + d.i_pet);
    if (io.forcing_t) {
        in.dP = __ldg(io.forcing_t + fo + d.i_prcp);
        in.dT = __ldg(io.forcing_t + fo + d.i_tmean);
        in.dPET = __ldg(io.forcing_t + fo + d.i_pet);
    } else {
        in.dP = in.dT = in.dPET = 0.f;
    }
    const int64_t ro = ((int64_t)t * d.B + b) * d.dyn_ncol + j;
#pragma unroll
    for (int i = 0; i < NPAR; ++i) {
        in.raw[i] = 0.f; in.draw[i] = 0.f;
        if ((dynmask >> i) & 1u) {
            in.raw[i] = __ldg(io.dyn + ro + d.col[i]);
            if (io.dyn_t) in.draw[i] = __ldg(io.dyn_t + ro + d.col[i]);
        }
    }
}

template <int VAR, bool BETAET, bool WF>
__global__ void __launch_bounds__(256)
hbv_tlm_kernel(const KDesc d, const TlmPtrs io) {
    using TR = Traits<VAR>;
    constexpr int NPAR = TR::NPAR;
    extern __shared__ __align__(16) float smem[];

    const int tid = threadIdx.x;
    const int NT = blockDim.x;
    const int nmul = d.nmul;
    const int bl = tid / nmul;
    const int j = tid - bl * nmul;
    const int b_raw = blockIdx.x * d.BPB + bl;
    const bool valid = b_raw < d.B;
    const int b = valid ? b_raw : d.B - 1;
    const int64_t lane = (int64_t)b * nmul + j;
    const int64_t nlane = (int64_t)d.B * nmul;

    LaneConst lc;
    lc.nearzero = d.nearzero; lc.dt = d.dt; lc.inv_dt = d.inv_dt;
    lc.Ac = 0.f; lc.Elev = 0.f; lc.lfexp = 0.f;
    if constexpr (TR::LAT) init_lane_const(lc, __ldg(io.attrs + b), __ldg(io.attrs + d.B + b));

    // ---- parameters and their tangents: resolve sources, descale the time-invariant ones -----
    float p[NPAR], dp[NPAR];
    uint32_t dynmask = 0;
    const int64_t last = ((int64_t)(d.T - 1) * d.B + b) * d.dyn_ncol + j;
#pragma unroll
    for (int i = 0; i < NPAR; ++i) {
        p[i] = 0.f; dp[i] = 0.f;
        if (i < d.n_par) {
            int src = d.src[i];
            if (src == HBV_SRC_DYN_T && io.drop != nullptr && io.drop[(int64_t)i * d.B + b]) src = HBV_SRC_DYN_LAST;
            if (src == HBV_SRC_DYN_T) {
                dynmask |= (1u << i);
            } else {
                float raw, rt = 0.f;
                if (src == HBV_SRC_STA) {
                    const int64_t o = (int64_t)b * d.sta_ncol + d.col[i] + j;
                    raw = __ldg(io.sta + o);
                    if (io.sta_t) rt = __ldg(io.sta_t + o);
                } else {
                    raw = __ldg(io.dyn + last + d.col[i]);
                    if (io.dyn_t) rt = __ldg(io.dyn_t + last + d.col[i]);
                }
                // primal as K1 descales it; the derivative from an opaque copy of the raw value, so
                // that s * (hi - lo) is not shared with the primal's FMA (see step_tlm)
                p[i] = descale(d, i, raw);
                dp[i] = descale_grad(d, i, opaque(raw)) * rt;
            }
        }
    }

    float S[5], dS[5];
#pragma unroll
    for (int s = 0; s < 5; ++s) {
        S[s] = __ldg(io.state_in + s * nlane + lane);
        dS[s] = io.state_in_t ? __ldg(io.state_in_t + s * nlane + lane) : 0.f;
    }
    const float* mu_lane = io.muwts ? io.muwts + lane : nullptr;
    const float* mut_lane = io.muwts_t ? io.muwts_t + lane : nullptr;

    // ---- output staging tile: [tc][basin][component][24] ----------------------------------------
    const int bstride = tlm_bstride(nmul);
    float* my_slot = smem + bl * bstride + j * TLM_NFP;
    const int tstride_s = d.BPB * bstride;
    const float inv_nmul = 1.0f / (float)nmul;
    const int items = TLM_TC * d.BPB * 6;
    auto reduce_item = [&](int it, int t0, int tcn) {
        const int q = it % 6;          // quads 0..2: primal fluxes, 3..5: tangents
        const int r = it / 6;
        const int bl2 = r % d.BPB;
        const int tc = r / d.BPB;
        const int bb = blockIdx.x * d.BPB + bl2;
        if (bb >= d.B || tc >= tcn) return;
        const bool tan = q >= 3;
        const int f0 = (tan ? q - 3 : q) * 4;
        float* const* out = tan ? io.flux_t : io.flux;
        if (!out[f0] && !out[f0 + 1] && !out[f0 + 2] && !out[f0 + 3]) return;
        const float* src = smem + tc * tstride_s + bl2 * bstride + q * 4;
        float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
        for (int jj = 0; jj < nmul; ++jj) {
            const float4 v = *reinterpret_cast<const float4*>(src + jj * TLM_NFP);
            acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w;
        }
        const float s0 = (f0 == 0 && io.muwts != nullptr) ? 1.0f : inv_nmul;
        const int64_t o = (int64_t)(t0 + tc) * d.B + bb;
        if (out[f0 + 0]) out[f0 + 0][o] = acc.x * s0;
        if (out[f0 + 1]) out[f0 + 1][o] = acc.y * inv_nmul;
        if (out[f0 + 2]) out[f0 + 2][o] = acc.z * inv_nmul;
        if (out[f0 + 3]) out[f0 + 3][o] = acc.w * inv_nmul;
    };

    TlmIn<NPAR> cur, nxt;
    tlm_load<NPAR>(d, io, 0, b, j, dynmask, cur);
    for (int t0 = 0; t0 < d.T; t0 += TLM_TC) {
        const int tcn = min(TLM_TC, d.T - t0);
        for (int u = 0; u < tcn; ++u) {
            const int t = t0 + u;
            if (t + 1 < d.T) tlm_load<NPAR>(d, io, t + 1, b, j, dynmask, nxt);
#pragma unroll
            for (int i = 0; i < NPAR; ++i)
                if ((dynmask >> i) & 1u) {
                    p[i] = descale(d, i, cur.raw[i]);          // as K1 (ring_apply_dyn)
                    dp[i] = descale_grad(d, i, opaque(cur.raw[i])) * cur.draw[i];
                }
            float P = cur.P, PET = cur.PET, dP = cur.dP, dPET = cur.dPET;
            if constexpr (TR::HOURLY) { P = P * d.inv_dt; PET = PET * d.inv_dt; dP = dP * d.inv_dt; dPET = dPET * d.inv_dt; }
            float F[HBV_MAX_FLUX], dF[HBV_MAX_FLUX];
            step_tlm<VAR, BETAET>(S, dS, p, dp, P, cur.T, PET, dP, cur.dT, dPET, lc, F, dF);
            if (io.series_t != nullptr && valid) {
                float* ss = io.series_t + (int64_t)t * nlane + lane;
#pragma unroll
                for (int s = 0; s < 5; ++s) ss[(int64_t)s * d.T * nlane] = dS[s];
            }
            if constexpr (WF) {
                if (mu_lane) {
                    const float m = __ldg(mu_lane + (int64_t)t * d.muwts_t_stride);
                    const float dm = mut_lane ? __ldg(mut_lane + (int64_t)t * d.muwts_t_stride) : 0.f;
                    dF[HBV_F_QSIM] = dF[HBV_F_QSIM] * m + F[HBV_F_QSIM] * dm;
                    F[HBV_F_QSIM] *= m;
                }
                float4* slot = reinterpret_cast<float4*>(my_slot + u * tstride_s);
                slot[0] = make_float4(F[0], F[1], F[2], F[3]);
                slot[1] = make_float4(F[4], F[5], F[6], F[7]);
                slot[2] = make_float4(F[8], F[9], F[10], TR::NFLUX > 11 ? F[11] : 0.f);
                slot[3] = make_float4(dF[0], dF[1], dF[2], dF[3]);
                slot[4] = make_float4(dF[4], dF[5], dF[6], dF[7]);
                slot[5] = make_float4(dF[8], dF[9], dF[10], TR::NFLUX > 11 ? dF[11] : 0.f);
            }
            cur = nxt;
        }
        if constexpr (WF) {
            __syncthreads();
            for (int it = tid; it < items; it += NT) reduce_item(it, t0, tcn);
            __syncthreads();
        }
    }
    if (valid) {
#pragma unroll
        for (int s = 0; s < 5; ++s) {
            if (io.state_out != nullptr) io.state_out[s * nlane + lane] = S[s];
            if (io.state_out_t != nullptr) io.state_out_t[s * nlane + lane] = dS[s];
        }
    }
}

template <int VAR, bool BETAET, bool WF>
static int launch_tlm(const KDesc& d, const TlmPtrs& io, cudaStream_t st) {
    const int NT = d.BPB * d.nmul;
    const int grid = (d.B + d.BPB - 1) / d.BPB;
    const size_t smem = WF ? (size_t)TLM_TC * d.BPB * tlm_bstride(d.nmul) * sizeof(float) : 0;
    auto k = hbv_tlm_kernel<VAR, BETAET, WF>;
    cudaError_t e;
    static std::atomic<int> optin[HBV_MAX_DEVICES];
    int dev = 0;
    cudaGetDevice(&dev);
    if (smem > 48 * 1024) {
        if (smem > 160 * 1024) { set_error("nmul too large for the tangent kernel's output tile"); return HBV_E_NMUL; }
        if (dev >= HBV_MAX_DEVICES || optin[dev].load(std::memory_order_acquire) == 0) {
            e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, 160 * 1024);
            if (e != cudaSuccess) { set_error(cudaGetErrorString(e)); return (int)e; }
            if (dev < HBV_MAX_DEVICES) optin[dev].store(1, std::memory_order_release);
        }
    }
    k<<<grid, NT, smem, st>>>(d, io);
    count_launch();
    e = cudaGetLastError();
    if (e != cudaSuccess) set_error(cudaGetErrorString(e));
    return (int)e;
}

template <int VAR, bool BETAET>
static int launch_tlm_v(const KDesc& d, const TlmPtrs& io, bool wf, cudaStream_t st) {
    return wf ? launch_tlm<VAR, BETAET, true>(d, io, st) : launch_tlm<VAR, BETAET, false>(d, io, st);
}

int make_kdesc(const hbv_desc_t* desc, KDesc& d);  // hbv_cabi.cu

int tlm_dispatch(const hbv_desc_t* desc, const hbv_tlm_io_t* io, cudaStream_t st) {
    KDesc d;
    const int rc = make_kdesc(desc, d);
    if (rc) return rc;
    TlmPtrs p;
    p.forcing = io->forcing; p.dyn = io->dyn; p.sta = io->sta; p.drop = io->drop;
    p.attrs = io->attrs; p.muwts = io->muwts; p.state_in = io->state_in;
    p.forcing_t = io->forcing_t; p.dyn_t = io->dyn_t; p.sta_t = io->sta_t;
    p.muwts_t = io->muwts ? io->muwts_t : nullptr; p.state_in_t = io->state_in_t;
    p.state_out_t = io->state_out_t; p.series_t = io->series_t; p.state_out = io->state_out;
    bool wf = false;
    for (int f = 0; f < HBV_MAX_FLUX; ++f) {
        p.flux_t[f] = io->flux_t[f]; p.flux[f] = io->flux[f];
        wf |= (io->flux_t[f] != nullptr) || (io->flux[f] != nullptr);
    }
    switch (desc->variant) {
        case HBV_VARIANT_HBV:
            return desc->betaet ? launch_tlm_v<HBV_VARIANT_HBV, true>(d, p, wf, st)
                                : launch_tlm_v<HBV_VARIANT_HBV, false>(d, p, wf, st);
        case HBV_VARIANT_HBV11P: return launch_tlm_v<HBV_VARIANT_HBV11P, true>(d, p, wf, st);
        case HBV_VARIANT_HBV2: return launch_tlm_v<HBV_VARIANT_HBV2, true>(d, p, wf, st);
        case HBV_VARIANT_HOURLY: return launch_tlm_v<HBV_VARIANT_HOURLY, true>(d, p, wf, st);
    }
    set_error("unknown variant");
    return HBV_E_VARIANT;
}

}  // namespace hbv
