// uh_route.cu — K4: gamma unit hydrograph, causal per-basin convolution, BFI; and its adjoint.
//
// Replaces core/calc/uh_routing.py:5-22 (`uh_gamma`: relu, lgamma, exp, pow, sum, div, with the
// time vector built on the CPU and copied H2D), core/calc/uh_routing.py:25-57 (`uh_conv`: flip +
// grouped conv1d with groups = B, called 4x per forward at hbv.py:528-538) and the BFI reduction
// hbv.py:562-567 by two launches: `uh_weights` (one thread per basin) and `uh_conv` (one thread
// per (basin, time-chunk), all series in one pass, the <=16 UH taps and a 31-value sliding
// window in registers; adjacent threads are adjacent basins so every [T, B] row access is
// coalesced).  BFI partial sums go to a small workspace and are reduced deterministically.
//
// Note on uh_gamma: the factor 1/(Gamma(aa) theta^aa) is common to all taps and cancels in the
// normalisation w / w.sum(0); it is dropped here (same value up to rounding, no lgamma needed).
#include "hbv_common.cuh"

namespace hbv {

constexpr int MAXM = 16;   // register-window path handles lenF <= 16 (reference uses 15)
constexpr int RB = 128;    // basins per CTA

struct RDesc {
    int T, B, M, nser, apply_sigmoid, route_stride, bfi_num, bfi_den, nchunk, tch;
    float a_lo, a_span, b_lo, b_span, nearzero;
};

__device__ __forceinline__ void route_ab(const RDesc& d, const float* route, int b, float& aa,
                                         float& th, float& da_draw, float& db_draw) {
    const float r0 = __ldg(route + (int64_t)b * d.route_stride);
    const float r1 = __ldg(route + (int64_t)b * d.route_stride + 1);
    float s0 = r0, s1 = r1, g0 = 1.f, g1 = 1.f;
    if (d.apply_sigmoid) { s0 = sigmoidf_(r0); s1 = sigmoidf_(r1); g0 = s0 * (1.f - s0); g1 = s1 * (1.f - s1); }
    const float a = s0 * d.a_span + d.a_lo;
    const float bb = s1 * d.b_span + d.b_lo;
    aa = fmaxf(a, 0.f) + 0.1f;
    th = fmaxf(bb, 0.f) + 0.5f;
    da_draw = (a > 0.f ? 1.f : 0.f) * d.a_span * g0;   // relu'(0) = 0
    db_draw = (bb > 0.f ? 1.f : 0.f) * d.b_span * g1;
}

__global__ void uh_weights_kernel(const RDesc d, const float* __restrict__ route, float* __restrict__ uh) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= d.B) return;
    float aa, th, g0, g1;
    route_ab(d, route, b, aa, th, g0, g1);
    float w[MAXM];
    float sum = 0.f;
#pragma unroll
    for (int k = 0; k < MAXM; ++k) {
        w[k] = 0.f;
        if (k < d.M) {
            const float t = (float)k + 0.5f;
            w[k] = powf(t, aa - 1.f) * expf(-t / th);
            sum += w[k];
        }
    }
#pragma unroll
    for (int k = 0; k < MAXM; ++k)
        if (k < d.M) uh[(int64_t)k * d.B + b] = w[k] / sum;
}

// y[s][t][b] = sum_k uh[k][b] * x[s][t-k][b]; thread = (basin, time chunk)
__global__ void __launch_bounds__(RB)
uh_conv_kernel(const RDesc d, const float* __restrict__ uh, const float* __restrict__ x,
               int64_t x_stride, float* __restrict__ y, int64_t y_stride,
               float* __restrict__ bfi_ws) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    const int c = blockIdx.y;
    if (b >= d.B) return;
    const int ts = c * d.tch;
    const int te = min(d.T, ts + d.tch);
    float u[MAXM];
#pragma unroll
    for (int k = 0; k < MAXM; ++k) u[k] = (k < d.M) ? __ldg(uh + (int64_t)k * d.B + b) : 0.f;

    {
        const int s = blockIdx.z;     // one series per grid plane
        const float* xs = x + s * x_stride + b;
        float* ys = y + s * y_stride + b;
        float win[MAXM - 1 + MAXM];   // win[i] = x[tb - (MAXM-1) + i]
#pragma unroll
        for (int i = 0; i < MAXM - 1; ++i) {
            const int t = ts - (MAXM - 1) + i;
            win[i] = (t >= 0) ? __ldg(xs + (int64_t)t * d.B) : 0.f;
        }
        float acc_sum = 0.f;
        for (int tb = ts; tb < te; tb += MAXM) {
#pragma unroll
            for (int i = 0; i < MAXM; ++i) {
                const int t = tb + i;
                win[MAXM - 1 + i] = (t < te) ? __ldg(xs + (int64_t)t * d.B) : 0.f;
            }
#pragma unroll
            for (int i = 0; i < MAXM; ++i) {
                float acc = 0.f;
#pragma unroll
                for (int k = 0; k < MAXM; ++k) acc = fmaf(u[k], win[MAXM - 1 + i - k], acc);
                const int t = tb + i;
                if (t < te) { ys[(int64_t)t * d.B] = acc; acc_sum += acc; }
            }
#pragma unroll
            for (int i = 0; i < MAXM - 1; ++i) win[i] = win[MAXM + i];
        }
        if (bfi_ws != nullptr) {
            if (s == d.bfi_num) bfi_ws[((int64_t)0 * d.nchunk + c) * d.B + b] = acc_sum;
            if (s == d.bfi_den) bfi_ws[((int64_t)1 * d.nchunk + c) * d.B + b] = acc_sum;
        }
    }
}

__global__ void bfi_kernel(const RDesc d, const float* __restrict__ bfi_ws, float* __restrict__ bfi) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= d.B) return;
    float num = 0.f, den = 0.f;
#pragma unroll 8
    for (int c = 0; c < d.nchunk; ++c) {
        num += __ldg(bfi_ws + ((int64_t)0 * d.nchunk + c) * d.B + b);
        den += __ldg(bfi_ws + ((int64_t)1 * d.nchunk + c) * d.B + b);
    }
    bfi[b] = 100.f * (num / (den + d.nearzero));
}

// Adjoint conv: gx[s][t] = sum_k u[k] gy[s][t+k];  dU[k] += sum_t gy[s][t] x[s][t-k]
// gy = g_out (if present) + BFI term (constant in t).
__global__ void __launch_bounds__(RB)
uh_conv_bwd_kernel(const RDesc d, const float* __restrict__ uh, const float* __restrict__ x,
                   int64_t x_stride, const float* __restrict__ bfi_ws,
                   const float* __restrict__ g_out, int64_t g_stride, uint32_t g_mask,
                   const float* __restrict__ g_bfi, float* __restrict__ g_in, int64_t gin_stride,
                   float* __restrict__ ws) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    const int c = blockIdx.y;
    if (b >= d.B) return;
    const int ts = c * d.tch;
    const int te = min(d.T, ts + d.tch);
    float u[MAXM], dU[MAXM];
#pragma unroll
    for (int k = 0; k < MAXM; ++k) { u[k] = (k < d.M) ? __ldg(uh + (int64_t)k * d.B + b) : 0.f; dU[k] = 0.f; }

    float gnum = 0.f, gden = 0.f;
    if (g_bfi != nullptr) {
        float num = 0.f, den = 0.f;
        for (int cc = 0; cc < d.nchunk; ++cc) {
            num += bfi_ws[((int64_t)0 * d.nchunk + cc) * d.B + b];
            den += bfi_ws[((int64_t)1 * d.nchunk + cc) * d.B + b];
        }
        const float g = __ldg(g_bfi + b) * 100.f;
        const float dn = den + d.nearzero;
        gnum = g / dn;
        gden = -g * num / (dn * dn);
    }

    for (int s = 0; s < d.nser; ++s) {
        const bool has_g = (g_mask >> s) & 1u;
        // a series with neither an upstream gradient nor a BFI term has an all-zero adjoint:
        // its g_in plane is left unwritten (the caller skips it, see hbv_b200.h)
        if (!has_g && !(g_bfi != nullptr && (s == d.bfi_num || s == d.bfi_den))) continue;
        const float cst = (s == d.bfi_num ? gnum : 0.f) + (s == d.bfi_den ? gden : 0.f);
        const float* gs = g_out ? g_out + s * g_stride + b : nullptr;
        const float* xs = x + s * x_stride + b;
        float* gxs = g_in + s * gin_stride + b;
        auto gy = [&](int t) -> float {
            if (t >= d.T) return 0.f;
            return (has_g ? __ldg(gs + (int64_t)t * d.B) : 0.f) + cst;
        };
        // wing[i] = gy[tb + i], i in [0, 2*MAXM-1)
        float wing[MAXM + MAXM - 1];
        float winx[MAXM - 1 + MAXM];   // winx[i] = x[tb - (MAXM-1) + i]
#pragma unroll
        for (int i = 0; i < MAXM - 1; ++i) {
            const int t = ts - (MAXM - 1) + i;
            winx[i] = (t >= 0) ? __ldg(xs + (int64_t)t * d.B) : 0.f;
        }
#pragma unroll
        for (int i = 0; i < MAXM; ++i) wing[i] = gy(ts + i);
        for (int tb = ts; tb < te; tb += MAXM) {
#pragma unroll
            for (int i = 0; i < MAXM - 1; ++i) wing[MAXM + i] = gy(tb + MAXM + i);
#pragma unroll
            for (int i = 0; i < MAXM; ++i) {
                const int t = tb + i;
                winx[MAXM - 1 + i] = (t < te) ? __ldg(xs + (int64_t)t * d.B) : 0.f;
            }
#pragma unroll
            for (int i = 0; i < MAXM; ++i) {
                const int t = tb + i;
                float acc = 0.f;
#pragma unroll
                for (int k = 0; k < MAXM; ++k) acc = fmaf(u[k], wing[i + k], acc);
                if (t < te) {
                    gxs[(int64_t)t * d.B] = acc;
                    const float g = wing[i];
#pragma unroll
                    for (int k = 0; k < MAXM; ++k) dU[k] = fmaf(g, winx[MAXM - 1 + i - k], dU[k]);
                }
            }
#pragma unroll
            for (int i = 0; i < MAXM - 1; ++i) wing[i] = wing[MAXM + i];
            wing[MAXM - 1] = gy(tb + 2 * MAXM - 1);
#pragma unroll
            for (int i = 0; i < MAXM - 1; ++i) winx[i] = winx[MAXM + i];
        }
    }
#pragma unroll
    for (int k = 0; k < MAXM; ++k)
        if (k < d.M) ws[((int64_t)k * d.nchunk + c) * d.B + b] = dU[k];
}

// reduce dU partials over chunks, push through the normalised gamma pdf to (route_a, route_b).
// 16 threads per basin (one per tap): the chunk sums are independent loads, the five per-basin
// moments are reduced with shuffles inside the 16-lane group.
__global__ void __launch_bounds__(128)
uh_param_bwd_kernel(const RDesc d, const float* __restrict__ route,
                    const float* __restrict__ uh, const float* __restrict__ ws,
                    float* __restrict__ g_route) {
    const int k = threadIdx.x & (MAXM - 1);
    const int b_raw = blockIdx.x * (blockDim.x / MAXM) + threadIdx.x / MAXM;
    const int b = min(b_raw, d.B - 1);
    float g = 0.f, u = 0.f;
    if (k < d.M) {
        const float* w = ws + (int64_t)k * d.nchunk * d.B + b;
#pragma unroll 8
        for (int c = 0; c < d.nchunk; ++c) g += __ldg(w + (int64_t)c * d.B);
        u = __ldg(uh + (int64_t)k * d.B + b);
    }
    const float t = (float)k + 0.5f;
    const float L = logf(t);
    float mL = u * L, mT = u * t;     // sum_j u_j ln t_j, sum_j u_j t_j
    float sL = g * u * L, sT = g * u * t, s0 = g * u;
#pragma unroll
    for (int o = MAXM / 2; o > 0; o >>= 1) {
        mL += __shfl_xor_sync(0xffffffffu, mL, o);
        mT += __shfl_xor_sync(0xffffffffu, mT, o);
        sL += __shfl_xor_sync(0xffffffffu, sL, o);
        sT += __shfl_xor_sync(0xffffffffu, sT, o);
        s0 += __shfl_xor_sync(0xffffffffu, s0, o);
    }
    if (k != 0 || b_raw >= d.B) return;
    float aa, th, da_draw, db_draw;
    route_ab(d, route, b, aa, th, da_draw, db_draw);
    // du_k/daa = u_k (L_k - mL);  du_k/dth = u_k (t_k - mT) / th^2
    const float gaa = sL - s0 * mL;
    const float gth = (sT - s0 * mT) / (th * th);
    g_route[(int64_t)b * d.route_stride] = gaa * da_draw;
    g_route[(int64_t)b * d.route_stride + 1] = gth * db_draw;
}

// ---- K4t: tangent of the routing ------------------------------------------------------------
// y_t[s][t] = sum_k uh[k] x_t[s][t-k] + uh_t[k] x[s][t-k], with the tangent of the normalised
// gamma UH  uh_t[k] = uh[k] ((ln t_k - sum_j uh_j ln t_j) aa_t + (t_k - sum_j uh_j t_j) th_t / th^2)
// (the closed form uh_param_bwd_kernel transposes).  Same (basin, time chunk) threads and register
// windows as uh_conv_kernel, one series per grid plane; BFI partial sums of the tangent planes go
// to bfi_ws_t.
__global__ void __launch_bounds__(RB)
uh_conv_tlm_kernel(const RDesc d, const float* __restrict__ route, const float* __restrict__ route_t,
                   const float* __restrict__ uh, const float* __restrict__ x, int64_t x_stride,
                   const float* __restrict__ xt, int64_t xt_stride, float* __restrict__ yt, int64_t yt_stride,
                   float* __restrict__ bfi_ws_t) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    const int c = blockIdx.y;
    if (b >= d.B) return;
    const int ts = c * d.tch;
    const int te = min(d.T, ts + d.tch);
    float aa, th, da_draw, db_draw;
    route_ab(d, route, b, aa, th, da_draw, db_draw);
    float ra_t = 0.f, rb_t = 0.f;
    if (route_t != nullptr) {
        ra_t = __ldg(route_t + (int64_t)b * d.route_stride);
        rb_t = __ldg(route_t + (int64_t)b * d.route_stride + 1);
    }
    const float aa_t = da_draw * ra_t;
    const float th_t = db_draw * rb_t / (th * th);
    float u[MAXM], ud[MAXM];
    float mL = 0.f, mT = 0.f;
#pragma unroll
    for (int k = 0; k < MAXM; ++k) {
        u[k] = (k < d.M) ? __ldg(uh + (int64_t)k * d.B + b) : 0.f;
        const float tk = (float)k + 0.5f;
        mL += u[k] * logf(tk);
        mT += u[k] * tk;
    }
#pragma unroll
    for (int k = 0; k < MAXM; ++k) {
        const float tk = (float)k + 0.5f;
        ud[k] = u[k] * ((logf(tk) - mL) * aa_t + (tk - mT) * th_t);
    }

    const int s = blockIdx.z;
    const float* xs = x + s * x_stride + b;
    const float* xts = xt + s * xt_stride + b;
    float* ys = yt + s * yt_stride + b;
    float win[MAXM - 1 + MAXM], wint[MAXM - 1 + MAXM];
#pragma unroll
    for (int i = 0; i < MAXM - 1; ++i) {
        const int t = ts - (MAXM - 1) + i;
        win[i] = (t >= 0) ? __ldg(xs + (int64_t)t * d.B) : 0.f;
        wint[i] = (t >= 0) ? __ldg(xts + (int64_t)t * d.B) : 0.f;
    }
    float acc_sum = 0.f;
    for (int tb = ts; tb < te; tb += MAXM) {
#pragma unroll
        for (int i = 0; i < MAXM; ++i) {
            const int t = tb + i;
            win[MAXM - 1 + i] = (t < te) ? __ldg(xs + (int64_t)t * d.B) : 0.f;
            wint[MAXM - 1 + i] = (t < te) ? __ldg(xts + (int64_t)t * d.B) : 0.f;
        }
#pragma unroll
        for (int i = 0; i < MAXM; ++i) {
            float acc = 0.f;
#pragma unroll
            for (int k = 0; k < MAXM; ++k) {
                acc = fmaf(u[k], wint[MAXM - 1 + i - k], acc);
                acc = fmaf(ud[k], win[MAXM - 1 + i - k], acc);
            }
            const int t = tb + i;
            if (t < te) { ys[(int64_t)t * d.B] = acc; acc_sum += acc; }
        }
#pragma unroll
        for (int i = 0; i < MAXM - 1; ++i) { win[i] = win[MAXM + i]; wint[i] = wint[MAXM + i]; }
    }
    if (bfi_ws_t != nullptr) {
        if (s == d.bfi_num) bfi_ws_t[((int64_t)0 * d.nchunk + c) * d.B + b] = acc_sum;
        if (s == d.bfi_den) bfi_ws_t[((int64_t)1 * d.nchunk + c) * d.B + b] = acc_sum;
    }
}

// BFI tangent: the primal sums reduced exactly as bfi_kernel does, the tangent sums the same way
__global__ void bfi_tlm_kernel(const RDesc d, const float* __restrict__ bfi_ws, const float* __restrict__ bfi_ws_t,
                               float* __restrict__ bfi_t) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= d.B) return;
    float num = 0.f, den = 0.f, num_t = 0.f, den_t = 0.f;
#pragma unroll 8
    for (int c = 0; c < d.nchunk; ++c) {
        num += __ldg(bfi_ws + ((int64_t)0 * d.nchunk + c) * d.B + b);
        den += __ldg(bfi_ws + ((int64_t)1 * d.nchunk + c) * d.B + b);
        num_t += __ldg(bfi_ws_t + ((int64_t)0 * d.nchunk + c) * d.B + b);
        den_t += __ldg(bfi_ws_t + ((int64_t)1 * d.nchunk + c) * d.B + b);
    }
    const float D = den + d.nearzero;
    bfi_t[b] = 100.f * ((num_t * D - num * den_t) / (D * D));
}

// threads (= basins) per CTA of the conv kernels: small CTAs for small B so the (basin-block,
// chunk) grid still covers the SMs
static int route_block(int B) { return B >= 8192 ? RB : (B >= 2048 ? 64 : 32); }

static int make_rdesc(const hbv_route_desc_t* r, RDesc& d) {
    if (!r) { set_error("null route desc"); return HBV_E_NULL; }
    if (r->abi_version != HBV_B200_ABI_VERSION) { set_error("ABI version mismatch"); return HBV_E_ABI; }
    if (r->T <= 0 || r->B <= 0 || r->nser <= 0 || r->nser > 8 || r->lenF <= 0) { set_error("bad route shape"); return HBV_E_SHAPE; }
    d.T = r->T; d.B = r->B; d.M = r->lenF < r->T ? r->lenF : r->T;
    if (d.M > MAXM) { set_error("lenF > 16 not supported by the register-window routing kernel"); return HBV_E_SHAPE; }
    d.nser = r->nser; d.apply_sigmoid = r->apply_sigmoid; d.route_stride = r->route_stride;
    d.bfi_num = r->bfi_num; d.bfi_den = r->bfi_den;
    d.a_lo = r->a_lo; d.a_span = r->a_hi - r->a_lo; d.b_lo = r->b_lo; d.b_span = r->b_hi - r->b_lo;
    d.nearzero = r->nearzero;
    d.nchunk = hbv_b200_route_chunks(r->T, r->B);
    d.tch = (r->T + d.nchunk - 1) / d.nchunk;
    d.tch = ((d.tch + MAXM - 1) / MAXM) * MAXM;
    return 0;
}

}  // namespace hbv

using namespace hbv;

extern "C" int hbv_b200_route_chunks(int32_t T, int32_t B) {
    if (T <= 0 || B <= 0) return 1;
    // one thread per (basin, time chunk): enough chunks to fill the 148 SMs (~1.5k threads
    // each); a chunk is at least one MAXM-step block (the lenF-1 halo re-read then doubles the
    // reads, which only small problems — where a thread's serial chunk is the whole latency of
    // the launch — ever reach: C2 uses 46 chunks of 16 steps)
    const long long target = 148LL * 1536;
    int want = (int)((target + B - 1) / B);
    int maxc = (T + MAXM - 1) / MAXM;
    if (want > maxc) want = maxc;
    if (want < 1) want = 1;
    // chunk length is rounded up to a multiple of MAXM: recompute the chunk count it implies
    int tch = (T + want - 1) / want;
    tch = ((tch + MAXM - 1) / MAXM) * MAXM;
    return (T + tch - 1) / tch;
}

extern "C" int hbv_b200_route_fwd(const hbv_route_desc_t* desc, const float* route,
                                  const float* q_in, int64_t q_stride, float* q_out,
                                  int64_t out_stride, float* uh, float* bfi, float* bfi_ws,
                                  void* stream) {
    RDesc d;
    int rc = make_rdesc(desc, d);
    if (rc) return rc;
    if (!route || !q_in || !q_out || !uh || (bfi && !bfi_ws)) { set_error("null pointer"); return HBV_E_NULL; }
    cudaStream_t st = (cudaStream_t)stream;
    uh_weights_kernel<<<(d.B + 127) / 128, 128, 0, st>>>(d, route, uh);
    const int rb = route_block(d.B);
    dim3 grid((d.B + rb - 1) / rb, d.nchunk, d.nser);
    uh_conv_kernel<<<grid, rb, 0, st>>>(d, uh, q_in, q_stride, q_out, out_stride, bfi ? bfi_ws : nullptr);
    count_launch(2);
    if (bfi) { bfi_kernel<<<(d.B + 127) / 128, 128, 0, st>>>(d, bfi_ws, bfi); count_launch(); }
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) set_error(cudaGetErrorString(e));
    return (int)e;
}

extern "C" int hbv_b200_route_bwd(const hbv_route_desc_t* desc, const float* route,
                                  const float* q_in, int64_t q_stride, const float* q_out,
                                  int64_t out_stride, const float* uh, const float* bfi_ws,
                                  const float* g_out, int64_t g_stride, uint32_t g_out_mask,
                                  const float* g_bfi, float* g_in, int64_t gin_stride,
                                  float* g_route, float* ws, void* stream) {
    (void)q_out; (void)out_stride;
    RDesc d;
    int rc = make_rdesc(desc, d);
    if (rc) return rc;
    if (!route || !q_in || !uh || !g_in || !g_route || !ws || (g_bfi && !bfi_ws) || (g_out_mask && !g_out)) {
        set_error("null pointer"); return HBV_E_NULL;
    }
    cudaStream_t st = (cudaStream_t)stream;
    const int rb = route_block(d.B);
    dim3 grid((d.B + rb - 1) / rb, d.nchunk);
    uh_conv_bwd_kernel<<<grid, rb, 0, st>>>(d, uh, q_in, q_stride, bfi_ws, g_out, g_stride, g_out_mask,
                                            g_bfi, g_in, gin_stride, ws);
    const int bpb = 128 / MAXM;
    uh_param_bwd_kernel<<<(d.B + bpb - 1) / bpb, 128, 0, st>>>(d, route, uh, ws, g_route);
    count_launch(2);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) set_error(cudaGetErrorString(e));
    return (int)e;
}

extern "C" int hbv_b200_route_tlm(const hbv_route_desc_t* desc, const float* route, const float* route_t,
                                  const float* q_in, int64_t q_stride, const float* q_in_t, int64_t qt_stride,
                                  const float* uh, const float* bfi_ws, float* q_out_t, int64_t out_stride,
                                  float* bfi_t, float* bfi_ws_t, void* stream) {
    RDesc d;
    int rc = make_rdesc(desc, d);
    if (rc) return rc;
    if (!route || !q_in || !q_in_t || !uh || !q_out_t || (bfi_t && (!bfi_ws || !bfi_ws_t))) {
        set_error("null pointer"); return HBV_E_NULL;
    }
    cudaStream_t st = (cudaStream_t)stream;
    const int rb = route_block(d.B);
    dim3 grid((d.B + rb - 1) / rb, d.nchunk, d.nser);
    uh_conv_tlm_kernel<<<grid, rb, 0, st>>>(d, route, route_t, uh, q_in, q_stride, q_in_t, qt_stride,
                                            q_out_t, out_stride, bfi_t ? bfi_ws_t : nullptr);
    count_launch();
    if (bfi_t) { bfi_tlm_kernel<<<(d.B + 127) / 128, 128, 0, st>>>(d, bfi_ws, bfi_ws_t, bfi_t); count_launch(); }
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) set_error(cudaGetErrorString(e));
    return (int)e;
}
