// pair_route.cu — K4': distributed (gage, unit) pair routing of hbv_2_hourly, forward + adjoint.
//
// Replaces Hbv_2_hourly.distr_routing / _frac_shift1d (models/hbv/hbv_2_hourly.py:800-897): the
// reference gathers the area-weighted runoff of every (gage, unit) pair into a [T, n_pairs]
// tensor, builds a 72-tap gamma UH per pair (uh_gamma), shifts it by a fractional lag
// (two torch.gather + masks), convolves with a grouped conv1d (groups = n_pairs), scatter_adds
// the pairs to their gages and divides by the upstream area.  Here:
//   pair_uh        one thread per pair: normalised gamma pdf + fractional shift -> uh[M][P]
//   pair_conv      shared-memory-staged convolution, one CTA = 32 pairs x 64 time steps; the
//                  gather x[t][p] = Qs[t][unit(p)] * area(unit(p)) is fused into the tile load
//   seg_sum        deterministic segmented sum (CSR by gage / CSC by unit) + scaling
//   pair_conv_bwd  adjoint conv (gradient gather g[t][gage(p)] / denom fused into the tile load)
//                  + per-tap dot products for d/dUH, reduced over time chunks
//   pair_uh_bwd    d/dUH -> (route_a, route_b, route_tau) through the shift and the gamma pdf
// The same conv kernels serve the plain per-unit routing of the hourly model (lenF = 72, identity
// gather), which the 16-tap register-window kernel of uh_route.cu cannot hold.
#include "hbv_common.cuh"

namespace hbv {

constexpr int PM = 128;       // max taps
constexpr int PTT = 128;      // time steps per tile
constexpr int PPB = 32;       // pairs per CTA (one per lane)
constexpr int PTY = 8;        // time threads per pair
constexpr int PR = PTT / PTY; // conv: consecutive outputs per thread (register window)
constexpr int DK = 8;         // d/dUH: consecutive taps per work item (register window)
constexpr int DTS = 32;       // d/dUH: time steps per work item
constexpr int DNS = PTT / DTS;

struct PDesc {
    int T, P, M, lag_uh, tchunk, nchunk;
    float a_lo, a_span, b_lo, b_span, t_lo, t_span;
};

__host__ __device__ constexpr int round_up(int x, int m) { return (x + m - 1) / m * m; }

__device__ __forceinline__ float gamma_w(float t, float aa, float th) {
    return powf(t, aa - 1.f) * expf(-t / th);
}

// uh[k][p] = fractional shift of the normalised gamma pdf (uh_routing.py:5-22 +
// hbv_2_hourly.py:858-897).  par: [P, 3] in [0, 1] (route_a, route_b, route_tau).
// CTA = 32 pairs (lanes: coalesced rows of uh / the d/dUH workspace) x PTY tap threads; a thread
// evaluates taps ty, ty + PTY, ... (powf + expf each: one thread per pair walking all 72 taps was
// a 40 / 140 us serial chain on 79 warps); the normalisation sum and the adjoint's moments are
// reduced over the tap threads through shared memory in a fixed order.
constexpr int PKT = PM / PTY;      // taps per thread

__global__ void __launch_bounds__(PPB * PTY)
pair_uh_kernel(const PDesc d, const float* __restrict__ par, float* __restrict__ uh) {
    __shared__ float red[PTY][PPB];
    __shared__ float wn[PM][PPB];          // normalised pdf (the shift reads two neighbours)
    const int px = threadIdx.x % PPB, ty = threadIdx.x / PPB;
    const int p = blockIdx.x * PPB + px;
    const bool pv = p < d.P;
    const int pc = pv ? p : d.P - 1;
    const float a = par[pc * 3 + 0] * d.a_span + d.a_lo;
    const float b = par[pc * 3 + 1] * d.b_span + d.b_lo;
    const float aa = fmaxf(a, 0.f) + 0.1f;
    const float th = fmaxf(b, 0.f) + 0.5f;
    float w[PKT];
    float part = 0.f;
#pragma unroll
    for (int q = 0; q < PKT; ++q) {
        const int k = ty + PTY * q;
        w[q] = (k < d.M) ? gamma_w((float)k + 0.5f, aa, th) : 0.f;
        part += w[q];
    }
    red[ty][px] = part;
    __syncthreads();
    float sum = 0.f;
#pragma unroll
    for (int y = 0; y < PTY; ++y) sum += red[y][px];
    const float inv = 1.f / sum;
#pragma unroll
    for (int q = 0; q < PKT; ++q) {
        const int k = ty + PTY * q;
        if (k < d.M) wn[k][px] = w[q] * inv;
    }
    __syncthreads();
    int kk = 0;
    float f = 0.f;
    if (d.lag_uh) {
        const float tau = par[pc * 3 + 2] * d.t_span + d.t_lo;
        const float fl = floorf(tau);
        kk = (int)fl;
        f = tau - fl;
    }
    if (!pv) return;
    for (int k = ty; k < d.M; k += PTY) {
        const int i0 = k - kk, i1 = k - kk - 1;
        const float w0 = (i0 >= 0 && i0 < d.M) ? wn[i0][px] : 0.f;
        const float w1 = (i1 >= 0 && i1 < d.M) ? wn[i1][px] : 0.f;
        uh[(int64_t)k * d.P + p] = d.lag_uh ? ((1.f - f) * w0 + f * w1) : w0;
    }
}

// y[t][p] = sum_k uh[k][p] * x[t-k][p],  x[t][p] = src[t][col[p]] * scale[col[p]]
// REV: y[t][p] = sum_k uh[k][p] * x[t+k][p] (adjoint)
// One CTA = 32 pairs (lanes) x PTT time steps; a thread owns PR consecutive outputs of its pair and
// slides a PR-wide register window of x over the taps: per tap one LDS for the weight and one for
// the window's new element against PR FMAs (the plain form read both operands of every FMA from
// shared memory and was bound by LDS issue).  Taps are padded to a multiple of PR with zero
// weights so the window rotation unrolls with compile-time register indices.
template <bool REV>
__global__ void __launch_bounds__(PPB * PTY)
pair_conv_kernel(const PDesc d, const float* __restrict__ uh, const float* __restrict__ src, int src_stride,
                 const int* __restrict__ col, const float* __restrict__ scale, float* __restrict__ y) {
    extern __shared__ float sm[];
    const int Mp = round_up(d.M, PR);
    const int nrow = PTT + Mp - 1;
    float* us = sm;                       // [Mp][PPB]
    // [nrow + 1][PPB]: the window rows plus one pad row (in front for the forward, behind for the
    // adjoint) that the last, unused window refill reads — no index clamp in the tap loop
    float* xs = sm + Mp * PPB + (REV ? 0 : PPB);
    const int px = threadIdx.x % PPB;
    const int ty = threadIdx.x / PPB;
    const int p = blockIdx.x * PPB + px;
    const int t0 = blockIdx.y * PTT;
    const bool pv = p < d.P;
    int c = 0;
    float sc = 0.f;
    if (pv) { c = col ? col[p] : p; sc = scale ? scale[c] : 1.f; }
    for (int k = ty; k < Mp; k += PTY) us[k * PPB + px] = (pv && k < d.M) ? uh[(int64_t)k * d.P + p] : 0.f;
    // window rows r = 0..nrow-1 map to time  t0 - (Mp-1) + r  (forward)  /  t0 + r  (reverse)
    for (int r = ty; r < nrow; r += PTY) {
        const int t = REV ? (t0 + r) : (t0 - (Mp - 1) + r);
        xs[r * PPB + px] = (pv && t >= 0 && t < d.T) ? src[(int64_t)t * src_stride + c] * sc : 0.f;
    }
    if (ty == 0) xs[(REV ? nrow : -1) * PPB + px] = 0.f;
    __syncthreads();
    const int i0 = ty * PR;
    float acc[PR], w[PR];
#pragma unroll
    for (int r = 0; r < PR; ++r) acc[r] = 0.f;
    const float* up = us + px;
    if constexpr (!REV) {
        // logical window W_k[r] = xs[i0 + r + Mp-1-k], kept in register w[(r - k) mod PR]
#pragma unroll
        for (int r = 0; r < PR; ++r) w[r] = xs[(i0 + r + Mp - 1) * PPB + px];
        const float* xp = xs + (i0 + Mp - 2) * PPB + px;              // W_1[0]
        for (int kb = 0; kb < Mp; kb += PR) {
#pragma unroll
            for (int kk = 0; kk < PR; ++kk) {
                const float u = up[kk * PPB];
#pragma unroll
                for (int r = 0; r < PR; ++r) acc[r] = fmaf(u, w[(r - kk + PR) % PR], acc[r]);
                w[PR - 1 - kk] = xp[-kk * PPB];                       // W_{k+1}[0] (row -1 after the last tap)
            }
            up += PR * PPB;
            xp -= PR * PPB;
        }
    } else {
        // W_k[r] = xs[i0 + r + k], kept in register w[(r + k) mod PR]
#pragma unroll
        for (int r = 0; r < PR; ++r) w[r] = xs[(i0 + r) * PPB + px];
        const float* xp = xs + (i0 + PR) * PPB + px;                  // W_1[PR-1]
        for (int kb = 0; kb < Mp; kb += PR) {
#pragma unroll
            for (int kk = 0; kk < PR; ++kk) {
                const float u = up[kk * PPB];
#pragma unroll
                for (int r = 0; r < PR; ++r) acc[r] = fmaf(u, w[(r + kk) % PR], acc[r]);
                w[kk] = xp[kk * PPB];                                  // W_{k+1}[PR-1] (row nrow after the last tap)
            }
            up += PR * PPB;
            xp += PR * PPB;
        }
    }
    if (pv) {
#pragma unroll
        for (int r = 0; r < PR; ++r) {
            const int t = t0 + i0 + r;
            if (t < d.T) y[(int64_t)t * d.P + p] = acc[r];
        }
    }
}

// out[t][s] = mul[s] * sum_{i in [off[s], off[s+1])} val[t][perm ? perm[i] : i]
// Two thread mappings, both deterministic:
//   rows  lanes along the segments (short segments — the per-unit sums of the adjoint: reads of
//         neighbouring pairs and the writes are coalesced)
//   wide  one warp per (t, segment), lanes along the segment's members, xor-tree reduction (long
//         segments — the gage sums of the forward: 40 pairs per gage in BASELINE config 4)
constexpr int SST = 4;        // time steps per thread / warp (independent loads in flight)

__global__ void seg_sum_rows_kernel(int T, int S, int P, const int* __restrict__ off, const int* __restrict__ perm,
                                    const float* __restrict__ val, const float* __restrict__ mul,
                                    float* __restrict__ out, int out_stride) {
    const int s = blockIdx.x * 32 + threadIdx.x;
    if (s >= S) return;
    const int i0 = off[s], i1 = off[s + 1];
    const float m = mul ? mul[s] : 1.f;
    for (int t = (blockIdx.y * blockDim.y + threadIdx.y) * SST; t < T; t += gridDim.y * blockDim.y * SST) {
        float acc[SST];
#pragma unroll
        for (int q = 0; q < SST; ++q) acc[q] = 0.f;
        for (int i = i0; i < i1; ++i) {
            const int c = perm ? perm[i] : i;
#pragma unroll
            for (int q = 0; q < SST; ++q)
                if (t + q < T) acc[q] += val[(int64_t)(t + q) * P + c];
        }
#pragma unroll
        for (int q = 0; q < SST; ++q)
            if (t + q < T) out[(int64_t)(t + q) * out_stride + s] = acc[q] * m;
    }
}

__global__ void seg_sum_wide_kernel(int T, int S, int P, const int* __restrict__ off, const int* __restrict__ perm,
                                    const float* __restrict__ val, const float* __restrict__ mul,
                                    float* __restrict__ out, int out_stride) {
    const int s = blockIdx.x;
    const int i0 = off[s], i1 = off[s + 1];
    const float m = mul ? mul[s] : 1.f;
    for (int t = (blockIdx.y * blockDim.y + threadIdx.y) * SST; t < T; t += gridDim.y * blockDim.y * SST) {
        float acc[SST];
#pragma unroll
        for (int q = 0; q < SST; ++q) acc[q] = 0.f;
        for (int i = i0 + threadIdx.x; i < i1; i += 32) {
            const int c = perm ? perm[i] : i;
#pragma unroll
            for (int q = 0; q < SST; ++q)
                if (t + q < T) acc[q] += val[(int64_t)(t + q) * P + c];
        }
#pragma unroll
        for (int q = 0; q < SST; ++q) {
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) acc[q] += __shfl_xor_sync(0xffffffffu, acc[q], o);
        }
        if (threadIdx.x == 0) {
#pragma unroll
            for (int q = 0; q < SST; ++q)
                if (t + q < T) out[(int64_t)(t + q) * out_stride + s] = acc[q] * m;
        }
    }
}

static void seg_sum(int T, int S, int P, const int* off, const int* perm, const float* val, const float* mul,
                    float* out, int out_stride, cudaStream_t st) {
    const dim3 blk(32, 8);
    const int gy = (int)min((int64_t)(T + 8 * SST - 1) / (8 * SST), (int64_t)32768);
    if ((int64_t)P >= (int64_t)8 * S) seg_sum_wide_kernel<<<dim3(S, gy), blk, 0, st>>>(T, S, P, off, perm, val, mul, out, out_stride);
    else seg_sum_rows_kernel<<<dim3((S + 31) / 32, gy), blk, 0, st>>>(T, S, P, off, perm, val, mul, out, out_stride);
}

// dU[k][chunk][p] = sum_{t in chunk} g[t][p] * x[t-k][p]
//   g[t][p] = gsrc[t][gcol[p]] * gscale[gcol[p]],  x[t][p] = src[t][col[p]] * scale[col[p]]
// One CTA = 32 pairs x one time chunk, walked in tiles of PTT steps.  A tile's work is cut into
// items of DK consecutive taps x DTS time steps; an item slides a DK-wide register window of x
// along time (per step one LDS for g and one for the window's new element against DK FMAs) and
// adds its DK partial sums to its own slot of a shared accumulator du[time slice][tap][pair]; an
// item is always handled by the same thread, so the accumulation order is fixed.
__global__ void __launch_bounds__(PPB * PTY)
pair_duh_kernel(const PDesc d, const float* __restrict__ gsrc, int g_stride, const int* __restrict__ gcol,
                const float* __restrict__ gscale, const float* __restrict__ src, int src_stride,
                const int* __restrict__ col, const float* __restrict__ scale, float* __restrict__ ws) {
    extern __shared__ float sm[];
    const int Mp = round_up(d.M, DK);
    const int nrow = PTT + Mp - 1;
    float* gs = sm;                        // [PTT][PPB]
    float* xs = gs + PTT * PPB;            // [nrow + 1][PPB] (one zero pad row behind: the last window refill)
    float* du = xs + (nrow + 1) * PPB;     // [DNS][Mp][PPB]
    const int px = threadIdx.x % PPB;
    const int ty = threadIdx.x / PPB;
    const int p = blockIdx.x * PPB + px;
    const int ch = blockIdx.y;
    const bool pv = p < d.P;
    int c = 0, gc = 0;
    float sc = 0.f, gsc = 0.f;
    if (pv) {
        c = col ? col[p] : p; sc = scale ? scale[c] : 1.f;
        gc = gcol ? gcol[p] : p; gsc = gscale ? gscale[gc] : 1.f;
    }
    for (int e = ty; e < DNS * Mp; e += PTY) du[e * PPB + px] = 0.f;
    if (ty == 0) xs[nrow * PPB + px] = 0.f;
    const int ngrp = Mp / DK, nitem = ngrp * DNS;
    const int tbeg = ch * d.tchunk;
    const int tend = min(d.T, tbeg + d.tchunk);
    for (int t0 = tbeg; t0 < tend; t0 += PTT) {
        __syncthreads();
        for (int i = ty; i < PTT; i += PTY) {
            const int t = t0 + i;
            gs[i * PPB + px] = (pv && t < tend) ? gsrc[(int64_t)t * g_stride + gc] * gsc : 0.f;
        }
        for (int r = ty; r < nrow; r += PTY) {
            const int t = t0 - (Mp - 1) + r;
            xs[r * PPB + px] = (pv && t >= 0 && t < d.T) ? src[(int64_t)t * src_stride + c] * sc : 0.f;
        }
        __syncthreads();
        for (int item = ty; item < nitem; item += PTY) {
            const int grp = item % ngrp, sl = item / ngrp;
            const int k0 = grp * DK, ib = sl * DTS;
            // x[t0+i-k] sits in row i + Mp-1-k; logical window V_i[q] = xs[i + Mp-1-k0-q], kept in
            // register v[(q - i) mod DK] (ib is a multiple of DK)
            float acc[DK], v[DK];
#pragma unroll
            for (int q = 0; q < DK; ++q) { acc[q] = 0.f; v[q] = xs[(ib + Mp - 1 - k0 - q) * PPB + px]; }
            const float* gp = gs + ib * PPB + px;
            const float* xp = xs + (ib + Mp - k0) * PPB + px;          // V_{ib+1}[0]
            for (int i8 = 0; i8 < DTS; i8 += DK) {
#pragma unroll
                for (int ii = 0; ii < DK; ++ii) {
                    const float g = gp[ii * PPB];
#pragma unroll
                    for (int q = 0; q < DK; ++q) acc[q] = fmaf(g, v[(q - ii + DK) % DK], acc[q]);
                    v[DK - 1 - ii] = xp[ii * PPB];                     // V_{i+1}[0] (the pad row at the very end)
                }
                gp += DK * PPB;
                xp += DK * PPB;
            }
            float* dst = du + ((size_t)sl * Mp + k0) * PPB + px;
#pragma unroll
            for (int q = 0; q < DK; ++q) dst[q * PPB] += acc[q];
        }
    }
    __syncthreads();
    if (pv) {
        for (int k = ty; k < d.M; k += PTY) {
            float a = 0.f;
#pragma unroll
            for (int sl = 0; sl < DNS; ++sl) a += du[((size_t)sl * Mp + k) * PPB + px];
            ws[((int64_t)k * d.nchunk + ch) * d.P + p] = a;
        }
    }
}

// d/dUH -> d/d(par) through the fractional shift and the normalised gamma pdf
__global__ void __launch_bounds__(PPB * PTY)
pair_uh_bwd_kernel(const PDesc d, const float* __restrict__ par, const float* __restrict__ ws,
                   float* __restrict__ gpar) {
    __shared__ float red[PTY][4][PPB];
    const int px = threadIdx.x % PPB, ty = threadIdx.x / PPB;
    const int p = blockIdx.x * PPB + px;
    const bool pv = p < d.P;
    const int pc = pv ? p : d.P - 1;
    const float a = par[pc * 3 + 0] * d.a_span + d.a_lo;
    const float b = par[pc * 3 + 1] * d.b_span + d.b_lo;
    const float aa = fmaxf(a, 0.f) + 0.1f;
    const float th = fmaxf(b, 0.f) + 0.5f;
    float w[PKT];
    float part = 0.f;
#pragma unroll
    for (int q = 0; q < PKT; ++q) {
        const int j = ty + PTY * q;
        w[q] = (j < d.M) ? gamma_w((float)j + 0.5f, aa, th) : 0.f;
        part += w[q];
    }
    red[ty][0][px] = part;
    __syncthreads();
    float sum = 0.f;
#pragma unroll
    for (int y = 0; y < PTY; ++y) sum += red[y][0][px];
    const float inv = 1.f / sum;
    __syncthreads();
    int kk = 0;
    float f = 0.f;
    if (d.lag_uh) {
        const float tau = par[pc * 3 + 2] * d.t_span + d.t_lo;
        const float fl = floorf(tau);
        kk = (int)fl;
        f = tau - fl;
    }
    // g_y[k] = dL/d(shifted uh[k]);  g_u[j] = dL/d(normalised w[j]) = (1-f) g_y[j+kk] + f g_y[j+kk+1]
    // (g_y = 0 outside [0, M): a negative lag, given physically, shifts the UH forward)
    // With u[j] = w[j] / sum(w), L = log t, s0 = sum g_u u, mL = sum u L, mT = sum u t (sum u = 1):
    //   d/d(aa) = sum_j (g_u[j] - s0) u[j] (L[j] - mL),   d/d(th) = sum_j (g_u[j] - s0) u[j] (t[j] - mT) / th^2
    // in this centred form, from the moments of a first pass.  g_u has a common part much larger
    // than its variation over the taps (every tap's d/dUH is a sum over the same inputs); the
    // expanded form sum g_u u L - s0 mL cancels that part after rounding it, and came out up to
    // ~10x further from float64 than the reference's own float32 gradient (which centres g_u).
    float gu[PKT], lt[PKT];
    float gf = 0.f, mL = 0.f, mT = 0.f, s0 = 0.f;
#pragma unroll
    for (int q = 0; q < PKT; ++q) {
        const int j = ty + PTY * q;
        gu[q] = lt[q] = 0.f;
        w[q] *= inv;                               // u[j]
        if (j < d.M) {
            const float t = (float)j + 0.5f;
            const float u = w[q];
            float gy0 = 0.f, gy1 = 0.f;
            const int k0 = j + kk, k1 = j + kk + 1;
            if (k0 >= 0 && k0 < d.M) for (int c = 0; c < d.nchunk; ++c) gy0 += ws[((int64_t)k0 * d.nchunk + c) * d.P + pc];
            if (d.lag_uh && k1 >= 0 && k1 < d.M) for (int c = 0; c < d.nchunk; ++c) gy1 += ws[((int64_t)k1 * d.nchunk + c) * d.P + pc];
            gu[q] = d.lag_uh ? ((1.f - f) * gy0 + f * gy1) : gy0;
            gf += u * (gy1 - gy0);                 // d/df of (1-f) u[k-kk] + f u[k-kk-1]
            lt[q] = logf(t);
            mL += u * lt[q]; mT += u * t; s0 += gu[q] * u;
        }
    }
    red[ty][0][px] = gf; red[ty][1][px] = mL; red[ty][2][px] = mT; red[ty][3][px] = s0;
    __syncthreads();
    gf = mL = mT = s0 = 0.f;
#pragma unroll
    for (int y = 0; y < PTY; ++y) {                // every thread sums in the same order
        gf += red[y][0][px]; mL += red[y][1][px]; mT += red[y][2][px]; s0 += red[y][3][px];
    }
    __syncthreads();
    float ca = 0.f, cb = 0.f;
#pragma unroll
    for (int q = 0; q < PKT; ++q) {
        const int j = ty + PTY * q;
        if (j < d.M) {
            const float t = (float)j + 0.5f;
            const float du = (gu[q] - s0) * w[q];
            ca += du * (lt[q] - mL);
            cb += du * (t - mT);
        }
    }
    red[ty][0][px] = ca; red[ty][1][px] = cb;
    __syncthreads();
    if (ty != 0 || !pv) return;
    ca = cb = 0.f;
#pragma unroll
    for (int y = 0; y < PTY; ++y) { ca += red[y][0][px]; cb += red[y][1][px]; }
    const float gaa = ca;
    const float gth = cb / (th * th);
    gpar[p * 3 + 0] = (a > 0.f ? gaa : 0.f) * d.a_span;
    gpar[p * 3 + 1] = (b > 0.f ? gth : 0.f) * d.b_span;
    gpar[p * 3 + 2] = d.lag_uh ? gf * d.t_span : 0.f;
}

static size_t conv_smem(const PDesc& d) {
    const int Mp = round_up(d.M, PR);
    return (size_t)(Mp + PTT + Mp) * PPB * sizeof(float);
}
static size_t duh_smem(const PDesc& d) {
    const int Mp = round_up(d.M, DK);
    return (size_t)(PTT + PTT + Mp + DNS * Mp) * PPB * sizeof(float);
}
// the largest tap count needs more than the 48 KB a kernel gets without asking (once per process)
static void pair_smem_opt_in() {
    static const bool done = [] {
        PDesc m{};
        m.M = PM;
        cudaFuncSetAttribute(pair_conv_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)conv_smem(m));
        cudaFuncSetAttribute(pair_conv_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)conv_smem(m));
        cudaFuncSetAttribute(pair_duh_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)duh_smem(m));
        return true;
    }();
    (void)done;
}

static int make_pdesc(const hbv_pair_desc_t* s, PDesc& d) {
    if (!s) { set_error("null pair desc"); return HBV_E_NULL; }
    if (s->abi_version != HBV_B200_ABI_VERSION) { set_error("ABI version mismatch"); return HBV_E_ABI; }
    if (s->T <= 0 || s->n_pairs <= 0 || s->lenF <= 0 || s->n_units <= 0 || s->n_gages <= 0) { set_error("bad pair-routing shape"); return HBV_E_SHAPE; }
    d.T = s->T; d.P = s->n_pairs; d.M = s->lenF < s->T ? s->lenF : s->T;
    if (d.M > PM) { set_error("lenF > 128 not supported"); return HBV_E_SHAPE; }
    d.lag_uh = s->lag_uh;
    d.a_lo = s->a_lo; d.a_span = s->a_hi - s->a_lo; d.b_lo = s->b_lo; d.b_span = s->b_hi - s->b_lo;
    d.t_lo = s->tau_lo; d.t_span = s->tau_hi - s->tau_lo;
    d.nchunk = hbv_b200_pair_chunks(s->T);
    d.tchunk = ((s->T + d.nchunk - 1) / d.nchunk + PTT - 1) / PTT * PTT;
    pair_smem_opt_in();
    return 0;
}

}  // namespace hbv

using namespace hbv;

extern "C" int hbv_b200_pair_chunks(int32_t T) {
    int n = (T + 2047) / 2048;
    return n < 1 ? 1 : n;
}

extern "C" int hbv_b200_pair_route_fwd(const hbv_pair_desc_t* desc, const float* par, const float* qs,
                                       const float* areas, const int32_t* pair_col,
                                       const int32_t* gage_off, const float* inv_denom, float* uh,
                                       float* lag, float* out, void* stream) {
    PDesc d;
    int rc = make_pdesc(desc, d);
    if (rc) return rc;
    if (!par || !qs || !gage_off || !uh || !lag || !out) { set_error("null pointer"); return HBV_E_NULL; }
    cudaStream_t st = (cudaStream_t)stream;
    pair_uh_kernel<<<(d.P + PPB - 1) / PPB, PPB * PTY, 0, st>>>(d, par, uh);
    dim3 grid((d.P + PPB - 1) / PPB, (d.T + PTT - 1) / PTT);
    pair_conv_kernel<false><<<grid, PPB * PTY, conv_smem(d), st>>>(d, uh, qs, desc->n_units, pair_col, areas, lag);
    seg_sum(d.T, desc->n_gages, d.P, gage_off, nullptr, lag, inv_denom, out, desc->n_gages, st);
    count_launch(3);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) set_error(cudaGetErrorString(e));
    return (int)e;
}

extern "C" int hbv_b200_pair_route_bwd(const hbv_pair_desc_t* desc, const float* par, const float* qs,
                                       const float* areas, const int32_t* pair_col,
                                       const int32_t* pair_row, const float* inv_denom,
                                       const int32_t* unit_off, const int32_t* unit_perm,
                                       const float* uh, const float* g_out, float* g_lag_ws,
                                       float* duh_ws, float* g_qs, float* g_par, void* stream) {
    PDesc d;
    int rc = make_pdesc(desc, d);
    if (rc) return rc;
    if (!par || !qs || !pair_row || !unit_off || !unit_perm || !uh || !g_out || !g_lag_ws || !duh_ws || !g_qs || !g_par) {
        set_error("null pointer"); return HBV_E_NULL;
    }
    cudaStream_t st = (cudaStream_t)stream;
    dim3 grid((d.P + PPB - 1) / PPB, (d.T + PTT - 1) / PTT);
    // g_x[t][p] = sum_k uh[k][p] * g[t+k][p],  g[t][p] = g_out[t][row[p]] * inv_denom[row[p]]
    pair_conv_kernel<true><<<grid, PPB * PTY, conv_smem(d), st>>>(d, uh, g_out, desc->n_gages, pair_row, inv_denom, g_lag_ws);
    // g_qs[t][u] = area[u] * sum_{pairs of unit u} g_x[t][p]
    seg_sum(d.T, desc->n_units, d.P, unit_off, unit_perm, g_lag_ws, areas, g_qs, desc->n_units, st);
    dim3 g3((d.P + PPB - 1) / PPB, d.nchunk);
    pair_duh_kernel<<<g3, PPB * PTY, duh_smem(d), st>>>(d, g_out, desc->n_gages, pair_row, inv_denom, qs, desc->n_units,
                                                         pair_col, areas, duh_ws);
    pair_uh_bwd_kernel<<<(d.P + PPB - 1) / PPB, PPB * PTY, 0, st>>>(d, par, duh_ws, g_par);
    count_launch(4);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) set_error(cudaGetErrorString(e));
    return (int)e;
}
