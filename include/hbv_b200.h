/*
 * hbv_b200.h — C-ABI of the B200-native HBV recurrence + unit-hydrograph routing.
 *
 * This is the drop-in boundary (SURVEY.md §8 b2).  The reference
 * (mhpi/hydrodl2) has no FFI: its hot path is Python that issues ~70 ATen
 * kernels per time step.  Each entry point below replaces one span of that
 * Python (cited as reference file:line, paths relative to
 * /root/reference/src/hydrodl2/) and is what a reference maintainer would
 * bind with ctypes from inside `_PBM` (see INTEGRATION.md).
 *
 * Conventions
 *   - every pointer is a DEVICE pointer owned by the caller (PyTorch) unless stated otherwise
 *     (hbv_b200_copy_cols / memcpy2d also take pinned host pointers); the library never
 *     allocates and never frees.  Its only process-wide state is bookkeeping that does not
 *     change results: the launch counters (hbv_b200_*_launches) and the table of experiment
 *     switches (hbv_b200_set_option; initialised from the environment once) — kernels of
 *     different families give the same numbers to fp32 round-off;
 *   - all tensors are float32, contiguous in the layouts stated below;
 *   - `stream` is the caller's cudaStream_t (0 = legacy default stream);
 *   - return value: 0 ok, >0 a cudaError_t from launch, <0 argument error
 *     (HBV_E_*); functions never throw and are re-entrant / thread-safe;
 *   - the last error text of the calling thread: hbv_b200_last_error().
 */
#ifndef HBV_B200_H
#define HBV_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define HBV_B200_ABI_VERSION 5

#if defined(__GNUC__)
#define HBV_API __attribute__((visibility("default")))
#else
#define HBV_API
#endif

#define HBV_MAX_PAR 20   /* physical parameters per variant (max 19 used) */
#define HBV_MAX_FLUX 12  /* per-step flux series reduced over nmul */
#define HBV_NSTATE 5     /* SNOWPACK, MELTWATER, SM, SUZ, SLZ (hbv.py:61-67) */

/* argument errors */
#define HBV_E_NULL (-1)
#define HBV_E_SHAPE (-2)
#define HBV_E_VARIANT (-3)
#define HBV_E_NMUL (-4)
#define HBV_E_CKPT (-5)
#define HBV_E_ABI (-6)

/* variants (which step arithmetic) */
enum {
    HBV_VARIANT_HBV = 0,      /* models/hbv/hbv.py:423-505            */
    HBV_VARIANT_HBV11P = 1,   /* models/hbv/hbv_1_1p.py:422-516       */
    HBV_VARIANT_HBV2 = 2,     /* models/hbv/hbv_2.py:464-575          */
    HBV_VARIANT_HOURLY = 3,   /* models/hbv/hbv_2_hourly.py:527-675   */
    HBV_VARIANT_ADJ = 4       /* models/hbv/hbv_adj.py:341-498 (implicit scheme; hbv_b200_adj_* only) */
};

/* physical parameter slots — the order of `parameter_bounds`
 * (hbv.py:88-101, hbv_1_1p.py:87-102, hbv_2.py:90-107, hbv_2_hourly.py:91-115) */
enum {
    HBV_P_BETA = 0, HBV_P_FC, HBV_P_K0, HBV_P_K1, HBV_P_K2, HBV_P_LP, HBV_P_PERC,
    HBV_P_UZL, HBV_P_TT, HBV_P_CFMAX, HBV_P_CFR, HBV_P_CWH, HBV_P_BETAET, HBV_P_C,
    HBV_P_RT, HBV_P_AC, HBV_P_F0, HBV_P_FMIN, HBV_P_ALPHA
};

/* flux slots written by hbv_b200_fwd (each a [T, B] plane, nmul-reduced) */
enum {
    HBV_F_QSIM = 0,   /* Q0+Q1+Q2 (+IE hourly): mean or muwts-weighted (hbv.py:494,508-511) */
    HBV_F_Q0, HBV_F_Q1, HBV_F_Q2, HBV_F_AET, HBV_F_SWE, HBV_F_RECHARGE, HBV_F_EXCS,
    HBV_F_EVAPFACTOR, HBV_F_TOSOIL, HBV_F_PERC, HBV_F_CAPILLARY
};

/* where a physical parameter's [0,1]/raw value is read from */
enum {
    HBV_SRC_DYN_T = 0,    /* dyn[t, b, col + j]      time-varying (dynamic)          */
    HBV_SRC_DYN_LAST = 1, /* dyn[T-1, b, col + j]    static value of the packed form */
    HBV_SRC_STA = 2       /* sta[b, col + j]         static tensor of the hbv_2 form */
};

/*
 * Problem descriptor.  Plain data, passed by pointer, copied by the callee.
 *
 * Parameter addressing restates hbv.py:182-256 (packed raw tensor, sigmoid,
 * static value = last row of the slice) and hbv_2.py:190-290 (split dynamic /
 * static tensors already in [0,1]):
 *     v01 = apply_sigmoid ? sigmoid(raw) : raw
 *     par = v01 * (hi - lo) + lo                     (core/calc/utils.py:24)
 * A dynamic parameter whose dropout mask is set for a basin reads row T-1 of
 * `dyn` instead of row t (hbv.py:242-246, hbv_2.py:258-265).
 */
typedef struct hbv_desc {
    int32_t abi_version;           /* HBV_B200_ABI_VERSION */
    int32_t variant;               /* HBV_VARIANT_* */
    int32_t T;                     /* time steps in this call */
    int32_t B;                     /* basins (grid cells / units) */
    int32_t nmul;                  /* parallel components per basin */
    int32_t n_par;                 /* physical parameters of the variant */
    int32_t betaet;                /* 1: evapfactor **= parBETAET (hbv.py:475-476) */
    int32_t apply_sigmoid;         /* 1: raw parameters (hbv / hbv_1_1p) */
    int32_t nvar;                  /* last dim of forcing */
    int32_t i_prcp, i_tmean, i_pet;/* forcing columns (hbv.py:388-390) */
    int32_t dyn_ncol;              /* row width of `dyn` */
    int32_t sta_ncol;              /* row width of `sta` (0 if unused) */
    int32_t par_src[HBV_MAX_PAR];  /* HBV_SRC_* per parameter */
    int32_t par_col[HBV_MAX_PAR];  /* first column of parameter i in its source */
    float par_lo[HBV_MAX_PAR];
    float par_hi[HBV_MAX_PAR];
    float nearzero;                /* hbv.py:54 */
    float dt;                      /* 1 (daily) or 1/24 (hbv_2_hourly.py:58) */
    int32_t ckpt_interval;         /* K: state checkpoint every K steps (0 = none) */
    int32_t muwts_t_stride;        /* elements between time rows of muwts (0 = time-invariant) */
    int32_t adj_max_updates;       /* HBV_VARIANT_ADJ: Newton updates per step (0 = default 8;
                                      the reference allows 4, hbv_adj.py:518,544) */
    float adj_tol;                 /* HBV_VARIANT_ADJ: ||G||_inf stopping tolerance (0 = default
                                      1e-3, the reference's gtol, hbv_adj.py:519) */
    int32_t ckpt_layout;           /* layout of the caller-allocated state store `ckpt` (same value
                                      in the forward and the backward call; same size either way):
                                      0 = [ceil(T/K), 5, B, nmul] planes; 1 = warp-major
                                      [ceil(B*nmul/32)][ceil(T/K)][5][32] — one contiguous 640 B run
                                      per warp and stored step.  1 is served by the standard-layout
                                      (K1s / K2s) and the generic (K1 / K2) kernels; not valid together
                                      with the hbv_2 state series that aliases the store. */
    int32_t reserved[3];
} hbv_desc_t;

/* Forward I/O.  NULL output pointers are skipped. */
typedef struct hbv_fwd_io {
    const float* forcing;    /* [T, B, nvar]                              */
    const float* dyn;        /* [T, B, dyn_ncol]                          */
    const float* sta;        /* [B, sta_ncol] or NULL                     */
    const uint8_t* drop;     /* [n_par, B] 0/1 dropout masks or NULL      */
    const float* attrs;      /* [2, B]: Ac, Elevation (hbv_2 family) or NULL */
    const float* muwts;      /* [T or 1, B, nmul] or NULL (hbv.py:508-511) */
    const float* state_in;   /* [5, B, nmul]                              */
    float* state_out;        /* [5, B, nmul]                              */
    float* flux[HBV_MAX_FLUX];/* each [T, B]; all NULL = warm-up/initialize run (hbv.py:557-559) */
    float* state_series;     /* [5, T, B, nmul] or NULL (hbv_2.py:571-575) */
    float* ckpt;             /* [ceil(T/K), 5, B, nmul] or NULL           */
} hbv_fwd_io_t;

/* Backward I/O (hand-written adjoint of hbv_b200_fwd; replaces autograd over
 * the unrolled loop, SURVEY.md §3c). */
typedef struct hbv_bwd_io {
    const float* forcing;
    const float* dyn;
    const float* sta;
    const uint8_t* drop;
    const float* attrs;
    const float* muwts;
    const float* ckpt;                 /* from the forward call, same K     */
    const float* gflux[HBV_MAX_FLUX];  /* upstream grads, each [T, B] or NULL */
    const float* gstate_out;           /* [5, B, nmul] or NULL              */
    const float* gstate_series;        /* [5, T, B, nmul] or NULL           */
    float* gdyn;     /* [T, B, dyn_ncol].  gdyn_zero_fill = 0: ZERO-INITIALISED by the
                        caller, the kernel writes only entries that receive gradient
                        (row t for dynamic parameters, row T-1 for static ones).
                        gdyn_zero_fill = 1: uninitialised memory is fine — the kernel
                        writes EVERY element of rows 0..T-2 (zeros where no gradient
                        flows) and, in row T-1, every physical-parameter column; row T-1
                        columns beyond n_par*nmul (routing) are left untouched.          */
    float* gsta;     /* [B, sta_ncol] or NULL                               */
    float* gstate_in;/* [5, B, nmul] or NULL                                */
    int32_t gdyn_zero_fill;
    int32_t gdyn_rows_before;  /* with gdyn_zero_fill: this many rows in FRONT of gdyn (the no-grad
                                  warm-up rows of the caller's full [T_total, B, dyn_ncol] plane,
                                  hbv.py:328) are zeroed by the call as well — inside the
                                  stage-pipelined adjoint (TMA bulk stores of a zeroed shared-memory
                                  buffer, paced over its sweep), else by a memset in stream order */
    float* gforcing; /* [T, B, nvar] or NULL: gradient w.r.t. the forcings (P, T, PET columns),
                        summed over the nmul components; ZERO-INITIALISED by the caller.  The
                        rain/snow masks carry no gradient (hbv.py:431-434), T receives it through
                        melt and refreeze only */
    float* gmuwts;   /* [T or 1, B, nmul] (same time stride as muwts) or NULL: gradient w.r.t.
                        the component weights, dL/dQsim[t,b] * Qsim_lane[t,b,j]                 */
} hbv_bwd_io_t;

/* K1: fused forward recurrence + nmul aggregation (hbv.py:363-511).
 * K1 / K2 each exist in three interchangeable compilations, chosen from the descriptor alone (same
 * arithmetic, results equal to fp32 round-off): the general kernels (any dynamic set, dropout,
 * muwts, state series, any nmul), the standard-layout kernels (nvar 3 in prcp/tmean/pet order,
 * nmul 16, columns 16*i, the shipped dynamic sets; adjoint: ckpt_interval 1 and an upstream
 * gradient on the streamflow series only) and the TMA-staged kernels (>= 8 time-varying
 * parameters filling at least half of a row, full-GPU grids).  See DESIGN.md section 4. */
HBV_API int hbv_b200_fwd(const hbv_desc_t* desc, const hbv_fwd_io_t* io, void* stream);

/* K2: checkpointed adjoint of K1. */
HBV_API int hbv_b200_bwd(const hbv_desc_t* desc, const hbv_bwd_io_t* io, void* stream);

/*
 * K3: implicit (backward-Euler) HBV, `HbvAdj` (models/hbv/hbv_adj.py).
 *
 * hbv_b200_adj_fwd replaces the per-step NewtonSolve.apply loop (hbv_adj.py:689-712 calling
 * :504-615: batchJacobian + torch.linalg.solve + three host syncs per iteration) and the flux
 * read-out + nmul mean (:309-317) by one launch: each (basin, component) lane solves
 * G(x) = (x - xt)/dt - f(x, p_t, t) = 0 by Newton with the analytic block-triangular Jacobian,
 * stopping per lane (||G||_inf <= adj_tol, then one polishing update, <= adj_max_updates).
 * hbv_b200_adj_bwd is the adjoint the reference intends at hbv_adj.py:620-633
 * (lambda = (dG/dx)^-T dL/dx; dL/dp = -lambda^T dG/dp; dL/dxt = -lambda^T dG/dxt) with
 * analytic dG/dp in place of core/calc/fdj.py:46-92.  The same sweep also gives the gradient
 * w.r.t. the forcings, dL/d(P, T, Ep) = lambda^T df/d(P, T, Ep), and the initial state.
 * desc->variant must be HBV_VARIANT_ADJ, n_par 12 or 13 (betaet), parameters packed
 * (HBV_SRC_DYN_T / HBV_SRC_DYN_LAST), dt = 1.
 */
typedef struct hbv_adj_fwd_io {
    const float* forcing;    /* [T, B, nvar]                                   */
    const float* dyn;        /* [T, B, dyn_ncol] raw packed parameters         */
    const uint8_t* drop;     /* [n_par, B] or NULL                             */
    const float* state_in;   /* [5, B, nmul]  (hbv_adj.py:254: zeros)          */
    float* state_out;        /* [5, B, nmul] or NULL                           */
    float* qsim;             /* [T, B] nmul-mean of (q0+q1+q2)*dt or NULL      */
    float* ysol;             /* [T, 5, B, nmul] end-of-step states or NULL (required by bwd) */
    int32_t* stats;          /* [2] or NULL: max updates used (atomicMax), lane-steps that hit
                                adj_max_updates unconverged (atomicAdd); caller zeroes it */
} hbv_adj_fwd_io_t;

typedef struct hbv_adj_bwd_io {
    const float* forcing;
    const float* dyn;
    const uint8_t* drop;
    const float* ysol;         /* from the forward call                         */
    const float* gqsim;        /* [T, B] or NULL                                */
    const float* gstate_out;   /* [5, B, nmul] or NULL                          */
    float* gdyn;               /* [T, B, dyn_ncol]; zero-initialised by the caller unless
                                  gdyn_zero_fill is set.  NULL: no parameter gradient at all (no
                                  stores to it; gdyn_zero_fill must then be 0 and at least one of
                                  gforcing / gstate_in given) — e.g. precipitation data
                                  assimilation, where only dL/dP is wanted and the dense plane
                                  would be 6 GB at BASELINE config 5 */
    float* gstate_in;          /* [5, B, nmul] or NULL                          */
    int32_t gdyn_zero_fill;    /* 1 (nmul 16, even dyn_ncol only): the kernel zeroes rows 0 .. T-2 of
                                  gdyn itself before it writes its gradients, so the dense plane needs
                                  no memset (6 GB at BASELINE config 5); of row T-1 it writes the
                                  parameter columns only — the caller owns that row's other columns */
    float* gforcing;           /* [T, B, nvar] or NULL (ABI 5): gradient w.r.t. the forcings, same
                                  contract as hbv_bwd_io_t.gforcing — ZERO-INITIALISED by the caller;
                                  the kernel writes columns i_prcp, i_tmean, i_pet of every row of the
                                  call, each summed over the nmul components (a fixed-order sum, no
                                  atomics), and leaves the other columns untouched.  The rain/snow
                                  mask carries no gradient; T receives it through melt and refreeze */
} hbv_adj_bwd_io_t;

HBV_API int hbv_b200_adj_fwd(const hbv_desc_t* desc, const hbv_adj_fwd_io_t* io, void* stream);
HBV_API int hbv_b200_adj_bwd(const hbv_desc_t* desc, const hbv_adj_bwd_io_t* io, void* stream);

/*
 * K4: gamma unit hydrograph + causal convolution + BFI
 * (core/calc/uh_routing.py:5-57, hbv.py:523-538,562-567).
 *
 *   route     [B, route_stride]: columns 0,1 = route_a, route_b (raw or [0,1])
 *   q_in      nser planes [T, B] (plane stride q_stride elements)
 *   q_out     nser planes [T, B] (plane stride out_stride)
 *   uh        [lenF, B] workspace/output: the normalised UH weights
 *   bfi       [B] or NULL: 100 * sum_t out[bfi_num] / (sum_t out[bfi_den] + nearzero)
 *   bfi_ws    [2, nchunk, B] workspace when bfi != NULL (see hbv_b200_route_chunks)
 */
typedef struct hbv_route_desc {
    int32_t abi_version;
    int32_t T, B, lenF, nser;
    int32_t apply_sigmoid;
    int32_t route_stride;
    int32_t bfi_num, bfi_den;   /* series indices for BFI */
    float a_lo, a_hi, b_lo, b_hi;
    float nearzero;
    int32_t reserved[4];
} hbv_route_desc_t;

HBV_API int hbv_b200_route_chunks(int32_t T, int32_t B);

HBV_API int hbv_b200_route_fwd(const hbv_route_desc_t* desc, const float* route,
                       const float* q_in, int64_t q_stride, float* q_out,
                       int64_t out_stride, float* uh, float* bfi, float* bfi_ws,
                       void* stream);

/*
 * Adjoint of hbv_b200_route_fwd.
 *   g_out     nser planes [T, B] or per-series NULL via g_out_mask bit s
 *   g_bfi     [B] or NULL
 *   g_in      nser planes [T, B]; plane s is written only if series s is live, i.e. bit s of
 *             g_out_mask is set or g_bfi != NULL and s is bfi_num / bfi_den (a dead series has
 *             an all-zero adjoint; its plane is left untouched)
 *   g_route   [B, route_stride]: columns 0,1 written (gradient w.r.t. the raw /
 *             [0,1] routing parameters)
 *   ws        workspace [ min(lenF, T) * nchunk * B ] floats (per-tap d/dUH partial sums of the
 *             nchunk = hbv_b200_route_chunks(T, B) time chunks)
 */
HBV_API int hbv_b200_route_bwd(const hbv_route_desc_t* desc, const float* route,
                       const float* q_in, int64_t q_stride, const float* q_out,
                       int64_t out_stride, const float* uh, const float* bfi_ws,
                       const float* g_out, int64_t g_stride, uint32_t g_out_mask,
                       const float* g_bfi, float* g_in, int64_t gin_stride,
                       float* g_route, float* ws, void* stream);

/*
 * K4': distributed (gage, unit) pair routing (hbv_2_hourly.py:800-897: distr_routing +
 * _frac_shift1d).  Pairs are the non-zeros of outlet_topo in row-major order (sorted by gage).
 *
 *   par        [n_pairs, 3] in [0,1]: route_a, route_b, route_tau (descaled with the bounds below)
 *   qs         [T, n_units] unit runoff
 *   areas      [n_units]
 *   pair_col   [n_pairs] unit of each pair;  pair_row [n_pairs] gage of each pair
 *   gage_off   [n_gages + 1] CSR offsets of the pairs of each gage
 *   inv_denom  [n_gages] 1 / clamp(sum_u topo[g,u] * area[u], 1e-6)
 *   unit_off   [n_units + 1], unit_perm [n_pairs]: pairs grouped by unit (CSC) for the adjoint
 *   uh         [min(T,lenF), n_pairs] out: lagged unit hydrographs (kept for the adjoint)
 *   lag        [T, n_pairs] workspace: per-pair convolved runoff
 *   out        [T, n_gages] gage streamflow
 */
typedef struct hbv_pair_desc {
    int32_t abi_version;
    int32_t T, n_pairs, n_units, n_gages, lenF;
    int32_t lag_uh;                 /* 1: apply the fractional lag (hbv_2_hourly.py:832-833) */
    float a_lo, a_hi, b_lo, b_hi, tau_lo, tau_hi;
    int32_t reserved[4];
} hbv_pair_desc_t;

HBV_API int hbv_b200_pair_chunks(int32_t T);

HBV_API int hbv_b200_pair_route_fwd(const hbv_pair_desc_t* desc, const float* par, const float* qs,
                                    const float* areas, const int32_t* pair_col,
                                    const int32_t* gage_off, const float* inv_denom, float* uh,
                                    float* lag, float* out, void* stream);

/*   g_out [T, n_gages] upstream gradient;  g_lag_ws [T, n_pairs] workspace;
 *   duh_ws [min(T,lenF), hbv_b200_pair_chunks(T), n_pairs] workspace;
 *   g_qs [T, n_units] and g_par [n_pairs, 3] are written. */
HBV_API int hbv_b200_pair_route_bwd(const hbv_pair_desc_t* desc, const float* par, const float* qs,
                                    const float* areas, const int32_t* pair_col,
                                    const int32_t* pair_row, const float* inv_denom,
                                    const int32_t* unit_off, const int32_t* unit_perm,
                                    const float* uh, const float* g_out, float* g_lag_ws,
                                    float* duh_ws, float* g_qs, float* g_par, void* stream);

/* misc */
HBV_API int hbv_b200_abi_version(void);
HBV_API const char* hbv_b200_last_error(void);
/* checkpoint interval the library recommends for hbv_b200_fwd/bwd on a problem of this size:
 * 1 (store every state — 20 B per lane-step — and skip the adjoint's recompute pass) while the
 * stored states fit 16 GiB, 16 otherwise */
HBV_API int hbv_b200_auto_ckpt(int32_t T, int32_t B, int32_t nmul);
/* bytes of the caller-allocated state store (`ckpt`) hbv_b200_fwd writes and hbv_b200_bwd reads for
 * this problem: ceil(T / K) * 5 * B * nmul floats with K = desc->ckpt_interval, or
 * hbv_b200_auto_ckpt(T, B, nmul) when that is 0 (SURVEY.md section 8 b2: hbv_workspace_bytes).
 * Returns < 0 (HBV_E_*) on a bad descriptor.  The library itself never allocates. */
/* The checkpoint interval the library would pick for this run (descriptor-aware form of
 * hbv_b200_auto_ckpt: runs served by the standard-layout kernels use K = 4 on large grids —
 * measured crossover in csrc/hbv_cabi.cu).  desc->ckpt_interval is ignored. */
HBV_API int hbv_b200_auto_ckpt_desc(const hbv_desc_t* desc);
HBV_API int64_t hbv_b200_workspace_bytes(const hbv_desc_t* desc);
/* number of kernels this library has launched in this process (bench accounting) */
HBV_API int64_t hbv_b200_launch_count(void);
/* how many of those were the TMA-staged kernels of hbv_dense.cu (K1d / K2d), which
 * hbv_b200_fwd / hbv_b200_bwd select by themselves for dense-dynamic runs on large grids
 * (set HBV_B200_DENSE=0 in the environment to keep K1 / K2) */
HBV_API int64_t hbv_b200_dense_launches(void);
/* ... and how many were the standard-layout kernels of hbv_lean.cu (K1s / K2s), selected the same
 * way for the shipped dynamic sets on large grids (HBV_B200_LEAN=0 keeps K1 / K2) */
HBV_API int64_t hbv_b200_lean_launches(void);
/* Zero `nbytes` bytes at `ptr` (device memory) with a thin kernel: `n_ctas` one-warp CTAs (0 =
 * one per SM) streaming TMA bulk stores from a zeroed shared-memory buffer.  Made for zeroing the
 * dense parameter-gradient plane on a side stream underneath latency-bound kernels (csrc/fill.cu);
 * replaces the cudaMemsetAsync the torch side would otherwise issue for torch.zeros_like. */
HBV_API int hbv_b200_fill_zero(void* ptr, int64_t nbytes, int32_t n_ctas, void* stream);
/* Copy the [rows x ncols] float block at column `col0` of a row-major [rows, row_stride] matrix
 * from `src` to `dst` (same layout on both sides).  Either pointer may be mapped pinned HOST
 * memory (cudaHostAlloc / torch pin_memory under UVA): the GPU then reads or writes it directly
 * over PCIe, so a training loop stages only the column blocks the kernels read (the dynamic
 * parameters of hbv.py:201-208) and fetches only the non-zero blocks of the gradient.  Used by
 * hydrodl2_b200.hostio. */
HBV_API int hbv_b200_copy_cols(float* dst, const float* src, int64_t rows, int64_t row_stride,
                               int32_t col0, int32_t ncols, void* stream);
/* The same block copy through the DMA engine (cudaMemcpy2DAsync); kind 1 = host -> device,
 * 2 = device -> host.  Measured against copy_cols in scripts/experiments/stage_bw.py. */
HBV_API int hbv_b200_memcpy2d(float* dst, const float* src, int64_t rows, int64_t row_stride,
                              int32_t col0, int32_t ncols, int32_t kind, void* stream);
/* One-shot all-reduce (sum) of a small float vector over NVLink peer memory (csrc/allreduce.cu):
 * `peer_bufs_dev` is a DEVICE array of `world` pointers to the ranks' symmetric comm buffers
 * (each hbv_b200_allreduce_buffer_floats(world, n) floats, zero-initialised once, peer-mapped —
 * e.g. torch.distributed._symmetric_memory.rendezvous(...).buffer_ptrs_dev).  Every rank calls it
 * the same number of times; `out` receives the bit-identical sum on every rank.  A plain kernel
 * launch: capturable in a CUDA graph (the step counter lives in the buffer). */
HBV_API int64_t hbv_b200_allreduce_buffer_floats(int32_t world, int32_t n);
HBV_API int hbv_b200_oneshot_allreduce(float* const* peer_bufs_dev, int32_t rank, int32_t world,
                                       const float* in, float* out, int32_t n, void* stream);
/* Experiment / test switches.  Each is read from the environment (HBV_B200_<NAME>) once, when
 * the library is first used, and can be changed at run time here; value -1 = unset (the
 * library's own measured policy decides).  Names (case-insensitive): "lean" (0: never K1s / K2s /
 * K1p / K2p), "pipe" (0: never K1p / K2p), "pipe_max" (largest grid in lanes for K1p / K2p),
 * "ring" (0 / 1: force register / cp.async-ring inputs in K1 / K2; 0 also keeps K3's adjoint on
 * its register form), "lean_small", "lean_bwd_ring", "lean_deep" (largest grid in lanes whose
 * 128-thread K1s takes its inputs through the chunk ring; 0: register prefetch), "dense" (0: never
 * K1d / K2d, 2: wherever the shapes allow), "dense_ns", "dense_ns_bwd", "dense_minb", "ckpt" (the
 * interval hbv_b200_auto_ckpt returns), "adj_bpb" (basins per CTA of K3's forward), "copy_blocks"
 * (hbv_b200_copy_cols: blocks per SM), "ckpt_layout" (read by the Python host side: forces
 * hbv_desc_t.ckpt_layout).  Returns 0, or
 * HBV_E_SHAPE for an unknown name (get: INT64_MIN). */
HBV_API int hbv_b200_set_option(const char* name, int64_t value);
HBV_API int64_t hbv_b200_get_option(const char* name);
/* launches of the stage-pipelined kernels K1p / K2p (csrc/hbv_pipe.cu; a subset of lean_launches) */
HBV_API int64_t hbv_b200_pipe_launches(void);

#ifdef __cplusplus
}
#endif
#endif /* HBV_B200_H */
