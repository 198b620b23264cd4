// hbv_cabi.cu — extern "C" entry points, argument validation, error text, launch accounting.
#include <atomic>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include "hbv_common.cuh"

namespace hbv {

static thread_local char g_err[256] = "";
static std::atomic<long long> g_launches{0};
static std::atomic<long long> g_dense_launches{0};
static std::atomic<long long> g_lean_launches{0};
static std::atomic<long long> g_pipe_launches{0};

// option table: environment at first use, then hbv_b200_set_option
static const char* const kOptNames[OPT_COUNT] = {
    "LEAN", "PIPE", "PIPE_MAX", "RING", "LEAN_SMALL", "LEAN_BWD_RING", "LEAN_DEEP", "DENSE", "DENSE_NS", "DENSE_NS_BWD",
    "DENSE_MINB", "CKPT", "ADJ_BPB", "COPY_BLOCKS", "CKPT_LAYOUT"};
static std::atomic<long long> g_opt[OPT_COUNT];
static std::atomic<int> g_opt_init{0};
static void opt_init() {
    if (g_opt_init.load(std::memory_order_acquire)) return;
    for (int i = 0; i < OPT_COUNT; ++i) {
        char name[64];
        std::snprintf(name, sizeof(name), "HBV_B200_%s", kOptNames[i]);
        const char* e = std::getenv(name);
        g_opt[i].store((e && *e) ? std::atoll(e) : -1, std::memory_order_relaxed);
    }
    g_opt_init.store(1, std::memory_order_release);
}
long long opt(Opt o) {
    opt_init();
    return g_opt[o].load(std::memory_order_relaxed);
}
static int opt_index(const char* name) {
    if (!name) return -1;
    for (int i = 0; i < OPT_COUNT; ++i) {
        const char* a = kOptNames[i];
        const char* b = name;
        while (*a && *b && (*a == *b || *a == *b - 32)) { ++a; ++b; }   // case-insensitive on lower-case input
        if (!*a && !*b) return i;
    }
    return -1;
}

void set_error(const char* msg) {
    std::snprintf(g_err, sizeof(g_err), "%s", msg ? msg : "");
}
void count_launch(int n) { g_launches.fetch_add(n, std::memory_order_relaxed); }
void count_dense_launch() { g_dense_launches.fetch_add(1, std::memory_order_relaxed); }
void count_lean_launch() { g_lean_launches.fetch_add(1, std::memory_order_relaxed); }
void count_pipe_launch() { g_pipe_launches.fetch_add(1, std::memory_order_relaxed); }

int fwd_dispatch(const hbv_desc_t* desc, const hbv_fwd_io_t* io, cudaStream_t st);
int bwd_dispatch(const hbv_desc_t* desc, const hbv_bwd_io_t* io, cudaStream_t st);
int adj_fwd_dispatch(const hbv_desc_t* desc, const hbv_adj_fwd_io_t* io, cudaStream_t st);
int adj_bwd_dispatch(const hbv_desc_t* desc, const hbv_adj_bwd_io_t* io, cudaStream_t st);
int tlm_dispatch(const hbv_desc_t* desc, const hbv_tlm_io_t* io, cudaStream_t st);   // hbv_tlm.cu

static int expected_npar(int variant, int betaet) {
    switch (variant) {
        case HBV_VARIANT_HBV: return betaet ? 13 : 12;
        case HBV_VARIANT_HBV11P: return 14;
        case HBV_VARIANT_HBV2: return 16;
        case HBV_VARIANT_HOURLY: return 19;
        case HBV_VARIANT_ADJ: return betaet ? 13 : 12;
    }
    return -1;
}

// basins per CTA: 128-256 threads when there is enough work, fewer for small problems so the
// grid still covers the 148 SMs (SURVEY.md §7 "low parallelism configs")
static int choose_bpb(int B, int nmul) {
    int bpb = 128 / nmul;
    if (bpb < 1) bpb = 1;
    while (bpb > 1 && (B + bpb - 1) / bpb < 2 * 148) bpb >>= 1;
    // keep at least one full warp per CTA where possible
    while (bpb * nmul < 32 && bpb * 2 * nmul <= 128 && bpb * 2 <= B) bpb <<= 1;
    return bpb;
}

int make_kdesc(const hbv_desc_t* s, KDesc& d) {
    if (!s) { set_error("null descriptor"); return HBV_E_NULL; }
    if (s->abi_version != HBV_B200_ABI_VERSION) { set_error("ABI version mismatch"); return HBV_E_ABI; }
    const int np = expected_npar(s->variant, s->betaet);
    if (np < 0) { set_error("unknown variant"); return HBV_E_VARIANT; }
    if (s->n_par != np) { set_error("n_par does not match variant"); return HBV_E_SHAPE; }
    if (s->T <= 0 || s->B <= 0 || s->nvar <= 0 || s->dyn_ncol < 0 || s->sta_ncol < 0) { set_error("non-positive dimension"); return HBV_E_SHAPE; }
    if (s->nmul <= 0 || s->nmul > 256) { set_error("nmul must be in [1, 256]"); return HBV_E_NMUL; }
    if (s->i_prcp < 0 || s->i_prcp >= s->nvar || s->i_tmean < 0 || s->i_tmean >= s->nvar ||
        s->i_pet < 0 || s->i_pet >= s->nvar) { set_error("forcing column out of range"); return HBV_E_SHAPE; }
    if (s->ckpt_interval < 0) { set_error("negative ckpt_interval"); return HBV_E_CKPT; }
    for (int i = 0; i < np; ++i) {
        const int src = s->par_src[i];
        if (src < HBV_SRC_DYN_T || src > HBV_SRC_STA) { set_error("bad par_src"); return HBV_E_SHAPE; }
        const int ncol = (src == HBV_SRC_STA) ? s->sta_ncol : s->dyn_ncol;
        if (s->par_col[i] < 0 || s->par_col[i] + s->nmul > ncol) { set_error("parameter column out of range"); return HBV_E_SHAPE; }
    }
    std::memset(&d, 0, sizeof(d));
    d.T = s->T; d.B = s->B; d.nmul = s->nmul; d.n_par = np;
    d.nvar = s->nvar; d.i_prcp = s->i_prcp; d.i_tmean = s->i_tmean; d.i_pet = s->i_pet;
    d.dyn_ncol = s->dyn_ncol; d.sta_ncol = s->sta_ncol; d.apply_sigmoid = s->apply_sigmoid;
    d.K = s->ckpt_interval; d.muwts_t_stride = s->muwts_t_stride;
    if (s->ckpt_layout != 0 && s->ckpt_layout != 1) { set_error("ckpt_layout must be 0 or 1"); return HBV_E_CKPT; }
    d.ck_layout = s->ckpt_layout;
    d.nearzero = s->nearzero; d.dt = s->dt; d.inv_dt = 1.0f / s->dt;
    d.BPB = choose_bpb(s->B, s->nmul);
    for (int i = 0; i < np; ++i) {
        d.src[i] = s->par_src[i]; d.col[i] = s->par_col[i];
        d.lo[i] = s->par_lo[i]; d.span[i] = s->par_hi[i] - s->par_lo[i];
    }
    return 0;
}

}  // namespace hbv

extern "C" {

int hbv_b200_abi_version(void) { return HBV_B200_ABI_VERSION; }
const char* hbv_b200_last_error(void) { return hbv::g_err; }
int64_t hbv_b200_launch_count(void) { return (int64_t)hbv::g_launches.load(); }
int64_t hbv_b200_dense_launches(void) { return (int64_t)hbv::g_dense_launches.load(); }
int64_t hbv_b200_lean_launches(void) { return (int64_t)hbv::g_lean_launches.load(); }
int64_t hbv_b200_pipe_launches(void) { return (int64_t)hbv::g_pipe_launches.load(); }

int hbv_b200_set_option(const char* name, int64_t value) {
    const int i = hbv::opt_index(name);
    if (i < 0) { hbv::set_error("unknown option"); return HBV_E_SHAPE; }
    hbv::opt_init();
    hbv::g_opt[i].store((long long)value, std::memory_order_relaxed);
    return 0;
}
int64_t hbv_b200_get_option(const char* name) {
    const int i = hbv::opt_index(name);
    if (i < 0) { hbv::set_error("unknown option"); return INT64_MIN; }
    return (int64_t)hbv::opt((hbv::Opt)i);
}

int hbv_b200_auto_ckpt(int32_t T, int32_t B, int32_t nmul) {
    // Store every state (20 B per lane-step) whenever that fits 16 GiB of the 180 GB HBM: the
    // adjoint then needs no recompute pass — a third of its instructions and, with many
    // time-varying parameters, a second read of the parameter tensor that costs more HBM bytes
    // than the states do (measured on B200: hbv_1_1p all-dynamic 22.5k basins, K 16 -> 1:
    // fwd 4.2 -> 4.8 ms, bwd 11.2 -> 7.4 ms).  Longer or wider runs fall back to K = 16.
    if (hbv::opt(hbv::OPT_CKPT) >= 1) return (int)hbv::opt(hbv::OPT_CKPT);
    const long long lanes = (long long)B * nmul;
    if (lanes * T * 20 <= (16LL << 30)) return 1;
    return 16;
}

int hbv_b200_auto_ckpt_desc(const hbv_desc_t* desc) {
    // The interval for one concrete run.  Every state (K = 1) is the default (hbv_b200_auto_ckpt).
    // Runs the standard-layout kernels serve (nmul 16, 3-wide x_phy, the shipped dynamic sets) have
    // a second option, the segment sweep of K1s / K2s with K = 4: three of four states are
    // recomputed in registers instead of travelling through HBM.  Measured on B200 (`hbv`, dynamic
    // [parBETA, parBETAET], fwd + bwd step, K = 1 / 2 / 4): 531 basins 0.67 / 0.67 / 0.69 ms,
    // 5,000: 2.19 / 1.96 / 1.86, 10,000: 4.57 / 3.53 / 3.22, 22,500: 8.38 / 7.51 / 6.99 —
    // so K = 4 from four warps per scheduler up.  The hourly model's adjoint is issue-bound
    // earlier (2,500 units: 25.1 / 27.8 / 33.0 ms) and keeps K = 1 while the states fit.
    if (!desc) { hbv::set_error("null descriptor"); return HBV_E_NULL; }
    const int base = hbv_b200_auto_ckpt(desc->T, desc->B, desc->nmul);
    if (hbv::opt(hbv::OPT_CKPT) >= 1) return base;
    if (desc->nmul != 16 || desc->nvar != 3 || hbv::opt(hbv::OPT_LEAN) == 0) return base;
    int dm = 0;
    for (int i = 0; i < desc->n_par && i < HBV_MAX_PAR; ++i)
        if (desc->par_src[i] == HBV_SRC_DYN_T) dm |= 1 << i;
    const bool packed = desc->variant == HBV_VARIANT_HBV || desc->variant == HBV_VARIANT_HBV11P;
    const bool lean_set = packed ? (dm == hbv::DM_D2 && desc->betaet) : (dm == hbv::DM_D3);
    if (!lean_set) return base;
    const long long lanes = (long long)desc->B * desc->nmul;
    if (base == 1) return (desc->variant != HBV_VARIANT_HOURLY && lanes >= 148LL * 4 * 32 * 4) ? 4 : 1;
    // the states of a K = 1 run would not fit 16 GiB: K = 4 while a quarter of them fits 32 GiB
    return (lanes * desc->T * 20 / 4 <= (32LL << 30)) ? 4 : base;
}

int64_t hbv_b200_workspace_bytes(const hbv_desc_t* desc) {
    if (!desc) { hbv::set_error("null descriptor"); return HBV_E_NULL; }
    if (desc->T <= 0 || desc->B <= 0 || desc->nmul <= 0) { hbv::set_error("non-positive dimension"); return HBV_E_SHAPE; }
    if (desc->ckpt_interval < 0) { hbv::set_error("negative ckpt_interval"); return HBV_E_CKPT; }
    const int K = desc->ckpt_interval > 0 ? desc->ckpt_interval : hbv_b200_auto_ckpt(desc->T, desc->B, desc->nmul);
    const int64_t nseg = ((int64_t)desc->T + K - 1) / K;
    const int64_t nlane = (int64_t)desc->B * desc->nmul;
    // warp-major layout: whole 32-lane groups
    const int64_t lanes = desc->ckpt_layout == 1 ? (nlane + 31) / 32 * 32 : nlane;
    return nseg * 5 * lanes * (int64_t)sizeof(float);
}

int hbv_b200_fwd(const hbv_desc_t* desc, const hbv_fwd_io_t* io, void* stream) {
    if (!desc || !io) { hbv::set_error("null argument"); return HBV_E_NULL; }
    if (desc->variant == HBV_VARIANT_ADJ) { hbv::set_error("HBV_VARIANT_ADJ runs through hbv_b200_adj_fwd"); return HBV_E_VARIANT; }
    if (!io->forcing || !io->state_in) { hbv::set_error("null input pointer"); return HBV_E_NULL; }
    if (desc->variant >= HBV_VARIANT_HBV2 && !io->attrs) { hbv::set_error("attrs (Ac, Elevation) required"); return HBV_E_NULL; }
    for (int i = 0; i < desc->n_par && i < HBV_MAX_PAR; ++i)
        if (desc->par_src[i] == HBV_SRC_STA ? !io->sta : !io->dyn) { hbv::set_error("parameter tensor required"); return HBV_E_NULL; }
    if (io->ckpt && desc->ckpt_interval <= 0) { hbv::set_error("ckpt buffer without ckpt_interval"); return HBV_E_CKPT; }
    return hbv::fwd_dispatch(desc, io, (cudaStream_t)stream);
}

int hbv_b200_bwd(const hbv_desc_t* desc, const hbv_bwd_io_t* io, void* stream) {
    if (!desc || !io) { hbv::set_error("null argument"); return HBV_E_NULL; }
    if (desc->variant == HBV_VARIANT_ADJ) { hbv::set_error("HBV_VARIANT_ADJ runs through hbv_b200_adj_bwd"); return HBV_E_VARIANT; }
    if (!io->forcing || !io->ckpt) { hbv::set_error("null input pointer"); return HBV_E_NULL; }
    if (desc->variant >= HBV_VARIANT_HBV2 && !io->attrs) { hbv::set_error("attrs (Ac, Elevation) required"); return HBV_E_NULL; }
    for (int i = 0; i < desc->n_par && i < HBV_MAX_PAR; ++i)
        if (desc->par_src[i] == HBV_SRC_STA ? (!io->sta || !io->gsta) : (!io->dyn || !io->gdyn)) { hbv::set_error("parameter tensor + gradient required"); return HBV_E_NULL; }
    return hbv::bwd_dispatch(desc, io, (cudaStream_t)stream);
}

int hbv_b200_tlm(const hbv_desc_t* desc, const hbv_tlm_io_t* io, void* stream) {
    if (!desc || !io) { hbv::set_error("null argument"); return HBV_E_NULL; }
    if (desc->variant == HBV_VARIANT_ADJ) { hbv::set_error("hbv_b200_tlm does not serve HBV_VARIANT_ADJ"); return HBV_E_VARIANT; }
    if (!io->forcing || !io->state_in) { hbv::set_error("null input pointer"); return HBV_E_NULL; }
    if (desc->variant >= HBV_VARIANT_HBV2 && !io->attrs) { hbv::set_error("attrs (Ac, Elevation) required"); return HBV_E_NULL; }
    for (int i = 0; i < desc->n_par && i < HBV_MAX_PAR; ++i)
        if (desc->par_src[i] == HBV_SRC_STA ? !io->sta : !io->dyn) { hbv::set_error("parameter tensor required"); return HBV_E_NULL; }
    return hbv::tlm_dispatch(desc, io, (cudaStream_t)stream);
}

int hbv_b200_adj_fwd(const hbv_desc_t* desc, const hbv_adj_fwd_io_t* io, void* stream) {
    if (!desc || !io) { hbv::set_error("null argument"); return HBV_E_NULL; }
    if (desc->variant != HBV_VARIANT_ADJ) { hbv::set_error("hbv_b200_adj_fwd needs HBV_VARIANT_ADJ"); return HBV_E_VARIANT; }
    if (!io->forcing || !io->dyn || !io->state_in) { hbv::set_error("null input pointer"); return HBV_E_NULL; }
    return hbv::adj_fwd_dispatch(desc, io, (cudaStream_t)stream);
}

int hbv_b200_adj_bwd(const hbv_desc_t* desc, const hbv_adj_bwd_io_t* io, void* stream) {
    if (!desc || !io) { hbv::set_error("null argument"); return HBV_E_NULL; }
    if (desc->variant != HBV_VARIANT_ADJ) { hbv::set_error("hbv_b200_adj_bwd needs HBV_VARIANT_ADJ"); return HBV_E_VARIANT; }
    if (!io->forcing || !io->dyn || !io->ysol) { hbv::set_error("null input pointer"); return HBV_E_NULL; }
    if (!io->gdyn) {
        if (io->gdyn_zero_fill) { hbv::set_error("adj_bwd: gdyn_zero_fill needs gdyn"); return HBV_E_SHAPE; }
        if (!io->gforcing && !io->gstate_in) { hbv::set_error("adj_bwd: no output (gdyn, gforcing and gstate_in all NULL)"); return HBV_E_NULL; }
    }
    return hbv::adj_bwd_dispatch(desc, io, (cudaStream_t)stream);
}

}  // extern "C"
