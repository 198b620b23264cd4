"""PyTorch-facing operators over the C-ABI CUDA library.

``hbv_run`` is the `_PBM` replacement (hbv.py:363-596 and siblings): one
``torch.autograd.Function`` whose forward launches K1 (fused recurrence) + K4
(UH routing + BFI) and whose backward launches K4's adjoint + K2 (checkpointed
adjoint of the recurrence) — no autograd tape over time steps.

PyTorch is used for device memory, streams and autograd plumbing only; all
arithmetic happens in ``libhbv_b200.so``.  There is no CPU fallback.
"""

from __future__ import annotations

import ctypes as C
import os
import threading
from dataclasses import dataclass, field
from typing import Optional, Sequence

import torch
import torch.autograd.forward_ad as fwAD

from . import _cabi as A

_ROUTED = (A.F_QSIM, A.F_Q0, A.F_Q1, A.F_Q2)

# Optional per-call device timing (bench.py): when PROFILE is a dict, every C-ABI call is
# bracketed by CUDA events recorded on the stream the kernels are launched on.
PROFILE = None

# How the dense [T_total, B, ncol] parameter-gradient tensor gets its zeros:
#   False (default): allocated and memset on a side stream while the forward kernel runs (the
#                    forward is FP32-issue bound and leaves HBM idle, so the memset is hidden);
#   True:            K2 writes every element itself (hbv_bwd_io_t.gdyn_zero_fill = 1);
#   None (auto):     fused when at least half of the columns are time-varying parameters — K2
#                    overwrites most of the tensor anyway and a memset would double the HBM
#                    writes of an HBM-bound run (hbv_1_1p all-dynamic: 14.8 GB per step at the
#                    22.5k-basin shard) — and for nmul 16 with an even row width (K2s zeroes its
#                    rows itself); side-stream memset otherwise.
#   Environment override for experiments: HBV_B200_FUSED_ZERO=0/1.
FUSED_ZERO_FILL = {'0': False, '1': True}.get(os.environ.get('HBV_B200_FUSED_ZERO', ''), None)


def _fused_zero_fill(spec, dyn_ncol, n_basins) -> bool:
    if dyn_ncol > 32 * spec.nmul:      # K2's per-thread zero map covers 32 elements per thread
        return False
    if FUSED_ZERO_FILL is not None:
        return bool(FUSED_ZERO_FILL)
    n_dyn = sum(1 for s in spec.par_src[:spec.n_par] if s == A.SRC_DYN_T)
    if 2 * n_dyn * spec.nmul >= dyn_ncol:
        return True
    # nmul 16, even row width: the one-warp adjoint zeroes a step's rows itself before it writes the
    # gradients — K2s with a handful of 8 B stores (22.5k-basin shard: step 10.7 -> 9.4 ms against
    # a memset that competes with the forward kernels for HBM).  On small, latency-bound grids the
    # in-order memset is cheaper: plain stores sit in the single warp's critical path (K2s: 0.57 vs
    # 0.56 ms), and K2p's variant — ONE TMA bulk store per row from a zeroed shared-memory buffer,
    # warm-up rows included (gdyn_rows_before; HBV_B200_BULK_ZERO=1) — was measured slower too.
    if spec.nmul != 16 or dyn_ncol % 2 != 0:
        return False
    lanes = n_basins * spec.nmul
    return lanes > _SMALL_GRID_LANES or (BULK_ZERO_FILL and lanes <= _PIPE_LANES)

# small grids: zero the gradient plane with the library's thin fill kernel on the side stream
# instead of a memset in stream order.  Off by default — measured on B200 (C2): even a fill that
# issues next to no instructions (TMA bulk stores, csrc/fill.cu) slows the latency-bound recurrence
# kernels it runs next to through the memory system; graph-replayed step 0.77 vs 0.47 ms.
THIN_FILL = os.environ.get('HBV_B200_THIN_FILL', '0') == '1'
_SIDE_STREAMS = {}
_SMALL_GRID_LANES = 148 * 4 * 32 * 2      # same boundary as the kernels' small-grid regime
_PIPE_LANES = 148 * 4 * 32                # K1p / K2p regime (csrc/hbv_pipe.cu: one warp per scheduler)
# Off by default: measured on B200 (C2) the zeros written from inside K2p — one TMA bulk store per
# row, 4 or 16 iterations ahead of the gradient stores — slow the sweep from 171 to 326 us (the
# step 0.465 -> 0.549 ms): 489 MB of extra write traffic next to a latency-bound kernel costs
# more than the 76 us in-order memset it replaces.
BULK_ZERO_FILL = os.environ.get('HBV_B200_BULK_ZERO', '0') == '1'


def _ckpt_layout(spec, n_basins: int, K: int) -> int:
    """hbv_desc_t.ckpt_layout of a training run's state store: warp-major (1) where the
    standard-layout kernels serve the run with the chunk-ring forward (grids above two warps per
    scheduler) and K = 1 or 4 — the five states of a stored step then sit at immediate offsets from
    one pointer (K1s 10, K2s 7 instructions per step less; BASELINE config 4's per-GPU grid: step
    21.27 -> 20.69 ms).  Planes (0) otherwise: K1p / K2p, the one-warp K1s, and the TMA-staged
    K1d / K2d (all parameters time-varying) move CTA-wide state rows.  The generic K1 / K2 read
    either.  Option `ckpt_layout` (HBV_B200_CKPT_LAYOUT) forces 0 / 1."""
    forced = int(A.load().hbv_b200_get_option(b'ckpt_layout'))
    if forced in (0, 1):
        return forced
    if spec.nmul != 16 or n_basins * spec.nmul <= _SMALL_GRID_LANES or K not in (1, 4):
        return 0
    n_dyn = sum(1 for s in spec.par_src[:spec.n_par] if s == A.SRC_DYN_T)
    if n_dyn == spec.n_par or int(A.load().hbv_b200_get_option(b'dense')) == 2:
        return 0
    return 1


def _side_stream(dev):
    key = (dev.type, dev.index)
    if key not in _SIDE_STREAMS:
        _SIDE_STREAMS[key] = torch.cuda.Stream(dev)
    return _SIDE_STREAMS[key]


class _timed:
    def __init__(self, name, dev):
        self.name, self.dev = name, dev

    def __enter__(self):
        if PROFILE is not None:
            self.e0 = torch.cuda.Event(enable_timing=True)
            self.e1 = torch.cuda.Event(enable_timing=True)
            self.e0.record(torch.cuda.current_stream(self.dev))
        return self

    def __exit__(self, *exc):
        if PROFILE is not None:
            self.e1.record(torch.cuda.current_stream(self.dev))
            PROFILE.setdefault(self.name, []).append((self.e0, self.e1))
        return False


@dataclass
class RunSpec:
    """Everything static about one `_PBM` call (mirrors hbv_desc_t)."""

    variant: int
    n_par: int
    betaet: bool
    apply_sigmoid: bool
    par_src: Sequence[int]
    par_col: Sequence[int]
    par_lo: Sequence[float]
    par_hi: Sequence[float]
    nmul: int
    nflux: int
    nearzero: float = 1e-5
    dt: float = 1.0
    var_index: Sequence[int] = (0, 1, 2)   # prcp, tmean, pet columns
    ckpt_interval: int = 0     # 0 = auto (hbv_b200_auto_ckpt)
    # routing (core/calc/uh_routing.py); route_src: 'dyn_last' (packed) or 'sta' (split)
    routing: bool = False
    route_src: str = 'dyn_last'
    route_col: int = 0
    route_bounds: Sequence[Sequence[float]] = ((0, 2.9), (0, 6.5))
    lenF: int = 15
    n_routed: int = 4          # series routed: Qsim, Q0, Q1, Q2 (hourly: Qsim only)
    bfi: bool = True
    state_series: bool = False
    extra: dict = field(default_factory=dict)


def _ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


def _stream(dev) -> int:
    return torch.cuda.current_stream(dev).cuda_stream


def _check_cuda(t: torch.Tensor, name: str) -> None:
    if not t.is_cuda:
        raise RuntimeError(
            f"hydrodl2_b200: `{name}` is on {t.device}; this implementation runs on CUDA "
            "(sm_100a) only — there is no CPU path."
        )
    if t.dtype != torch.float32:
        raise RuntimeError(f"hydrodl2_b200: `{name}` must be float32, got {t.dtype}")


def make_desc(spec: RunSpec, T: int, B: int, nvar: int, dyn_ncol: int, sta_ncol: int,
              muwts_t_stride: int = 0) -> A.HbvDesc:
    d = A.HbvDesc()
    d.abi_version = A.ABI_VERSION
    d.variant = spec.variant
    d.T, d.B, d.nmul, d.n_par = T, B, spec.nmul, spec.n_par
    d.betaet = int(spec.betaet)
    d.apply_sigmoid = int(spec.apply_sigmoid)
    d.nvar = nvar
    d.i_prcp, d.i_tmean, d.i_pet = spec.var_index
    d.dyn_ncol, d.sta_ncol = dyn_ncol, sta_ncol
    n = spec.n_par       # (slice assignment: one ctypes call per array, not one per element)
    d.par_src[:n] = spec.par_src[:n]
    d.par_col[:n] = spec.par_col[:n]
    d.par_lo[:n] = [float(v) for v in spec.par_lo[:n]]
    d.par_hi[:n] = [float(v) for v in spec.par_hi[:n]]
    d.nearzero = spec.nearzero
    d.dt = spec.dt
    d.ckpt_interval = spec.ckpt_interval
    d.muwts_t_stride = muwts_t_stride
    return d


def make_route_desc(spec: RunSpec, T: int, B: int, stride: int) -> A.HbvRouteDesc:
    r = A.HbvRouteDesc()
    r.abi_version = A.ABI_VERSION
    r.T, r.B, r.lenF, r.nser = T, B, spec.lenF, spec.n_routed
    r.apply_sigmoid = int(spec.apply_sigmoid)
    r.route_stride = stride
    r.bfi_num, r.bfi_den = 3, 0   # 100 * sum(Q2_rout) / (sum(Qs) + nearzero), hbv.py:562-567
    (r.a_lo, r.a_hi), (r.b_lo, r.b_hi) = spec.route_bounds
    r.nearzero = spec.nearzero
    return r


def _prep_muwts(muwts, T, B, nmul, dev):
    """-> (contiguous tensor or None, time stride in elements)."""
    if muwts is None:
        return None, 0
    m = muwts.detach().to(device=dev, dtype=torch.float32)
    if m.dim() == 3 and m.shape[0] == T and T > 1:
        return m.expand(T, B, nmul).contiguous(), B * nmul
    return m.expand(1, B, nmul).contiguous() if m.dim() == 3 else m.expand(B, nmul).contiguous(), 0


def hbv_states_only(spec: RunSpec, forcing, dyn, sta, state_in, drop=None, attrs=None):
    """Warm-up / `initialize=True` run (hbv.py:327-346,557-559): no flux output, no
    checkpoints, no gradient.  Returns the final state stack [5, B, nmul]."""
    lib = A.load()
    _check_cuda(forcing, 'x_phy')
    T, B, nvar = forcing.shape
    d = make_desc(spec, T, B, nvar, 0 if dyn is None else dyn.shape[-1],
                  0 if sta is None else sta.shape[-1])
    d.ckpt_interval = 0
    io = A.HbvFwdIO()
    state_out = torch.empty_like(state_in)
    io.forcing, io.dyn, io.sta = _ptr(forcing), _ptr(dyn), _ptr(sta)
    io.drop, io.attrs, io.muwts = _ptr(drop), _ptr(attrs), None
    io.state_in, io.state_out = _ptr(state_in), _ptr(state_out)
    with torch.cuda.device(forcing.device):
        with _timed('hbv_fwd_warmup', forcing.device):
            A.check(lib.hbv_b200_fwd(C.byref(d), C.byref(io), _stream(forcing.device)), 'fwd(warm-up)')
    return state_out


def is_dual(*tensors) -> bool:
    """True when any of `tensors` carries a forward-mode tangent (torch.autograd.forward_ad)."""
    for t in tensors:
        if isinstance(t, torch.Tensor) and fwAD.unpack_dual(t).tangent is not None:
            return True
    return False


def refuse_forward_ad(what: str, *tensors) -> None:
    """Raise NotImplementedError when a path that cannot carry tangents gets dual inputs, instead
    of returning outputs whose tangent silently misses a contribution."""
    if is_dual(*tensors):
        raise NotImplementedError(f'hydrodl2_b200: forward-mode AD (torch.autograd.forward_ad) is not '
                                  f'supported through {what}')


class _StatesOnly(torch.autograd.Function):
    """The warm-up run with forward-mode tangents: forward = hbv_states_only (K1 without flux
    outputs), jvp = K1t in states-only mode.  The reference runs its warm-up under no_grad without
    a detach (hbv.py:327-346), and no_grad does not stop forward-mode tangents, so the tangents of
    the warm-up's forcings, parameters and initial states reach the run's initial states.  No
    reverse-mode gradient, as before."""

    @staticmethod
    def forward(ctx, spec, forcing, dyn, state_in):
        ctx.spec = spec
        ctx.save_for_forward(forcing, dyn, state_in)
        return hbv_states_only(spec, forcing, dyn, None, state_in)

    @staticmethod
    def jvp(ctx, _spec_t, forcing_t, dyn_t, state_in_t):
        lib = A.load()
        spec = ctx.spec
        forcing, dyn, state_in = ctx.saved_tensors
        T, B, nvar = forcing.shape
        d = make_desc(spec, T, B, nvar, dyn.shape[-1], 0)
        d.ckpt_interval = 0
        cont = (lambda t: None if t is None else t.to(dtype=torch.float32).contiguous())
        forcing_t, dyn_t, state_in_t = cont(forcing_t), cont(dyn_t), cont(state_in_t)
        state_out_t = torch.empty_like(state_in)
        io = A.HbvTlmIO()
        io.forcing, io.dyn, io.state_in = _ptr(forcing), _ptr(dyn), _ptr(state_in)
        io.forcing_t, io.dyn_t, io.state_in_t = _ptr(forcing_t), _ptr(dyn_t), _ptr(state_in_t)
        io.state_out_t = _ptr(state_out_t)
        with torch.cuda.device(forcing.device):
            with _timed('hbv_tlm_warmup', forcing.device):
                A.check(lib.hbv_b200_tlm(C.byref(d), C.byref(io), _stream(forcing.device)), 'tlm(warm-up)')
        return state_out_t

    @staticmethod
    def backward(ctx, _g):
        return None, None, None, None


def hbv_states_only_dual(spec: RunSpec, forcing, dyn, state_in):
    """hbv_states_only for dual inputs (packed models' warm-up under forward-mode AD): the final
    state stack carries the tangent of the warm-up.  Runs under no_grad (no reverse-mode gradient
    through the warm-up, as in the plain path)."""
    _check_cuda(forcing, 'x_phy')
    with torch.no_grad():
        return _StatesOnly.apply(spec, forcing.contiguous(), dyn.contiguous(), state_in.contiguous())


# ---- clean gradient planes kept between steps ---------------------------------------------------
# On small, latency-bound grids the dense gradient plane is zeroed by an in-order memset (above):
# 488 MB = 76 us of BASELINE config 2's 437 us step, although the adjoint rewrites every entry that
# can be non-zero (the dynamic blocks of the run's rows, the last row) at every step and the rest
# never changes.  So the library keeps the plane it handed out and hands it out again — WITHOUT the
# memset — when that is provably the same as a fresh zeroed one:
#   * same shape / device / run plan (the set of entries the adjoint writes), no dropout mask;
#   * nobody else references its storage any more (the previous gradient, every view of it, has
#     been released: torch._C._storage_Use_Count back at the value measured when only the cache
#     held it);
#   * it has not been modified in place since (the handed-out tensor is an alias that shares the
#     cached tensor's version counter; the library's own kernels write through raw pointers).
# Anything else gets a new zeroed plane.  A plane handed out during CUDA-graph capture is pinned
# for the life of the process (the graph replays into it).  HBV_B200_REUSE_GRAD_PLANE=0 switches
# the cache off.
# (needs torch's storage use count; without that private hook every step gets a fresh plane)
REUSE_GRAD_PLANE = (os.environ.get('HBV_B200_REUSE_GRAD_PLANE', '1') == '1'
                    and hasattr(torch._C, '_storage_Use_Count'))
_PLANES_LOCK = threading.RLock()
_PLANES: dict = {}          # key -> list of [base tensor, version when clean, storage use count when idle, pinned]
_PLANES_PER_KEY = 2         # (double-buffered loops keep two gradients alive)
_PLANE_KEYS = 4             # run plans remembered (oldest forgotten first; pinned planes stay)


def _storage_refs(t: torch.Tensor) -> int:
    return int(torch._C._storage_Use_Count(t.untyped_storage()._cdata))


# idle planes kept in total, bytes (a 22,500-basin shard's plane is 20.7 GB); HBV_B200_PLANE_CACHE_GB
_PLANE_BYTES_MAX = int(float(os.environ.get('HBV_B200_PLANE_CACHE_GB', '48')) * (1 << 30))


def release_grad_planes() -> None:
    """Let go of every cached gradient plane no CUDA graph replays into (their memory returns to
    PyTorch's allocator once the last gradient aliasing them is released)."""
    with _PLANES_LOCK:
        for k in list(_PLANES):
            _PLANES[k] = [e for e in _PLANES[k] if e[3]]
            if not _PLANES[k]:
                del _PLANES[k]



def _plane_key(spec: RunSpec, dyn: torch.Tensor, t_off: int):
    return (dyn.device, tuple(dyn.shape), t_off, spec.variant, spec.nmul, spec.n_par, tuple(spec.par_src[:spec.n_par]),
            tuple(spec.par_col[:spec.n_par]), spec.routing, spec.route_src, spec.route_col)


def _lookup_plane(spec: RunSpec, dyn: torch.Tensor, t_off: int):
    """An alias of a cached plane that is provably clean, or None."""
    with _PLANES_LOCK:
        ents = _PLANES.get(_plane_key(spec, dyn, t_off))
        if not ents:
            return None
        capturing = torch.cuda.is_current_stream_capturing()
        for e in ents:
            base, ver, idle, pinned = e
            if not pinned and base._version == ver and _storage_refs(base) == idle:
                if capturing:
                    e[3] = True
                out = base.detach()
                out._hbv_clean_plane = True
                return out
        return None


def _register_plane(spec: RunSpec, dyn: torch.Tensor, t_off: int, base: torch.Tensor):
    """Remember `base` — every entry of it initialised, only this reference to its storage alive —
    and return the alias to hand out."""
    key = _plane_key(spec, dyn, t_off)
    nbytes = base.numel() * base.element_size()
    if nbytes > _PLANE_BYTES_MAX:
        return base
    with _PLANES_LOCK:
        return _register_plane_locked(key, nbytes, base)


def _register_plane_locked(key, nbytes: int, base: torch.Tensor):
    ents = _PLANES.get(key)
    if ents is None:
        ents = _PLANES[key] = []
        for k in list(_PLANES)[:-_PLANE_KEYS]:            # forget the oldest run plans' idle planes
            _PLANES[k] = [e for e in _PLANES[k] if e[3]]
            if not _PLANES[k]:
                del _PLANES[k]
    ent = [base, base._version, _storage_refs(base), torch.cuda.is_current_stream_capturing()]
    ents.append(ent)
    per_key = 1 if nbytes > (2 << 30) else _PLANES_PER_KEY
    while sum(1 for e in ents if not e[3]) > per_key:            # forget the oldest plane no graph replays into
        i = next(i for i, e in enumerate(ents) if not e[3] and e is not ent)
        del ents[i]

    def idle_bytes():
        return sum(e[0].numel() * 4 for v in _PLANES.values() for e in v if not e[3])
    for k in list(_PLANES):                                      # total budget: oldest run plans first
        if idle_bytes() <= _PLANE_BYTES_MAX:
            break
        if k != key:
            _PLANES[k] = [e for e in _PLANES[k] if e[3]]
    out = base.detach()
    out._hbv_clean_plane = True
    return out


def _clean_plane(spec: RunSpec, dyn: torch.Tensor, t_off: int):
    """-> (plane, reused): an alias of a cached clean plane, or a new zeroed one (now cached)."""
    hit = _lookup_plane(spec, dyn, t_off)
    if hit is not None:
        return hit, True
    return _register_plane(spec, dyn, t_off, torch.zeros_like(dyn, requires_grad=False)), False


def start_grad_plane(spec: RunSpec, dyn: Optional[torch.Tensor], t_off: int = 0, _checked: bool = False,
                     reusable: bool = True):
    """Allocate the dense gradient plane of `dyn` and start zeroing what the adjoint will not write
    on the side stream right away: everything (memset mode) or, when the adjoint writes its rows
    itself, the warm-up rows [:t_off] and the routing columns of the last row.  A model with a
    warm-up run calls this BEFORE the warm-up kernel, which moves almost no HBM bytes, so the fill
    overlaps it instead of K1 / K2.  Returns (plane, event or None, fused) for
    `hbv_run(gplane=...)`, or None when there is nothing to prepare."""
    if not _checked:      # (_HbvRun.forward has made these checks itself; grad mode is off in there)
        if dyn is None or not dyn.is_cuda or not (torch.is_grad_enabled() and dyn.requires_grad):
            return None
    fused = _fused_zero_fill(spec, dyn.shape[-1], dyn.shape[1])
    if fused and reusable and REUSE_GRAD_PLANE:
        # the adjoint would write every element of the run's rows itself (zeros included); a clean
        # plane kept from an earlier step needs none of that: the adjoint writes its entries only
        hit = _lookup_plane(spec, dyn, t_off)
        if hit is not None:
            return hit, None, False
    if fused and t_off == 0:
        return None           # only the routing columns of one row: the backward clears them in order
    if fused and dyn.shape[1] * spec.nmul <= _PIPE_LANES:
        return None           # K2p zeroes the warm-up rows itself (gdyn_rows_before, see backward)
    dev = dyn.device
    small = dyn.shape[1] * spec.nmul <= _SMALL_GRID_LANES
    if small and not fused and not THIN_FILL and reusable and REUSE_GRAD_PLANE:
        gbuf, _ = _clean_plane(spec, dyn, t_off)
        return gbuf, None, fused
    gbuf = torch.empty_like(dyn)

    def fill():
        if fused:
            gbuf[:t_off].zero_()
            if spec.n_par * spec.nmul < dyn.shape[-1]:
                gbuf[dyn.shape[0] - 1, :, spec.n_par * spec.nmul:].zero_()
        else:
            gbuf.zero_()

    if small and THIN_FILL:
        # Latency-bound regime (a warp or two per scheduler): a full-occupancy memset running next
        # to the recurrence kernels starves them for longer than the fill itself takes (C2: a 76 us
        # memset stretched the 88 us warm-up kernel to 275 us), and in stream order it is 76 us of
        # the critical path.  The library's thin fill (csrc/fill.cu: one warp per SM streaming TMA
        # bulk stores of a zeroed shared-memory buffer, next to no instruction issue) runs on the
        # side stream underneath the warm-up and forward kernels instead.
        lib = A.load()
        cur = torch.cuda.current_stream(dev)
        side = _side_stream(dev)
        side.wait_stream(cur)
        with torch.cuda.stream(side):
            rows = t_off if fused else dyn.shape[0]
            nbytes = rows * dyn.shape[1] * dyn.shape[2] * 4
            with _timed('grad_plane_fill', dev):
                A.check(lib.hbv_b200_fill_zero(gbuf.data_ptr(), nbytes, 0, side.cuda_stream), 'fill_zero')
            if fused and spec.n_par * spec.nmul < dyn.shape[-1]:
                gbuf[dyn.shape[0] - 1, :, spec.n_par * spec.nmul:].zero_()
            gev = torch.cuda.Event()
            gev.record(side)
        return gbuf, gev, fused
    if small:
        fill()      # (HBV_B200_THIN_FILL=0: the round-1 behaviour, a memset in stream order)
        return gbuf, None, fused
    cur = torch.cuda.current_stream(dev)
    side = _side_stream(dev)
    side.wait_stream(cur)
    with torch.cuda.stream(side):
        fill()
        gev = torch.cuda.Event()
        gev.record(side)
    return gbuf, gev, fused


class _HbvRun(torch.autograd.Function):
    """K1 + K4 forward, K4^T + K2 backward."""

    @staticmethod
    def forward(ctx, spec: RunSpec, forcing, dyn, sta, state_in, drop, attrs, muwts, t_off, gplane=None,
                track=True):
        # `dyn` is the FULL dynamic/packed tensor; rows [t_off:] belong to this run.
        lib = A.load()
        dev = forcing.device
        T, B, nvar = forcing.shape
        nmul = spec.nmul
        dyn_run = dyn[t_off:] if dyn is not None else None
        dyn_ncol = 0 if dyn is None else dyn.shape[-1]
        sta_ncol = 0 if sta is None else sta.shape[-1]
        mu, mu_ts = _prep_muwts(muwts, T, B, nmul, dev)
        d = make_desc(spec, T, B, nvar, dyn_ncol, sta_ncol, mu_ts)
        # `track`: grad mode of the caller (inside an autograd.Function it is always off, and a leaf
        # keeps requires_grad=True under no_grad): inference must not pay for stored states
        need_grad = track and any(t is not None and t.requires_grad for t in (dyn, sta, state_in, forcing, muwts))
        if need_grad and nmul > 128:
            # the adjoint kernels hold at most 128 lanes per CTA (csrc/hbv_bwd.cu): fail here, before
            # the forward has run, not in backward()
            raise RuntimeError(f'hydrodl2_b200: nmul = {nmul} > 128 is supported for inference only '
                               '(run under torch.no_grad(), or use nmul <= 128 for training)')
        if spec.ckpt_interval:
            K = spec.ckpt_interval
        elif spec.state_series:
            # the per-step state series rides on the K = 1 store (see below): keep every state
            K = int(lib.hbv_b200_auto_ckpt(T, B, nmul))
        else:
            K = int(lib.hbv_b200_auto_ckpt_desc(C.byref(d)))      # 0 = auto
        d.ckpt_interval = K
        nseg = (T + K - 1) // K
        # `hbv_2` family: the per-step state series (hbv_2.py:571-575, the state AFTER every step)
        # and the every-state store of the adjoint (the state BEFORE every step) are the same
        # numbers shifted by one step — with K = 1 one [T + 1, 5, B, nmul] buffer serves both (the
        # kernel writes planes 0 .. T-1, the final state becomes plane T): no second 20 B per
        # lane-step stream, and the run stays eligible for the standard-layout kernels.
        alias_series = bool(spec.state_series) and K == 1
        ck_full = None
        ck_layout = 0
        if alias_series:
            ck_full = torch.empty((T + 1, 5, B, nmul), device=dev, dtype=torch.float32)
            ckpt = ck_full[:T]
        else:
            if need_grad:
                ck_layout = _ckpt_layout(spec, B, K)
                d.ckpt_layout = ck_layout
                lanes = (B * nmul + 31) // 32 * 32 if ck_layout else B * nmul
                ckpt = torch.empty((nseg * 5 * lanes,), device=dev, dtype=torch.float32)
            else:
                ckpt = None
                d.ckpt_interval = 0

        # gradient buffer for `dyn`: zeroed on a side stream, overlapping the forward kernel
        gbuf = gev = None
        gfused = False
        if need_grad and dyn is not None and dyn.requires_grad:
            if gplane is None:
                gplane = start_grad_plane(spec, dyn, t_off, _checked=True, reusable=drop is None)
            if gplane is not None:
                gbuf, gev, gfused = gplane    # (possibly started before the warm-up kernel)

        flux = torch.empty((A.HBV_MAX_FLUX, T, B), device=dev, dtype=torch.float32)
        state_out = torch.empty((5, B, nmul), device=dev, dtype=torch.float32)
        series = (torch.empty((5, T, B, nmul), device=dev, dtype=torch.float32)
                  if (spec.state_series and not alias_series) else None)
        io = A.HbvFwdIO()
        io.forcing, io.dyn, io.sta = _ptr(forcing), _ptr(dyn_run), _ptr(sta)
        io.drop, io.attrs, io.muwts = _ptr(drop), _ptr(attrs), _ptr(mu)
        io.state_in, io.state_out = _ptr(state_in), _ptr(state_out)
        flux0, plane = flux.data_ptr(), T * B * 4
        for f in range(spec.nflux):
            io.flux[f] = flux0 + f * plane
        io.state_series, io.ckpt = _ptr(series), _ptr(ckpt)
        stream = _stream(dev)
        with torch.cuda.device(dev):
            with _timed('hbv_fwd', dev):
                A.check(lib.hbv_b200_fwd(C.byref(d), C.byref(io), stream), 'fwd')
            if alias_series:
                ck_full[T].copy_(state_out)
                series = ck_full[1:].permute(1, 0, 2, 3)          # [5, T, B, nmul] view
                if not need_grad:
                    ckpt = None

            routed = uh = bfi = bfi_ws = None
            rdesc = route_t = None
            if spec.routing:
                if spec.route_src == 'dyn_last':
                    route_t = dyn[dyn.shape[0] - 1, :, spec.route_col:]
                    stride = dyn_ncol
                else:
                    route_t = sta[:, spec.route_col:]
                    stride = sta_ncol
                rdesc = make_route_desc(spec, T, B, stride)
                nch = lib.hbv_b200_route_chunks(T, B)
                routed = torch.empty((spec.n_routed, T, B), device=dev, dtype=torch.float32)
                uh = torch.empty((min(spec.lenF, T), B), device=dev, dtype=torch.float32)
                if spec.bfi:
                    bfi = torch.empty((B,), device=dev, dtype=torch.float32)
                    bfi_ws = torch.empty((2, nch, B), device=dev, dtype=torch.float32)
                with _timed('route_fwd', dev):
                    A.check(lib.hbv_b200_route_fwd(C.byref(rdesc), route_t.data_ptr(), flux.data_ptr(),
                                                   T * B, routed.data_ptr(), T * B, uh.data_ptr(),
                                                   _ptr(bfi), _ptr(bfi_ws), stream), 'route_fwd')

        if gev is not None:
            # Everything enqueued on this stream from here on runs after the memset (K1 and the
            # routing above overlap it).  That also makes the buffer safe to hand back to this
            # stream's allocator pool at any later point without `record_stream`, whose deferred
            # reuse forces a fresh multi-GB cudaMalloc every step on large shards.
            torch.cuda.current_stream(dev).wait_event(gev)
        ctx.spec, ctx.t_off, ctx.dims = spec, t_off, (T, B, nvar, dyn_ncol, sta_ncol, mu_ts)
        ctx.K = K
        ctx.ck_layout = ck_layout
        ctx.has = (dyn is not None, sta is not None)
        ctx.muwts_shape = None if muwts is None else tuple(muwts.shape)
        ctx.gbuf, ctx.gev, ctx.gfused = gbuf, gev, gfused
        ctx.save_for_backward(forcing, dyn, sta, drop, attrs, mu, ckpt, flux, uh, bfi_ws, state_in)
        ctx.save_for_forward(forcing, dyn, sta, state_in, drop, attrs, mu, flux, uh, bfi_ws)
        ctx.alias_series = alias_series
        ctx.set_materialize_grads(False)
        outs = list(flux.unbind(0)[:spec.nflux])
        n_r = spec.n_routed if spec.routing else 0
        if n_r:
            outs += list(routed.unbind(0)[:n_r])
        outs.append(bfi)        # None when routing / BFI is off
        outs.append(state_out)
        outs.append(series)     # None unless spec.state_series
        ctx.n_r = n_r
        return tuple(outs)

    @staticmethod
    def jvp(ctx, _spec_t, forcing_t, dyn_t, sta_t, state_in_t, _drop_t, attrs_t, muwts_t, *_rest):
        """Forward mode: K1t (tangent-linear recurrence) + K4t (tangent of the routing and BFI).
        A tangent that is None is a zero tangent (NULL to the kernels).  Returns a tangent for
        every output, laid out like the primal outputs (views of one buffer)."""
        if attrs_t is not None:
            raise NotImplementedError('hydrodl2_b200: forward-mode AD with respect to the catchment '
                                      'attributes (Ac, elevation) is not supported; they enter only '
                                      'through branch conditions and the lateral-flux factor')
        lib = A.load()
        spec: RunSpec = ctx.spec
        forcing, dyn, sta, state_in, drop, attrs, mu, flux, uh, bfi_ws = ctx.saved_tensors
        T, B, nvar, dyn_ncol, sta_ncol, mu_ts = ctx.dims
        dev = forcing.device
        nmul, nf, n_r, t_off = spec.nmul, spec.nflux, ctx.n_r, ctx.t_off
        cont = (lambda t: None if t is None else t.to(dtype=torch.float32).contiguous())
        forcing_t, sta_t, state_in_t = cont(forcing_t), cont(sta_t), cont(state_in_t)
        dyn_t = cont(dyn_t)
        mu_t = None
        if mu is not None and muwts_t is not None:
            mu_t, _ = _prep_muwts(muwts_t, T, B, nmul, dev)
        d = make_desc(spec, T, B, nvar, dyn_ncol, sta_ncol, mu_ts)
        d.ckpt_interval = 0
        flux_t = torch.empty((A.HBV_MAX_FLUX, T, B), device=dev, dtype=torch.float32)
        state_out_t = torch.empty((5, B, nmul), device=dev, dtype=torch.float32)
        series_t = (torch.empty((5, T, B, nmul), device=dev, dtype=torch.float32)
                    if spec.state_series else None)
        io = A.HbvTlmIO()
        io.forcing, io.dyn, io.sta = _ptr(forcing), _ptr(dyn[t_off:] if dyn is not None else None), _ptr(sta)
        io.drop, io.attrs, io.muwts, io.state_in = _ptr(drop), _ptr(attrs), _ptr(mu), _ptr(state_in)
        io.forcing_t, io.sta_t, io.muwts_t = _ptr(forcing_t), _ptr(sta_t), _ptr(mu_t)
        io.dyn_t = _ptr(dyn_t[t_off:] if dyn_t is not None else None)
        io.state_in_t = _ptr(state_in_t)
        for f in range(nf):
            io.flux_t[f] = flux_t.data_ptr() + f * T * B * 4
        io.state_out_t, io.series_t = _ptr(state_out_t), _ptr(series_t)
        stream = _stream(dev)
        routed_t = bfi_t = None
        with torch.cuda.device(dev):
            with _timed('hbv_tlm', dev):
                A.check(lib.hbv_b200_tlm(C.byref(d), C.byref(io), stream), 'tlm')
            if n_r:
                # the routing parameters' tangent: the same columns the primal reads them from
                if spec.route_src == 'dyn_last':
                    route_p = dyn[dyn.shape[0] - 1, :, spec.route_col:]
                    route_pt = None if dyn_t is None else dyn_t[dyn_t.shape[0] - 1, :, spec.route_col:]
                    stride = dyn_ncol
                else:
                    route_p = sta[:, spec.route_col:]
                    route_pt = None if sta_t is None else sta_t[:, spec.route_col:]
                    stride = sta_ncol
                rdesc = make_route_desc(spec, T, B, stride)
                nch = lib.hbv_b200_route_chunks(T, B)
                routed_t = torch.empty((spec.n_routed, T, B), device=dev, dtype=torch.float32)
                bfi_ws_t = None
                if spec.bfi:
                    bfi_t = torch.empty((B,), device=dev, dtype=torch.float32)
                    bfi_ws_t = torch.empty((2, nch, B), device=dev, dtype=torch.float32)
                with _timed('route_tlm', dev):
                    A.check(lib.hbv_b200_route_tlm(
                        C.byref(rdesc), route_p.data_ptr(), _ptr(route_pt), flux.data_ptr(), T * B,
                        flux_t.data_ptr(), T * B, uh.data_ptr(), _ptr(bfi_ws), routed_t.data_ptr(), T * B,
                        _ptr(bfi_t), _ptr(bfi_ws_t), stream), 'route_tlm')
            if series_t is not None and ctx.alias_series:
                # the primal series is a view of the [T + 1, 5, B, nmul] state store: same layout here
                full = torch.empty((T + 1, 5, B, nmul), device=dev, dtype=torch.float32)
                view = full[1:].permute(1, 0, 2, 3)
                view.copy_(series_t)
                series_t = view
        outs = list(flux_t.unbind(0)[:nf])
        if n_r:
            outs += list(routed_t.unbind(0)[:n_r])
        outs.append(bfi_t)
        outs.append(state_out_t)
        outs.append(series_t)
        return tuple(outs)

    @staticmethod
    def backward(ctx, *grads):
        lib = A.load()
        spec: RunSpec = ctx.spec
        forcing, dyn, sta, drop, attrs, mu, ckpt, flux, uh, bfi_ws, state_in = ctx.saved_tensors
        T, B, nvar, dyn_ncol, sta_ncol, mu_ts = ctx.dims
        dev = forcing.device
        nmul, nf, n_r = spec.nmul, spec.nflux, ctx.n_r
        if ckpt is None:
            raise RuntimeError('hydrodl2_b200: backward called but no input required grad')
        g_flux = [None if g is None else g.contiguous() for g in grads[:nf]]
        g_rout = grads[nf:nf + n_r]
        g_bfi, g_state, g_series = grads[nf + n_r], grads[nf + n_r + 1], grads[nf + n_r + 2]
        t_off = ctx.t_off
        stream = _stream(dev)

        # The dense [T_total, B, ncol] parameter gradient is part of the contract.  K2 writes
        # every element of the run's rows itself (fused zero-fill); only the warm-up rows (no
        # gradient, hbv.py:328) and the non-parameter columns of the last row are zeroed here.
        gdyn_full = gdyn_run = None
        zero_fill = 0
        rows_before = 0
        if dyn is not None:
            if ctx.gbuf is not None:
                gdyn_full, ctx.gbuf = ctx.gbuf, None
                zero_fill = 1 if ctx.gfused else 0
                if ctx.gev is not None:
                    torch.cuda.current_stream(dev).wait_event(ctx.gev)
            elif _fused_zero_fill(spec, dyn_ncol, B):
                zero_fill = 1
                gdyn_full = torch.empty_like(dyn)
                if t_off > 0:
                    if B * nmul <= _PIPE_LANES:
                        rows_before = t_off       # zeroed by the call (K2p: bulk stores; else a memset in the library)
                    else:
                        gdyn_full[:t_off].zero_()
                if spec.n_par * nmul < dyn_ncol:
                    gdyn_full[dyn.shape[0] - 1, :, spec.n_par * nmul:].zero_()
            else:
                gdyn_full = torch.zeros_like(dyn)
            gdyn_run = gdyn_full[t_off:]
        gsta = torch.zeros_like(sta) if sta is not None else None

        routed_grads = False
        g_route = None
        with torch.cuda.device(dev):
            if spec.routing and (any(g is not None for g in g_rout) or g_bfi is not None):
                mask = 0
                live = [s for s, g in enumerate(g_rout) if g is not None]
                for s in live:
                    mask |= 1 << s
                if len(live) == 1:
                    # one routed series has a gradient (the usual streamflow loss): hand its
                    # plane to the kernel in place — series s is read at base + s * stride
                    g_keep = g_rout[live[0]].contiguous()
                    g_out_ptr = g_keep.data_ptr() - live[0] * T * B * 4
                else:
                    g_keep = torch.empty((n_r, T, B), device=dev, dtype=torch.float32)
                    for s in live:
                        g_keep[s].copy_(g_rout[s])
                    g_out_ptr = g_keep.data_ptr()
                g_in = torch.empty((n_r, T, B), device=dev, dtype=torch.float32)
                if spec.route_src == 'dyn_last':
                    route_t = dyn[dyn.shape[0] - 1, :, spec.route_col:]
                    g_route = gdyn_full[dyn.shape[0] - 1, :, spec.route_col:]
                    stride = dyn_ncol
                else:
                    route_t = sta[:, spec.route_col:]
                    g_route = gsta[:, spec.route_col:]
                    stride = sta_ncol
                rdesc = make_route_desc(spec, T, B, stride)
                nch = lib.hbv_b200_route_chunks(T, B)
                ws = torch.empty((min(spec.lenF, T), nch, B), device=dev, dtype=torch.float32)
                gb = None if g_bfi is None else g_bfi.contiguous()
                with _timed('route_bwd', dev):
                    A.check(lib.hbv_b200_route_bwd(
                        C.byref(rdesc), route_t.data_ptr(), flux.data_ptr(), T * B, None, T * B,
                        uh.data_ptr(), _ptr(bfi_ws), g_out_ptr, T * B, mask, _ptr(gb),
                        g_in.data_ptr(), T * B, g_route.data_ptr(), ws.data_ptr(), stream), 'route_bwd')
                routed_grads = True
                for s in range(n_r):
                    # a series without upstream gradient (and no BFI term) has an all-zero
                    # adjoint plane: do not make K2 read it
                    live = bool(mask >> s & 1) or (gb is not None and s in (rdesc.bfi_num, rdesc.bfi_den))
                    if not live:
                        continue
                    f = _ROUTED[s]
                    g_flux[f] = g_in[s] if g_flux[f] is None else g_flux[f] + g_in[s]

            if (gdyn_full is not None and getattr(gdyn_full, '_hbv_clean_plane', False) and not routed_grads
                    and spec.routing and spec.route_src == 'dyn_last' and spec.route_col < dyn_ncol):
                # a plane from the clean-plane cache whose routing columns nobody writes in this
                # backward (no routed cotangent): they may hold an earlier step's gradient.  The
                # in-place op also bumps the plane's version counter, so the cache lets go of it.
                gdyn_full[dyn.shape[0] - 1, :, spec.route_col:].zero_()
            d = make_desc(spec, T, B, nvar, dyn_ncol, sta_ncol, mu_ts)
            d.ckpt_interval = ctx.K
            d.ckpt_layout = ctx.ck_layout
            io = A.HbvBwdIO()
            io.forcing, io.dyn, io.sta = _ptr(forcing), _ptr(dyn[t_off:] if dyn is not None else None), _ptr(sta)
            io.drop, io.attrs, io.muwts, io.ckpt = _ptr(drop), _ptr(attrs), _ptr(mu), _ptr(ckpt)
            for f in range(nf):
                io.gflux[f] = _ptr(g_flux[f])
            gs = None if g_state is None else g_state.contiguous()
            gser = None if (g_series is None or not spec.state_series) else g_series.contiguous()
            io.gstate_out, io.gstate_series = _ptr(gs), _ptr(gser)
            io.gdyn, io.gsta = _ptr(gdyn_run), _ptr(gsta)
            io.gdyn_zero_fill = zero_fill
            io.gdyn_rows_before = rows_before
            gstate_in = torch.empty_like(state_in) if state_in.requires_grad else None
            io.gstate_in = _ptr(gstate_in)
            # f3: gradient w.r.t. the forcings (a by-product of the adjoint sweep) and w.r.t. muwts
            gforcing = torch.zeros_like(forcing) if ctx.needs_input_grad[1] else None
            gmu = torch.empty_like(mu) if (mu is not None and ctx.needs_input_grad[7]) else None
            io.gforcing, io.gmuwts = _ptr(gforcing), _ptr(gmu)
            with _timed('hbv_bwd', dev):
                A.check(lib.hbv_b200_bwd(C.byref(d), C.byref(io), stream), 'bwd')
        if gmu is not None:
            if g_flux[A.F_QSIM] is None:
                gmu.zero_()
            gmu = gmu.view((-1, B, nmul) if mu_ts else (1, B, nmul)).sum_to_size(ctx.muwts_shape)
        if not (ctx.needs_input_grad[2] or ctx.needs_input_grad[3]):
            gdyn_full = gsta = None
        if (REUSE_GRAD_PLANE and gdyn_full is not None and zero_fill == 1 and drop is None
                and not getattr(gdyn_full, '_hbv_clean_plane', False)):
            # this call has initialised every element of the plane (the adjoint's fused zero fill +
            # the warm-up rows / routing columns cleared above): keep it, so that the next step with
            # the same run plan can skip all of that (ops._clean_plane; the views must go first —
            # the cache remembers how many references the idle plane has)
            gdyn_run = g_route = None
            gdyn_full = _register_plane(spec, dyn, t_off, gdyn_full)
        return (None, gforcing, gdyn_full, gsta, gstate_in, None, None, gmu, None, None, None)


def hbv_run(spec: RunSpec, forcing, dyn, sta, state_in, drop=None, attrs=None, muwts=None,
            t_off: int = 0, gplane=None):
    """Run the recurrence (+ routing) on rows [t_off:] of `dyn`.

    forcing  [T, B, nvar]  (already sliced to the run)
    dyn      [T_total, B, dyn_ncol] full packed/dynamic tensor or None
    sta      [B, sta_ncol] or None
    state_in [5, B, nmul]
    Returns dict(flux=[nflux x [T,B]], routed=[n_routed x [T,B]] or None, bfi, state_out, series).
    """
    _check_cuda(forcing, 'x_phy')
    forcing = forcing.contiguous()
    if dyn is not None:
        _check_cuda(dyn, 'parameters')
        dyn = dyn.contiguous()
    if sta is not None:
        _check_cuda(sta, 'static parameters')
        sta = sta.contiguous()
    outs = _HbvRun.apply(spec, forcing, dyn, sta, state_in.contiguous(), drop, attrs, muwts, t_off, gplane,
                         torch.is_grad_enabled())
    nf = spec.nflux
    n_r = spec.n_routed if spec.routing else 0
    return {
        'flux': list(outs[:nf]),
        'routed': list(outs[nf:nf + n_r]) if n_r else None,
        'bfi': outs[nf + n_r] if (spec.routing and spec.bfi) else None,
        'state_out': outs[nf + n_r + 1],
        'series': outs[nf + n_r + 2] if spec.state_series else None,
    }


def route_with_history(spec: RunSpec, route_t: torch.Tensor, route_stride: int, q_run: torch.Tensor,
                       hist: Optional[torch.Tensor]):
    """Streaming inference (SURVEY f2): gamma-UH routing (K4) of the run's un-routed series
    `q_run` [n_routed, T, B] preceded by `hist` [n_routed, H, B], the last H <= lenF - 1 steps of
    the previous calls — so a series routed chunk by chunk equals the one-shot routing.  No
    gradient (raises under autograd).  Returns (routed [n_routed, T, B], new history)."""
    if torch.is_grad_enabled() and (q_run.requires_grad or route_t.requires_grad):
        raise RuntimeError('hydrodl2_b200: the UH history carry-over is an inference feature (use torch.no_grad())')
    lib = A.load()
    dev = q_run.device
    n_r, T, B = q_run.shape
    keep = max(spec.lenF - 1, 0)
    if hist is None:
        # "before the start" is zero flow: the window is always at least lenF long, so the unit
        # hydrograph is built over all lenF taps as in a one-shot run of >= lenF steps (the
        # reference normalises over min(lenF, T) taps, uh_routing.py:5-22)
        hist = q_run.new_zeros((n_r, keep, B))
    H = hist.shape[1]
    q_cat = q_run.contiguous() if H == 0 else torch.cat([hist, q_run], dim=1).contiguous()
    Tc = H + T
    rdesc = make_route_desc(spec, Tc, B, route_stride)
    rdesc.nser = n_r
    routed = torch.empty((n_r, Tc, B), device=dev, dtype=torch.float32)
    uh = torch.empty((min(spec.lenF, Tc), B), device=dev, dtype=torch.float32)
    with torch.cuda.device(dev):
        with _timed('route_fwd', dev):
            A.check(lib.hbv_b200_route_fwd(C.byref(rdesc), route_t.data_ptr(), q_cat.data_ptr(), Tc * B,
                                           routed.data_ptr(), Tc * B, uh.data_ptr(), None, None, _stream(dev)),
                    'route_fwd')
    return routed[:, H:], (q_cat[:, -keep:].clone() if keep > 0 else None)


# ----------------------------------------------------------------------------------------------
# K3: implicit HBV (`HbvAdj`, models/hbv/hbv_adj.py)
# ----------------------------------------------------------------------------------------------
class _HbvAdjRun(torch.autograd.Function):
    """Differentiable warm-up + run + routing of the implicit scheme (hbv_adj.py:227-330).

    forward : K3 (warm-up rows, all static) -> K3 (run rows) -> K4 (gamma UH, one series)
    backward: K4^T -> K3 adjoint (run) -> K3 adjoint (warm-up); one dense gradient tensor for
              `parameters`, written in place by the kernels, and — when `x_phy` requires grad —
              the forcing gradient of every row, warm-up rows included.  When only `x_phy` needs
              a gradient, no parameter-gradient plane is allocated at all."""

    @staticmethod
    def forward(ctx, spec_w: RunSpec, spec: RunSpec, forcing, dyn, state_in, drop, warm_up, newton, track=True):
        lib = A.load()
        dev = forcing.device
        Tt, B, nvar = forcing.shape
        nmul, ncol = spec.nmul, dyn.shape[-1]
        T = Tt - warm_up
        tol, maxu = newton
        need_grad = track and (dyn.requires_grad or state_in.requires_grad or forcing.requires_grad)
        stream = _stream(dev)
        stats = torch.zeros(2, dtype=torch.int32, device=dev)

        def desc_of(sp, nT):
            d = make_desc(sp, nT, B, nvar, ncol, 0)
            d.ckpt_interval = 0
            d.adj_tol, d.adj_max_updates = float(tol), int(maxu)
            return d

        ysol_w = state_w = None
        cur = state_in
        with torch.cuda.device(dev):
            if warm_up > 0:
                ysol_w = torch.empty((warm_up, 5, B, nmul), device=dev, dtype=torch.float32) if need_grad else None
                state_w = torch.empty_like(state_in)
                io = A.HbvAdjFwdIO()
                io.forcing, io.dyn, io.drop = _ptr(forcing), _ptr(dyn), None
                io.state_in, io.state_out, io.qsim = _ptr(cur), _ptr(state_w), None
                io.ysol, io.stats = _ptr(ysol_w), _ptr(stats)
                with _timed('hbv_adj_fwd_warmup', dev):
                    A.check(lib.hbv_b200_adj_fwd(C.byref(desc_of(spec_w, warm_up)), C.byref(io), stream), 'adj_fwd(warm-up)')
                cur = state_w
            ysol = torch.empty((T, 5, B, nmul), device=dev, dtype=torch.float32) if need_grad else None
            qsim = torch.empty((T, B), device=dev, dtype=torch.float32)
            state_out = torch.empty_like(state_in)
            io = A.HbvAdjFwdIO()
            io.forcing, io.dyn, io.drop = _ptr(forcing[warm_up:]), _ptr(dyn[warm_up:]), _ptr(drop)
            io.state_in, io.state_out, io.qsim = _ptr(cur), _ptr(state_out), _ptr(qsim)
            io.ysol, io.stats = _ptr(ysol), _ptr(stats)
            with _timed('hbv_adj_fwd', dev):
                A.check(lib.hbv_b200_adj_fwd(C.byref(desc_of(spec, T)), C.byref(io), stream), 'adj_fwd')

            routed = uh = None
            if spec.routing:
                route_t = dyn[Tt - 1, :, spec.route_col:]
                rdesc = make_route_desc(spec, T, B, ncol)
                routed = torch.empty((1, T, B), device=dev, dtype=torch.float32)
                uh = torch.empty((min(spec.lenF, T), B), device=dev, dtype=torch.float32)
                with _timed('route_fwd', dev):
                    A.check(lib.hbv_b200_route_fwd(C.byref(rdesc), route_t.data_ptr(), qsim.data_ptr(), T * B,
                                                   routed.data_ptr(), T * B, uh.data_ptr(), None, None,
                                                   stream), 'route_fwd')
        ctx.specs, ctx.dims, ctx.newton = (spec_w, spec), (Tt, T, B, nvar, ncol, warm_up), newton
        ctx.save_for_backward(forcing, dyn, drop, state_in, ysol_w, ysol, qsim, uh)
        ctx.set_materialize_grads(False)
        return qsim, (routed[0] if routed is not None else qsim.new_zeros(())), state_out, stats

    @staticmethod
    def jvp(ctx, *_tangents):
        raise NotImplementedError('hydrodl2_b200: forward-mode AD is not supported for HbvAdj (the implicit '
                                  'scheme); use reverse mode')

    @staticmethod
    def backward(ctx, g_q, g_rout, g_state, _g_stats):
        lib = A.load()
        spec_w, spec = ctx.specs
        forcing, dyn, drop, state_in, ysol_w, ysol, qsim, uh = ctx.saved_tensors
        Tt, T, B, nvar, ncol, warm_up = ctx.dims
        tol, maxu = ctx.newton
        dev = forcing.device
        stream = _stream(dev)
        if ysol is None:
            raise RuntimeError('hydrodl2_b200: backward called but no input required grad')
        # The dense gradient plane: K3's adjoint zeroes the rows it owns itself (gdyn_zero_fill)
        # instead of a 6 GB memset in front of it (BASELINE config 5); what it does not own — the
        # routing columns of the last row of each call's slice — is cleared here.  When only the
        # forcings need a gradient (data assimilation with fixed parameters) there is no plane:
        # the adjoint gets gdyn = NULL and makes no parameter-gradient stores.
        need_forcing = ctx.needs_input_grad[2]
        plane = ctx.needs_input_grad[3] or not need_forcing
        nmul = spec.nmul
        fused = plane and nmul == 16 and ncol % 2 == 0
        n_phy = spec.n_par * nmul
        kept = None
        if fused and REUSE_GRAD_PLANE and drop is None:
            kept = _lookup_plane(spec, dyn, warm_up)      # a clean plane kept from an earlier step (see _clean_plane)
        if kept is not None:
            gdyn, fused = kept, False                     # the adjoint writes its gradient entries only
            if not (spec.routing and g_rout is not None) and n_phy < ncol:
                gdyn[Tt - 1, :, n_phy:].zero_()           # nobody writes the routing columns this time (retires the plane)
        elif fused:
            gdyn = torch.empty_like(dyn)
            gdyn[Tt - 1, :, n_phy:].zero_()
            if warm_up > 0:
                gdyn[warm_up - 1, :, n_phy:].zero_()
        elif plane:
            gdyn = torch.zeros_like(dyn)
        else:
            gdyn = None
        gforcing = torch.zeros_like(forcing) if need_forcing else None

        def desc_of(sp, nT):
            d = make_desc(sp, nT, B, nvar, ncol, 0)
            d.ckpt_interval = 0
            d.adj_tol, d.adj_max_updates = float(tol), int(maxu)
            return d

        with torch.cuda.device(dev):
            gq = None if g_q is None else g_q.contiguous()
            if spec.routing and g_rout is not None:
                if gdyn is not None:
                    route_t = dyn[Tt - 1, :, spec.route_col:]
                    g_route = gdyn[Tt - 1, :, spec.route_col:]
                    rdesc = make_route_desc(spec, T, B, ncol)
                else:       # (the routing-parameter gradient K4^T must write goes to a scratch)
                    route_t = dyn[Tt - 1, :, spec.route_col:spec.route_col + 2].contiguous()
                    g_route = torch.empty((B, 2), device=dev, dtype=torch.float32)
                    rdesc = make_route_desc(spec, T, B, 2)
                nch = lib.hbv_b200_route_chunks(T, B)
                ws = torch.empty((min(spec.lenF, T), nch, B), device=dev, dtype=torch.float32)
                g_in = torch.empty((1, T, B), device=dev, dtype=torch.float32)
                g_out = g_rout.contiguous().view(1, T, B)
                with _timed('route_bwd', dev):
                    A.check(lib.hbv_b200_route_bwd(
                        C.byref(rdesc), route_t.data_ptr(), qsim.data_ptr(), T * B, None, T * B,
                        uh.data_ptr(), None, g_out.data_ptr(), T * B, 1, None,
                        g_in.data_ptr(), T * B, g_route.data_ptr(), ws.data_ptr(), stream), 'route_bwd')
                gq = g_in[0] if gq is None else gq + g_in[0]
            need_gin = warm_up > 0 or state_in.requires_grad
            gmid = torch.empty_like(state_in) if need_gin else None
            io = A.HbvAdjBwdIO()
            io.forcing, io.dyn, io.drop = _ptr(forcing[warm_up:]), _ptr(dyn[warm_up:]), _ptr(drop)
            io.ysol, io.gqsim = _ptr(ysol), _ptr(gq)
            io.gstate_out = None if g_state is None else _ptr(g_state.contiguous())
            io.gdyn, io.gstate_in = _ptr(gdyn[warm_up:] if plane else None), _ptr(gmid)
            io.gdyn_zero_fill = int(fused)
            io.gforcing = _ptr(gforcing[warm_up:] if need_forcing else None)
            with _timed('hbv_adj_bwd', dev):
                A.check(lib.hbv_b200_adj_bwd(C.byref(desc_of(spec, T)), C.byref(io), stream), 'adj_bwd')
            gstate_in = gmid
            if warm_up > 0:
                gstate_in = torch.empty_like(state_in) if state_in.requires_grad else None
                io = A.HbvAdjBwdIO()
                io.forcing, io.dyn, io.drop = _ptr(forcing), _ptr(dyn), None
                io.ysol, io.gqsim, io.gstate_out = _ptr(ysol_w), None, _ptr(gmid)
                io.gdyn, io.gstate_in = _ptr(gdyn), _ptr(gstate_in)
                io.gdyn_zero_fill = int(fused)
                io.gforcing = _ptr(gforcing)
                with _timed('hbv_adj_bwd_warmup', dev):
                    A.check(lib.hbv_b200_adj_bwd(C.byref(desc_of(spec_w, warm_up)), C.byref(io), stream), 'adj_bwd(warm-up)')
        if fused and kept is None and REUSE_GRAD_PLANE and drop is None:
            g_route = route_t = io = None                 # (views of the plane: the cache counts references)
            gdyn = _register_plane(spec, dyn, warm_up, gdyn)
        return (None, None, gforcing, gdyn, gstate_in if state_in.requires_grad else None, None, None, None, None)


def hbv_adj_run(spec_w: RunSpec, spec: RunSpec, forcing, dyn, state_in, drop=None, warm_up: int = 0,
                tol: float = 1e-3, max_updates: int = 8):
    """Implicit-scheme run.  forcing [T_total, B, nvar], dyn [T_total, B, ncol] raw packed
    parameters, state_in [5, B, nmul].  Rows [:warm_up] are the (differentiable) warm-up with
    static parameters taken from row warm_up-1 (hbv_adj.py:257-274).  `forcing`, `dyn` and
    `state_in` may each require grad; the forcing gradient covers the warm-up rows too.
    Returns dict(qsim [T,B], routed [T,B] or None, state_out, stats int32[2])."""
    _check_cuda(forcing, 'x_phy')
    _check_cuda(dyn, 'parameters')
    qsim, routed, state_out, stats = _HbvAdjRun.apply(
        spec_w, spec, forcing.contiguous(), dyn.contiguous(), state_in.contiguous(), drop,
        int(warm_up), (tol, max_updates), torch.is_grad_enabled())
    return {'qsim': qsim, 'routed': routed if spec.routing else None, 'state_out': state_out,
            'stats': stats}
