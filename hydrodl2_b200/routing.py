"""Distributed (gage, unit) pair routing — host side of K4' (csrc/pair_route.cu).

Drop-in for ``Hbv_2_hourly.distr_routing`` (hbv_2_hourly.py:800-855): same arguments and result
``[T, n_gages, 1]``.  The pair list is the row-major non-zero set of ``outlet_topo`` exactly as
``(outlet_topo == 1).nonzero()`` produces it; it and its CSR/CSC index arrays depend on the
topology only and are cached per topology tensor, so the reference's per-call ``nonzero``
device-to-host sync (hbv_2_hourly.py:822-824) happens once.
"""

from __future__ import annotations

import collections
import ctypes as C

import torch

from . import _cabi as A
from .ops import _check_cuda, _stream, _timed

_TOPO_CACHE: "collections.OrderedDict" = collections.OrderedDict()
_TOPO_CACHE_MAX = 16


class PairIndex:
    """Index arrays of one outlet topology (all int32, on `device`)."""

    def __init__(self, outlet_topo: torch.Tensor, areas: torch.Tensor, device=None):
        dev = torch.device(device) if device is not None else outlet_topo.device
        topo = outlet_topo.to(dev)
        idx = (topo == 1).nonzero(as_tuple=False)
        rows, cols = idx[:, 0].contiguous(), idx[:, 1].contiguous()
        self.n_gages, self.n_units = int(topo.shape[0]), int(topo.shape[1])
        self.n_pairs = int(rows.numel())
        self.pair_row = rows.to(torch.int32)
        self.pair_col = cols.to(torch.int32)
        z = torch.zeros(1, dtype=torch.int64, device=dev)
        self.gage_off = torch.cat([z, torch.bincount(rows, minlength=self.n_gages).cumsum(0)]).to(torch.int32)
        self.unit_off = torch.cat([z, torch.bincount(cols, minlength=self.n_units).cumsum(0)]).to(torch.int32)
        self.unit_perm = torch.argsort(cols, stable=True).to(torch.int32)
        a = areas.to(device=dev, dtype=torch.float32)
        denom = (topo.to(torch.float32) * a[None, :]).sum(dim=1).clamp(min=1e-6)  # :849
        self.inv_denom = (1.0 / denom).contiguous()
        self.areas = a.contiguous()

    @classmethod
    def identity(cls, n_units: int, device) -> "PairIndex":
        """One gage per unit, unit area 1: pair routing degenerates to per-unit UH routing
        (hbv_2_hourly.py:684-705 with lenF = 72) without a dense [n, n] topology."""
        self = cls.__new__(cls)
        dev = torch.device(device)
        ar = torch.arange(n_units + 1, dtype=torch.int32, device=dev)
        self.n_gages = self.n_units = self.n_pairs = int(n_units)
        self.pair_row = self.pair_col = self.unit_perm = ar[:n_units].contiguous()
        self.gage_off = self.unit_off = ar
        self.inv_denom = torch.ones(n_units, dtype=torch.float32, device=dev)
        self.areas = torch.ones(n_units, dtype=torch.float32, device=dev)
        return self


def pair_index(outlet_topo: torch.Tensor, areas: torch.Tensor, device=None) -> PairIndex:
    """Cached `PairIndex` of (outlet_topo, areas), built on `device` (default: the topology's).

    The key is the identity of the two tensors the CALLER holds (storage address, shape, version
    counter, device) and the entry keeps strong references to them: while an entry is cached its
    tensors cannot be freed, so the caching allocator cannot hand their addresses to a different
    topology of the same shape (which round 1's address-only key would have mistaken for a hit).
    An in-place edit bumps the version counter and misses.  Least-recently-used eviction."""
    dev = torch.device(device) if device is not None else outlet_topo.device
    key = (outlet_topo.data_ptr(), tuple(outlet_topo.shape), tuple(outlet_topo.stride()), outlet_topo._version,
           str(outlet_topo.device), areas.data_ptr(), tuple(areas.shape), areas._version, str(areas.device),
           str(dev))
    hit = _TOPO_CACHE.get(key)
    if hit is not None:
        _TOPO_CACHE.move_to_end(key)
        return hit[0]
    pi = PairIndex(outlet_topo, areas, dev)
    _TOPO_CACHE[key] = (pi, outlet_topo, areas)      # the references keep the addresses taken
    while len(_TOPO_CACHE) > _TOPO_CACHE_MAX:
        _TOPO_CACHE.popitem(last=False)
    return pi


def _desc(pi: PairIndex, T: int, lenF: int, lag_uh: bool, bounds) -> A.HbvPairDesc:
    d = A.HbvPairDesc()
    d.abi_version = A.ABI_VERSION
    d.T, d.n_pairs, d.n_units, d.n_gages, d.lenF = T, pi.n_pairs, pi.n_units, pi.n_gages, lenF
    d.lag_uh = int(lag_uh)
    (d.a_lo, d.a_hi), (d.b_lo, d.b_hi) = bounds[0], bounds[1]
    d.tau_lo, d.tau_hi = bounds[2] if len(bounds) > 2 else (0.0, 0.0)
    return d


class _PairRoute(torch.autograd.Function):
    @staticmethod
    def forward(ctx, qs, par, pi: PairIndex, lenF, lag_uh, bounds):
        lib = A.load()
        dev = qs.device
        T = qs.shape[0]
        d = _desc(pi, T, lenF, lag_uh, bounds)
        M = min(T, lenF)
        uh = torch.empty((M, pi.n_pairs), device=dev, dtype=torch.float32)
        lag = torch.empty((T, pi.n_pairs), device=dev, dtype=torch.float32)
        out = torch.empty((T, pi.n_gages), device=dev, dtype=torch.float32)
        with torch.cuda.device(dev), _timed('pair_route_fwd', dev):
            A.check(lib.hbv_b200_pair_route_fwd(
                C.byref(d), par.data_ptr(), qs.data_ptr(), pi.areas.data_ptr(), pi.pair_col.data_ptr(),
                pi.gage_off.data_ptr(), pi.inv_denom.data_ptr(), uh.data_ptr(), lag.data_ptr(),
                out.data_ptr(), _stream(dev)), 'pair_route_fwd')
        ctx.pi, ctx.args = pi, (lenF, lag_uh, bounds)
        ctx.save_for_backward(qs, par, uh)
        return out

    @staticmethod
    def jvp(ctx, *_tangents):
        raise NotImplementedError('hydrodl2_b200: forward-mode AD is not supported through the distributed '
                                  'pair routing or the per-unit UH routing with more than 16 taps (K4\')')

    @staticmethod
    def backward(ctx, g_out):
        lib = A.load()
        qs, par, uh = ctx.saved_tensors
        pi: PairIndex = ctx.pi
        lenF, lag_uh, bounds = ctx.args
        dev = qs.device
        T = qs.shape[0]
        d = _desc(pi, T, lenF, lag_uh, bounds)
        g_out = g_out.contiguous()
        nch = lib.hbv_b200_pair_chunks(T)
        g_lag = torch.empty((T, pi.n_pairs), device=dev, dtype=torch.float32)
        duh = torch.empty((uh.shape[0], nch, pi.n_pairs), device=dev, dtype=torch.float32)
        g_qs = torch.empty_like(qs)
        g_par = torch.empty_like(par)
        with torch.cuda.device(dev), _timed('pair_route_bwd', dev):
            A.check(lib.hbv_b200_pair_route_bwd(
                C.byref(d), par.data_ptr(), qs.data_ptr(), pi.areas.data_ptr(), pi.pair_col.data_ptr(),
                pi.pair_row.data_ptr(), pi.inv_denom.data_ptr(), pi.unit_off.data_ptr(),
                pi.unit_perm.data_ptr(), uh.data_ptr(), g_out.data_ptr(), g_lag.data_ptr(),
                duh.data_ptr(), g_qs.data_ptr(), g_par.data_ptr(), _stream(dev)), 'pair_route_bwd')
        return g_qs, g_par, None, None, None, None


def distr_routing(Qs, distr_params, outlet_topo, areas, lenF=72, lag_uh=True,
                  bounds=((0, 5.0), (0, 12.0), (0, 48.0))):
    """Qs [T, n_units, 1], distr_params [n_pairs, 3] in [0, 1] -> gage flow [T, n_gages, 1]."""
    _check_cuda(Qs, 'Qs')
    pi = outlet_topo if isinstance(outlet_topo, PairIndex) else pair_index(outlet_topo, areas, Qs.device)
    if distr_params.shape[0] != pi.n_pairs:
        raise ValueError(f'distr parameters have {distr_params.shape[0]} rows, topology has '
                         f'{pi.n_pairs} (gage, unit) pairs')
    qs = Qs.reshape(Qs.shape[0], -1).contiguous()
    par = distr_params.to(device=Qs.device, dtype=torch.float32).contiguous()
    if par.shape[1] < 3:
        par = torch.cat([par, par.new_zeros(par.shape[0], 3 - par.shape[1])], dim=1)
    out = _PairRoute.apply(qs, par, pi, lenF, lag_uh, tuple(tuple(b) for b in bounds))
    return out.unsqueeze(-1)


_IDENTITY_CACHE: dict = {}
_MAX_UNITS_PER_CALL = 32768      # seg_sum puts one gage per grid.y block


def unit_routing(q: torch.Tensor, route_ab: torch.Tensor, lenF: int, bounds) -> torch.Tensor:
    """Per-unit gamma-UH routing with up to 128 taps: q [T, B], route_ab [B, 2] in [0, 1]
    (route_a, route_b), bounds ((a_lo, a_hi), (b_lo, b_hi)) -> routed [T, B].

    Drop-in for the `routing=True` branch of the hourly model (hbv_2_hourly.py:684-705:
    `uh_gamma` with lenF = 72 + `uh_conv` on the nmul-mean runoff); the 16-tap register-window
    kernel of uh_route.cu cannot hold 72 taps, so this goes through the shared-memory-staged
    pair kernels (csrc/pair_route.cu) with an identity (gage = unit) index, no lag."""
    _check_cuda(q, 'Qs')
    T, B = q.shape
    dev = q.device
    par = torch.cat([route_ab.to(device=dev, dtype=torch.float32),
                     torch.zeros(B, 1, device=dev, dtype=torch.float32)], dim=1)
    b3 = (tuple(bounds[0]), tuple(bounds[1]), (0.0, 0.0))
    outs = []
    for b0 in range(0, B, _MAX_UNITS_PER_CALL):
        nb = min(_MAX_UNITS_PER_CALL, B - b0)
        key = (nb, str(dev))
        pi = _IDENTITY_CACHE.get(key)
        if pi is None:
            pi = _IDENTITY_CACHE[key] = PairIndex.identity(nb, dev)
        qs = q[:, b0:b0 + nb].contiguous()
        outs.append(_PairRoute.apply(qs, par[b0:b0 + nb].contiguous(), pi, lenF, False, b3))
    return outs[0] if len(outs) == 1 else torch.cat(outs, dim=1)
