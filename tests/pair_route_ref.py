"""Float64 reference and fp32 error bound for the pair-routing kernels (K4', csrc/pair_route.cu).

Shared by tests/test_pair_route_cpu.py, which pins this reference to the oracle, and
tests/test_pair_route_gpu.py, which holds the kernels to it.

The reference is put together from the oracle's own pieces (oracle/hbv_oracle.py): `uh_gamma`,
`frac_shift1d`, the shift-and-add `uh_conv_direct` (not the grouped `conv1d` of `uh_conv`; the two
are pinned to each other on the CPU), `scatter_add` over the gages and the `denom` clamp of
`distr_routing`.  It runs on whatever device its inputs are on, and autograd gives its gradients.

The kernels descale the parameters in float32 (`lo + p * (hi - lo)`, csrc/pair_route.cu) and
evaluate everything after that in float32.  `descale` gives the reference the same float32
physical values, so what is compared is the kernels' arithmetic and not the rounding of their
input.
"""

import numpy as np
import torch

from oracle import hbv_oracle as O

U32 = 2.0 ** -24        # unit roundoff of float32
DEFAULT_BOUNDS = ((0.0, 5.0), (0.0, 12.0), (0.0, 48.0))
UNIT_BOUNDS = ((0.0, 1.0), (0.0, 1.0), (0.0, 1.0))


def seg_sum_branch(n_pairs, n_segments):
    """Which `seg_sum` kernel of csrc/pair_route.cu runs: 'wide' (one warp per segment) when
    n_pairs >= 8 * n_segments, else 'rows'.  The forward sums over gages, the adjoint over units."""
    return 'wide' if n_pairs >= 8 * n_segments else 'rows'


def topo_pairs(topo):
    """(gage, unit) pairs of `topo` in the kernels' order: the row-major entries equal to 1."""
    idx = (topo == 1).nonzero(as_tuple=False)
    return idx[:, 0].contiguous(), idx[:, 1].contiguous()


def topo_denom(topo, areas, dtype=torch.float64):
    """Upstream area of every gage with the clamp of `distr_routing`: entries other than 1 (a
    0.5, say) count here although they are no pair."""
    return (topo.to(dtype) * areas.to(dtype)[None, :]).sum(dim=1).clamp(min=1e-6)


def descale(par, bounds, lag_uh=True):
    """Physical (route_a, route_b, route_tau) from `par` [P, 3] in the normalised convention.

    The value is what the kernel computes, fmaf(p, hi - lo, lo) in float32 with the bounds
    rounded to float32 (bit for bit when lo = 0, as in every bound used here); the gradient
    flows back to `par` with the factor hi - lo.  The result has `par`'s dtype."""
    out = []
    for i in range(3 if lag_uh else 2):
        lo32, hi32 = np.float32(bounds[i][0]), np.float32(bounds[i][1])
        span = float(np.float32(hi32 - lo32))
        v = par[:, i].double() * span + float(lo32)
        v = v + (v.float().double() - v).detach()
        out.append(v.to(par.dtype))
    return out


def route_ref(qs, par, rows, cols, n_gages, areas, denom, lenF, lag_uh=True, bounds=DEFAULT_BOUNDS,
              keep_uh=False):
    """Gage flow [T, n_gages] of the pair routing in `qs`'s dtype.

    qs [T, n_units]; par [n_pairs, 3] normalised with `bounds`; rows / cols the pair list;
    areas [n_units]; denom [n_gages].  With `keep_uh`, also returns the (shifted) unit hydrograph
    [M, n_pairs, 1], M = min(T, lenF), as a node of the graph."""
    T = qs.shape[0]
    M = min(T, lenF)
    ab = descale(par, bounds, lag_uh)
    a = ab[0].view(1, -1, 1).expand(M, -1, 1)
    b = ab[1].view(1, -1, 1).expand(M, -1, 1)
    uh = O.uh_gamma(a, b, lenF=M)
    if lag_uh:
        uh = O.frac_shift1d(uh, ab[2])
    x = (qs * areas.to(qs.dtype)[None, :])[:, cols].T.contiguous().unsqueeze(1)     # [P, 1, T]
    lag = O.uh_conv_direct(x, uh.permute(1, 2, 0).contiguous()).squeeze(1)         # [P, T]
    out = torch.zeros(n_gages, T, dtype=qs.dtype, device=qs.device)
    out = out.scatter_add(0, rows.view(-1, 1).expand(-1, T), lag)
    out = (out / denom.to(qs.dtype)[:, None]).T
    return (out, uh) if keep_uh else out


def sum_bound(s_abs, M, n_terms):
    """Elementwise bound on the error of an fp32 evaluation of a sum of M taps over n_terms
    pairs:  4 (M + n_terms) 2^-24 S_abs + 1e-30, with S_abs the same sum in float64 of the
    terms' absolute values.  Any summation order in float32 stays inside it (n products summed
    in float32 are within n 2^-24 of the sum of their magnitudes); a lost tap, step or pair is
    a whole term and misses it by orders of magnitude.  `n_terms` broadcasts against s_abs (one
    count per gage or per unit, along the last dimension)."""
    n = torch.as_tensor(n_terms, dtype=torch.float64, device=s_abs.device)
    return 4.0 * (M + n) * U32 * s_abs.double() + 1e-30


def bound_ratio(new, ref64, s_abs, M, n_terms):
    """(worst |new - ref64| / bound, index of that element)."""
    r = (new.double() - ref64.double()).abs() / sum_bound(s_abs, M, n_terms)
    r = torch.where(torch.isfinite(new), r, torch.full_like(r, float('inf')))
    i = int(r.argmax())
    return float(r.flatten()[i]), tuple(int(v) for v in np.unravel_index(i, tuple(r.shape)))


def check_bound(new, ref64, s_abs, M, n_terms, what):
    """Asserts the elementwise fp32 summation bound; returns the worst error over bound."""
    assert new.shape == ref64.shape, f'{what}: shape {tuple(new.shape)} vs {tuple(ref64.shape)}'
    worst, at = bound_ratio(new, ref64, s_abs, M, n_terms)
    assert worst <= 1.0, (f'{what}: error {worst:.3g} x the fp32 summation bound at {at} '
                          f'(new {float(new[at]):.9g}, fp64 {float(ref64[at]):.9g})')
    return worst


# --------------------------------------------------------------------------------------------
# Topologies
# --------------------------------------------------------------------------------------------
def config4_topology(n_units=2500, per_gage=40):
    """BASELINE config 4: consecutive blocks of `per_gage` units per gage (the last gage gets
    what is left: 20 units of 2,500)."""
    n_gages = (n_units + per_gage - 1) // per_gage
    topo = torch.zeros(n_gages, n_units)
    for g in range(n_gages):
        topo[g, g * per_gage:(g + 1) * per_gage] = 1.0
    return topo


def nested_topology(seed=0, per_step=7, n_chain=40, n_side=19):
    """A network of nested gauges, columns shuffled:
      * gages 0 .. n_chain-1 form one chain of nested basins: gage g drains the first
        per_step * (g + 1) chain units, so each of the first per_step units drains to all
        n_chain gages;
      * gage n_chain has no unit;
      * gage n_chain + 1 drains n_side further units, and has a 0.5 entry for the last unit,
        which drains to no gage (the 0.5 is no pair but counts in that gage's upstream area).
    """
    n_ch = per_step * n_chain
    n_units = n_ch + n_side + 1
    topo = torch.zeros(n_chain + 2, n_units)
    for g in range(n_chain):
        topo[g, :per_step * (g + 1)] = 1.0
    topo[n_chain + 1, n_ch:n_ch + n_side] = 1.0
    topo[n_chain + 1, n_units - 1] = 0.5
    perm = torch.randperm(n_units, generator=torch.Generator().manual_seed(seed))
    return topo[:, perm].contiguous()


def small_topology():
    """12 units, 4 gages, two of them nested in the others (24 pairs)."""
    topo = torch.zeros(4, 12)
    topo[0, 0:4] = 1.0
    topo[1, 0:8] = 1.0
    topo[2, 8:12] = 1.0
    topo[3, 4:12] = 1.0
    return topo


def many_gage_topology(n_units=6, n_gages=40):
    """Few units shared by many gages: gage g drains every unit u with (u + g) % n_units != 0
    (n_units - 1 units per gage, each unit on most gages)."""
    topo = torch.zeros(n_gages, n_units)
    for g in range(n_gages):
        for u in range(n_units):
            if (u + g) % n_units:
                topo[g, u] = 1.0
    return topo
