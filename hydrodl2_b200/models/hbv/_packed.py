"""Host-side logic shared by the packed-parameter models (HBV 1.0 and 1.1p).

Mirrors the reference's module interface for this path —
``Hbv.__init__/forward/get_states/load_states/_PBM`` in
``models/hbv/hbv.py:37-596`` and ``hbv_1_1p.py`` — same attribute names,
argument meaning and error behaviour, so δMG can use the class unchanged.
What differs is *where the arithmetic happens*: unpack / sigmoid / descale
(hbv.py:182-256), the time loop (hbv.py:423-505), the nmul mean
(hbv.py:508-511,575-588), UH routing (hbv.py:523-538) and BFI
(hbv.py:562-567) run inside ``libhbv_b200.so`` through
``hydrodl2_b200.ops.hbv_run``; this file only resolves configuration, draws the
dynamic-parameter dropout masks with the same CPU RNG stream as the reference
(hbv.py:240-246) and assembles the flux dictionary.
"""

from __future__ import annotations

from typing import Any, Optional, Union

import torch

from ... import _cabi as A
from ...ops import (RunSpec, hbv_run, hbv_states_only, hbv_states_only_dual, is_dual, refuse_forward_ad,
                   route_with_history, start_grad_plane)
from ._seam import PackedSeam

_FLUX_KEYS = (
    # (dict key, source) — source: ('r', i) routed plane i, ('f', slot) flux slot, 'pet'
    ('streamflow', ('r', 0)), ('srflow', ('r', 1)), ('ssflow', ('r', 2)), ('gwflow', ('r', 3)),
    ('AET_hydro', ('f', A.F_AET)), ('PET_hydro', 'pet'), ('SWE', ('f', A.F_SWE)),
    ('streamflow_no_rout', ('f', A.F_QSIM)), ('srflow_no_rout', ('f', A.F_Q0)),
    ('ssflow_no_rout', ('f', A.F_Q1)), ('gwflow_no_rout', ('f', A.F_Q2)),
    ('recharge', ('f', A.F_RECHARGE)), ('excs', ('f', A.F_EXCS)),
    ('evapfactor', ('f', A.F_EVAPFACTOR)), ('tosoil', ('f', A.F_TOSOIL)),
    ('percolation', ('f', A.F_PERC)), ('capillary', ('f', A.F_CAPILLARY)),
)


class PackedHbv(PackedSeam, torch.nn.Module):
    """Base of `Hbv` and `Hbv_1_1p` (packed raw parameter tensor + sigmoid)."""

    _variant = A.VARIANT_HBV
    _name = 'HBV'
    _capillary = False
    _always_betaet = False
    _extra_bounds: dict = {}

    def __init__(
        self,
        config: Optional[dict[str, Any]] = None,
        device: Optional[torch.device] = None,
    ) -> None:
        super().__init__()
        self.name = self._name
        self.config = config
        self.initialize = False
        self.warm_up = 0
        self.pred_cutoff = 0
        self.warm_up_states = True
        self.dynamic_params = []
        self.dy_drop = 0.0
        self.variables = ['prcp', 'tmean', 'pet']
        self.routing = True
        self.comprout = False
        self.nearzero = 1e-5
        self.nmul = 1
        self.cache_states = False
        self.device = device
        # K of the checkpointed adjoint (extension, not in reference): 0 = let the library pick
        # (every state for small problems, every 16th otherwise), or 1..64
        self.ckpt_interval = 0
        # extension (SURVEY f2, not in the reference): with `cache_states`, also carry the last
        # lenF - 1 steps of the un-routed series into the next call, so that the ROUTED flows of a
        # run stepped chunk by chunk equal the one-shot run (in the reference — and here by
        # default — the daily UH convolution restarts from an empty history at every call)
        self.uh_carry_over = False
        self._uh_hist = None

        self.states, self._states_cache = None, None

        self.state_names = ['SNOWPACK', 'MELTWATER', 'SM', 'SUZ', 'SLZ']
        self.flux_names = [k for k, _ in _FLUX_KEYS if (k != 'capillary' or self._capillary)]
        self.flux_names.append('BFI')

        self.parameter_bounds = {
            'parBETA': [1.0, 6.0], 'parFC': [50, 1000], 'parK0': [0.05, 0.9],
            'parK1': [0.01, 0.5], 'parK2': [0.001, 0.2], 'parLP': [0.2, 1],
            'parPERC': [0, 10], 'parUZL': [0, 100], 'parTT': [-2.5, 2.5],
            'parCFMAX': [0.5, 10], 'parCFR': [0, 0.1], 'parCWH': [0, 0.2],
        }
        self.parameter_bounds.update(self._extra_bounds)
        self.routing_parameter_bounds = {'route_a': [0, 2.9], 'route_b': [0, 6.5]}

        if not device:
            self.device = torch.device('cuda' if torch.cuda.is_available() else 'cpu')

        if config is not None:
            self.warm_up = config.get('warm_up', self.warm_up)
            self.warm_up_states = config.get('warm_up_states', self.warm_up_states)
            self.dy_drop = config.get('dy_drop', self.dy_drop)
            self.dynamic_params = config['dynamic_params'].get(
                self.__class__.__name__, self.dynamic_params
            )
            self.variables = config.get('variables', self.variables)
            self.routing = config.get('routing', self.routing)
            self.comprout = config.get('comprout', self.comprout)
            self.nearzero = config.get('nearzero', self.nearzero)
            self.nmul = config.get('nmul', self.nmul)
            self.cache_states = config.get('cache_states', False)
            self.ckpt_interval = config.get('ckpt_interval', self.ckpt_interval)
            self.uh_carry_over = config.get('uh_carry_over', self.uh_carry_over)
            if (not self._always_betaet) and 'parBETAET' in self.dynamic_params:
                self.parameter_bounds['parBETAET'] = [0.3, 5]   # hbv.py:124-125
        self._set_parameters()

    # ------------------------------------------------------------------ state API
    def _init_states(self, ngrid: int) -> tuple[torch.Tensor, ...]:
        """hbv.py:128-136 — every store starts at 0.001."""
        return tuple(
            torch.full((ngrid, self.nmul), 0.001, dtype=torch.float32, device=self.device)
            for _ in self.state_names
        )

    def _init_stack(self, ngrid: int) -> torch.Tensor:
        """The same initial state as one read-only [5, B, nmul] tensor, built once per shape
        (the kernels never write their state input)."""
        c = getattr(self, '_init_cache', None)
        if c is None or c.shape[1] != ngrid or c.shape[2] != self.nmul or c.device != torch.device(self.device):
            c = torch.full((5, ngrid, self.nmul), 0.001, dtype=torch.float32, device=self.device)
            self._init_cache = c
        return c

    def get_states(self) -> Optional[tuple[torch.Tensor, ...]]:
        """Final states of the last forward (SNOWPACK, MELTWATER, SM, SUZ, SLZ)."""
        return self._states_cache

    def load_states(self, states: tuple[torch.Tensor, ...]) -> None:
        """hbv.py:148-168 (same checks, same errors)."""
        for state in states:
            if not isinstance(state, torch.Tensor):
                raise ValueError("Each element in `states` must be a tensor.")
        nstates = len(self.state_names)
        if not (isinstance(states, tuple) and len(states) == nstates):
            raise ValueError(f"`states` must be a tuple of {nstates} tensors.")
        self.states = tuple(s.detach().to(self.device, dtype=torch.float32) for s in states)
        self._uh_hist = None         # a new starting point: no runoff history to route

    def _set_parameters(self) -> None:
        self.phy_param_names = self.parameter_bounds.keys()
        self.routing_param_names = self.routing_parameter_bounds.keys() if self.routing else []
        self.learnable_param_count = len(self.phy_param_names) * self.nmul + len(
            self.routing_param_names
        )

    # ------------------------------------------------------------------ run plan
    def _spec(self, dyn_names, routing: bool) -> RunSpec:
        names = list(self.parameter_bounds.keys())
        n = len(names)
        src = [A.SRC_DYN_T if nm in dyn_names else A.SRC_DYN_LAST for nm in names]
        return RunSpec(
            variant=self._variant, n_par=n, betaet='parBETAET' in self.parameter_bounds,
            apply_sigmoid=True, par_src=src, par_col=[i * self.nmul for i in range(n)],
            par_lo=[self.parameter_bounds[k][0] for k in names],
            par_hi=[self.parameter_bounds[k][1] for k in names],
            nmul=self.nmul, nflux=12 if self._capillary else 11, nearzero=self.nearzero,
            var_index=tuple(self.variables.index(v) for v in ('prcp', 'tmean', 'pet')),
            ckpt_interval=self.ckpt_interval, routing=routing, route_src='dyn_last',
            route_col=n * self.nmul,
            route_bounds=tuple(tuple(v) for v in self.routing_parameter_bounds.values()),
            lenF=15, n_routed=4, bfi=True,
        )

    def _draw_drop(self, ngrid: int) -> Optional[torch.Tensor]:
        """One CPU `torch.bernoulli` draw per dynamic parameter in bounds order
        (hbv.py:240-246) -> uint8 [n_par, B] on device, or None if nothing dropped."""
        names = list(self.parameter_bounds.keys())
        pmat = torch.ones([1, ngrid, 1]) * self.dy_drop
        mask = torch.zeros(len(names), ngrid, dtype=torch.uint8)
        anyset = False
        for i, nm in enumerate(names):
            if nm in self.dynamic_params:
                dr = torch.bernoulli(pmat).view(ngrid)
                if self.dy_drop > 0:
                    mask[i] = dr.to(torch.uint8)
                    anyset = anyset or bool(dr.any())
        return mask.to(self.device) if anyset else None

    def io_footprint(self, n_rows: int) -> dict:
        """Which entries of a `parameters` tensor [n_rows, B, ncol] this model's kernels read
        ('read') and which entries of its dense gradient can be non-zero ('grad') — for
        column-sparse host staging (hydrodl2_b200.hostio.sparse_copy).  Time-varying parameters
        are read at every run row (hbv.py:236-246); everything else only at the last row
        (static values, hbv.py:242; routing, hbv.py:212-214) and, for the no-grad warm-up, at
        its last row (hbv.py:329-332)."""
        names = list(self.parameter_bounds.keys())
        warm = self.warm_up if self.warm_up_states else 0
        blocks = [(i * self.nmul, self.nmul) for i, nm in enumerate(names) if nm in self.dynamic_params]
        rows = sorted({n_rows - 1} | ({warm - 1} if warm > 0 else set()))
        return {'read': {'rows_full': rows, 'col_blocks': blocks, 'row_range': (warm, n_rows)},
                'grad': {'rows_full': [n_rows - 1], 'col_blocks': blocks, 'row_range': (warm, n_rows)}}

    # ------------------------------------------------------------------ forward
    def forward(
        self,
        x_dict: dict[str, torch.Tensor],
        parameters: torch.Tensor,
    ) -> Union[tuple, dict[str, torch.Tensor]]:
        """Same contract as hbv.py:284-361: returns the flux dictionary."""
        x = x_dict['x_phy']
        self.muwts = x_dict.get('muwts', None)
        ngrid = x.shape[1]
        if self.comprout:
            # the reference raises here too (UH has B rows, signal B*nmul — SURVEY.md §8 a-notes)
            raise RuntimeError('comprout=True is not supported (it fails in the reference as well)')
        n_expected = self.learnable_param_count
        if parameters.shape[-1] < len(self.parameter_bounds) * self.nmul + (2 if self.routing else 0):
            raise ValueError(f'parameters last dim {parameters.shape[-1]} < {n_expected}')

        if self.warm_up_states:
            warm_up = self.warm_up
        else:
            self.pred_cutoff = self.warm_up
            warm_up = 0

        if (not self.states) or (not self.cache_states):
            current = self._init_stack(ngrid)
            self._uh_hist = None
        else:
            current = torch.stack(tuple(self.states))

        parameters = parameters.contiguous()
        x = x.contiguous()
        if self.routing:     # `routing_param_dict` (hbv.py:311-312), materialised only if someone reads it
            n_phy = len(self.parameter_bounds) * self.nmul
            self._remember_routing(lambda p=parameters.detach(): torch.sigmoid(p[-1, :, n_phy:n_phy + 2]))
        spec = self._spec(self.dynamic_params, self.routing)
        gplane = None
        if warm_up > 0:
            # the dense gradient plane starts zeroing while the warm-up kernel runs
            gplane = start_grad_plane(spec, parameters, warm_up, reusable=(self.dy_drop == 0))
            spec_w = self._spec(dyn_names=(), routing=False)
            if is_dual(parameters, x, current):
                # forward mode: the warm-up carries tangents into the initial states, as the
                # reference's no_grad warm-up does (hbv.py:327-346)
                current = hbv_states_only_dual(spec_w, x[:warm_up], parameters[:warm_up], current)
            else:
                with torch.no_grad():
                    current = hbv_states_only(spec_w, x[:warm_up], parameters[:warm_up].detach(),
                                              None, current)

        drop = self._draw_drop(ngrid)
        res = hbv_run(spec, x[warm_up:], parameters, None, current, drop=drop,
                      muwts=self.muwts, t_off=warm_up, gplane=gplane)

        if self.uh_carry_over and self.cache_states and self.routing:
            # route [history of the previous calls ; this run] and keep this run's part
            if torch.is_grad_enabled() and parameters.requires_grad:
                raise RuntimeError('uh_carry_over is a streaming-inference option: call the model under '
                                   'torch.no_grad() (the routed history of earlier calls carries no gradient)')
            refuse_forward_ad('uh_carry_over (the routed history of earlier calls carries no tangent)',
                              parameters, x, current)
            n_phy = len(self.parameter_bounds) * self.nmul
            q_run = torch.stack([res['flux'][f] for f in _R2F]).detach()
            hist = self._uh_hist
            if hist is not None and hist.shape[2] != ngrid:
                hist = None
            routed, self._uh_hist = route_with_history(
                spec, parameters[parameters.shape[0] - 1, :, n_phy:].detach(), parameters.shape[-1], q_run, hist)
            res['routed'] = [routed[i] for i in range(routed.shape[0])]

        states = tuple(res['state_out'][i] for i in range(5))
        self._states_cache = [s.detach() for s in states]
        if self.cache_states:
            self.states = self._states_cache
        return self._flux_dict(res, x[warm_up:])

    def _flux_dict(self, res, x_run) -> dict[str, torch.Tensor]:
        flux, routed = res['flux'], res['routed']
        out = {}
        for key, src in _FLUX_KEYS:
            if key == 'capillary' and not self._capillary:
                continue
            if src == 'pet':
                val = x_run[:, :, self.variables.index('pet')]
            elif src[0] == 'r':
                # routing off: reference 2.0 semantics (hbv_2.py:620-626) — un-routed means
                val = routed[src[1]] if routed is not None else flux[_R2F[src[1]]]
            else:
                val = flux[src[1]]
            out[key] = val.unsqueeze(-1)
        if res['bfi'] is not None:
            out['BFI'] = res['bfi']
        else:
            out['BFI'] = 100 * (flux[A.F_Q2].sum(0) / (flux[A.F_QSIM].sum(0) + self.nearzero))
        if not self.warm_up_states:
            for key in out:
                if key != 'BFI':
                    out[key] = out[key][self.pred_cutoff:, :, :]
        return out

    # ------------------------------------------------------------------ seam
    def _PBM(self, forcing: torch.Tensor, states: tuple, full_param_dict: dict):
        """Reference-compatible seam (hbv.py:363-368): descaled parameter dict of
        [T, B, nmul] tensors in, (flux_dict, states) out (states only when
        ``self.initialize``).  The dict is packed once into a [T, B, n*nmul] tensor and
        handed to the same kernels with an identity descale."""
        names = list(self.parameter_bounds.keys())
        dyn = torch.cat([full_param_dict[k] for k in names], dim=-1).contiguous()
        n = len(names)
        spec = self._spec(dyn_names=names, routing=self.routing and not self.initialize)
        spec.apply_sigmoid = False
        spec.par_lo, spec.par_hi = [0.0] * n, [1.0] * n
        state_in = torch.stack(tuple(states))
        if self.initialize:
            refuse_forward_ad('the `initialize` run (its states are detached)', dyn, forcing, state_in)
            out = hbv_states_only(spec, forcing.contiguous(), dyn.detach(), None, state_in)
            return tuple(out[i] for i in range(5))
        if spec.routing:
            # routing parameters were descaled by the caller (self.routing_param_dict)
            ra = self.routing_param_dict['route_a'].view(-1, 1)
            rb = self.routing_param_dict['route_b'].view(-1, 1)
            T, B = forcing.shape[0], forcing.shape[1]
            rcols = torch.zeros(T, B, 2, device=dyn.device, dtype=dyn.dtype)
            rcols[-1] = torch.cat([ra, rb], dim=1)
            dyn = torch.cat([dyn, rcols], dim=-1).contiguous()
            spec.route_bounds = ((0.0, 1.0), (0.0, 1.0))
        res = hbv_run(spec, forcing.contiguous(), dyn, None, state_in, muwts=getattr(self, 'muwts', None))
        states = tuple(res['state_out'][i] for i in range(5))
        return self._flux_dict(res, forcing), states


_R2F = (A.F_QSIM, A.F_Q0, A.F_Q1, A.F_Q2)
