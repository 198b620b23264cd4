"""Host-side logic shared by the split-parameter models (HBV 2.0 and 2.0-hourly).

Mirrors ``Hbv_2`` (models/hbv/hbv_2.py:8-670) and ``Hbv_2_hourly``
(models/hbv/hbv_2_hourly.py:14-897): `parameters` is a tuple
``(dynamic [T, B, n_dy*nmul], static [B, n_sta*nmul (+2 routing)] [, distr [n_pairs, 3]])``
already in [0, 1] (no sigmoid, hbv_2.py:211-230), `x_dict` carries ``ac_all`` / ``elev_all``,
states are initialised to 0.001 or taken from ``self.states``.  Dynamic columns follow the
order of ``config['dynamic_params']``, static columns the order of ``parameter_bounds`` minus
the dynamic names (hbv_2.py:258,363-367).
"""

from __future__ import annotations

from typing import Any, Optional

import torch

from ... import _cabi as A
from ...ops import RunSpec, hbv_run, hbv_states_only, refuse_forward_ad
from ._seam import SplitSeam

_BASE_BOUNDS = {
    'parBETA': [1.0, 6.0], 'parFC': [50, 1000], 'parK0': [0.05, 0.9], 'parK1': [0.01, 0.5],
    'parK2': [0.001, 0.2], 'parLP': [0.2, 1], 'parPERC': [0, 10], 'parUZL': [0, 100],
    'parTT': [-2.5, 2.5], 'parCFMAX': [0.5, 10], 'parCFR': [0, 0.1], 'parCWH': [0, 0.2],
    'parBETAET': [0.3, 5], 'parC': [0, 1], 'parRT': [0, 20], 'parAC': [0, 2500],
}

_FLUX = (
    ('AET_hydro', A.F_AET), ('SWE', A.F_SWE), ('streamflow_no_rout', A.F_QSIM),
    ('srflow_no_rout', A.F_Q0), ('ssflow_no_rout', A.F_Q1), ('gwflow_no_rout', A.F_Q2),
    ('recharge', A.F_RECHARGE), ('excs', A.F_EXCS), ('evapfactor', A.F_EVAPFACTOR),
    ('tosoil', A.F_TOSOIL), ('percolation', A.F_PERC), ('capillary', A.F_CAPILLARY),
)


class SplitHbv(SplitSeam, torch.nn.Module):
    """Base of `Hbv_2` and `Hbv_2_hourly`."""

    _variant = A.VARIANT_HBV2
    _name = 'HBV 2.0'
    _lenF = 15
    _dt = 1.0
    _states_attr = '_state_cache'   # where forward stores the state series (the two reference
                                    # files disagree on the attribute name; both are kept)

    def __init__(self, config: Optional[dict[str, Any]] = None,
                 device: Optional[torch.device] = None) -> None:
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
        self.routing = False
        self.lenF = self._lenF
        self.comprout = False
        self.muwts = None
        self.nearzero = 1e-5
        self.nmul = 1
        self.cache_states = False
        self.device = device
        self.ckpt_interval = 0    # checkpoint interval of the adjoint: 0 = auto (see _packed.py)
        # extension: hbv_2.py:571-575 materialises 5 x [T, B, nmul] state series on every
        # forward (112 GB at BASELINE config 4).  True = reference behaviour; False keeps only
        # the final states, exposed as series of length 1 so `s[-1]` users keep working.
        self.state_series = True

        self.states, self._state_cache, self._states_cache = None, None, None
        # extension (SURVEY f2; see _packed.py): carry the runoff history of the fused <= 16-tap UH
        # routing across `cache_states` calls (the hourly model keeps its own `_qs_buffer`)
        self.uh_carry_over = False
        self._uh_hist = None

        self.state_names = ['SNOWPACK', 'MELTWATER', 'SM', 'SUZ', 'SLZ']
        self.flux_names = [
            'streamflow', 'srflow', 'ssflow', 'gwflow', 'AET_hydro', 'PET_hydro', 'SWE',
            'streamflow_no_rout', 'srflow_no_rout', 'ssflow_no_rout', 'gwflow_no_rout',
            'recharge', 'excs', 'evapfactor', 'tosoil', 'percolation', 'capillary', 'BFI',
        ]
        self.parameter_bounds = dict(_BASE_BOUNDS)
        self._extend_bounds()
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
            self.cache_states = config.get('cache_states', self.cache_states)
            self.uh_carry_over = config.get('uh_carry_over', self.uh_carry_over)
            self.ckpt_interval = config.get('ckpt_interval', self.ckpt_interval)
            self.state_series = config.get('state_series', self.state_series)
        self._set_parameters()

    def _extend_bounds(self) -> None:
        self.routing_parameter_bounds = {'route_a': [0, 2.9], 'route_b': [0, 6.5]}

    # ------------------------------------------------------------------ state API
    def _init_states(self, ngrid: int) -> tuple[torch.Tensor, ...]:
        return tuple(
            torch.full((ngrid, self.nmul), 0.001, dtype=torch.float32, device=self.device)
            for _ in self.state_names
        )

    def get_states(self):
        return self._state_cache

    def load_states(self, states: tuple[torch.Tensor, ...]) -> None:
        for state in states:
            if not isinstance(state, torch.Tensor):
                raise ValueError("Each element in `states` must be a tensor.")
        nstates = len(self.state_names)
        if not (isinstance(states, tuple) and len(states) == nstates):
            raise ValueError(f"`states` must be a tuple of {nstates} tensors.")
        self.states = tuple(s.detach().to(self.device, dtype=torch.float32) for s in states)
        self._uh_hist = None

    def _set_parameters(self) -> None:
        self.phy_param_names = self.parameter_bounds.keys()
        self.routing_param_names = self.routing_parameter_bounds.keys() if self.routing else []
        self.learnable_param_count1 = len(self.dynamic_params) * self.nmul
        self.learnable_param_count2 = (
            len(self.phy_param_names) - len(self.dynamic_params)
        ) * self.nmul + len(self.routing_param_names)
        self.learnable_param_count = self.learnable_param_count1 + self.learnable_param_count2

    # ------------------------------------------------------------------ run plan
    def _spec(self, routing: bool) -> RunSpec:
        names = list(self.parameter_bounds.keys())
        dyn = list(self.dynamic_params)
        sta = [n for n in names if n not in dyn]
        src, col = [], []
        for nm in names:
            if nm in dyn:
                src.append(A.SRC_DYN_T)
                col.append(dyn.index(nm) * self.nmul)
            else:
                src.append(A.SRC_STA)
                col.append(sta.index(nm) * self.nmul)
        return RunSpec(
            variant=self._variant, n_par=len(names), betaet=True, apply_sigmoid=False,
            par_src=src, par_col=col,
            par_lo=[self.parameter_bounds[k][0] for k in names],
            par_hi=[self.parameter_bounds[k][1] for k in names],
            nmul=self.nmul, nflux=12, nearzero=self.nearzero, dt=self._dt,
            var_index=tuple(self.variables.index(v) for v in ('prcp', 'tmean', 'pet')),
            ckpt_interval=self.ckpt_interval, routing=routing, route_src='sta',
            route_col=len(sta) * self.nmul,
            route_bounds=tuple(tuple(v) for v in self.routing_parameter_bounds.values()),
            lenF=self.lenF, n_routed=1 if self._variant == A.VARIANT_HOURLY else 4,
            bfi=self._variant != A.VARIANT_HOURLY, state_series=self.state_series,
        )

    def _draw_drop(self, ngrid: int) -> Optional[torch.Tensor]:
        """One CPU bernoulli draw per dynamic parameter in `dynamic_params` order
        (hbv_2.py:256-262) -> uint8 [n_par, B] on device or None."""
        names = list(self.parameter_bounds.keys())
        pmat = torch.ones([1, ngrid, 1]) * self.dy_drop
        mask = torch.zeros(len(names), ngrid, dtype=torch.uint8)
        anyset = False
        for nm in self.dynamic_params:
            dr = torch.bernoulli(pmat).view(ngrid)
            if self.dy_drop > 0:
                mask[names.index(nm)] = dr.to(torch.uint8)
                anyset = anyset or bool(dr.any())
        return mask.to(self.device) if anyset else None

    def _attrs(self, x_dict) -> torch.Tensor:
        ac = x_dict['ac_all'].to(self.device, dtype=torch.float32).reshape(-1)
        el = x_dict['elev_all'].to(self.device, dtype=torch.float32).reshape(-1)
        return torch.stack([ac, el]).contiguous()

    def _prep(self, x_dict, parameters, states=None):
        x = x_dict['x_phy'].contiguous()
        self.muwts = x_dict.get('muwts', None)
        ngrid = x.shape[1]
        dyn = parameters[0]
        sta = parameters[1]
        if dyn is not None and dyn.shape[-1] == 0:
            dyn = None
        if self.routing:     # `routing_param_dict` (hbv_2.py:349-350), materialised only if someone reads it
            rc = self._route_col()
            self._remember_routing(lambda s_=sta.detach(): s_[:, rc:rc + 2])
        if states is not None:
            current = torch.stack(tuple(states))
        elif (not self.states) or (not self.cache_states):
            current = torch.stack(self._init_states(ngrid))
            self._uh_hist = None
        else:
            current = torch.stack(tuple(self.states))
        return x, dyn, sta, current, ngrid

    def _store_states(self, res) -> tuple:
        if res['series'] is not None:
            series = tuple(res['series'][i] for i in range(5))
        else:
            series = tuple(res['state_out'][i].unsqueeze(0) for i in range(5))
        self._state_cache = series
        self._states_cache = series
        if self.cache_states:
            self.states = tuple(s[-1].detach() for s in series)
        return series

    def _run(self, x, dyn, sta, current, attrs, drop, routing):
        if self.comprout:
            raise RuntimeError('comprout=True is not supported (it fails in the reference as well)')
        # per-unit UH routing with more than 16 taps (the hourly model's lenF = 72,
        # hbv_2_hourly.py:684-705) runs after the recurrence through the shared-memory-staged
        # convolution of csrc/pair_route.cu (routing.unit_routing); <= 16 taps stay fused (K4)
        long_uh = routing and self.lenF > 16 and not self.initialize
        spec = self._spec(routing and not long_uh)
        if self.initialize:
            # hbv_2.py:630-632: only the storages are returned
            refuse_forward_ad('`initialize=True` (its states are detached; this includes Hbv_2_mts)',
                              x, dyn, sta, current)
            with torch.no_grad():
                spec.state_series = False
                out = hbv_states_only(spec, x, None if dyn is None else dyn.detach().contiguous(),
                                      sta.detach().contiguous(), current, drop=drop, attrs=attrs)
            return {'flux': None, 'routed': None, 'bfi': None, 'state_out': out, 'series': None}
        res = hbv_run(spec, x, dyn, sta, current, drop=drop, attrs=attrs, muwts=self.muwts)
        if (self.uh_carry_over and self.cache_states and spec.routing
                and self._variant != A.VARIANT_HOURLY):
            if torch.is_grad_enabled() and any(t is not None and t.requires_grad for t in (dyn, sta)):
                raise RuntimeError('uh_carry_over is a streaming-inference option: call the model under '
                                   'torch.no_grad() (the routed history of earlier calls carries no gradient)')
            refuse_forward_ad('uh_carry_over (the routed history of earlier calls carries no tangent)',
                              x, dyn, sta, current)
            from ...ops import route_with_history
            rc = self._route_col()
            q_run = torch.stack([res['flux'][f] for f in (A.F_QSIM, A.F_Q0, A.F_Q1, A.F_Q2)]).detach()
            hist = self._uh_hist
            if hist is not None and hist.shape[2] != x.shape[1]:
                hist = None
            routed, self._uh_hist = route_with_history(spec, sta.detach()[:, rc:], sta.shape[-1], q_run, hist)
            res['routed'] = [routed[i] for i in range(routed.shape[0])]
        if long_uh:
            rc = self._route_col()
            self._apply_long_uh(res, x.shape[0], sta[:, rc:rc + 2],
                                tuple(tuple(v) for v in self.routing_parameter_bounds.values()))
        return res

    def _apply_long_uh(self, res, T, route_ab, bounds) -> None:
        from ...routing import unit_routing
        n_r = 1 if self._variant == A.VARIANT_HOURLY else 4
        series = (A.F_QSIM, A.F_Q0, A.F_Q1, A.F_Q2)[:n_r]
        res['routed'] = [unit_routing(res['flux'][f], route_ab, min(self.lenF, T), bounds) for f in series]
        if self._variant != A.VARIANT_HOURLY:
            res['bfi'] = 100 * (res['routed'][3].sum(0) / (res['routed'][0].sum(0) + self.nearzero))

    def _route_col(self) -> int:
        """First routing column of the static tensor (after the static physical parameters)."""
        return (len(self.parameter_bounds) - len(self.dynamic_params)) * self.nmul

    # ------------------------------------------------------------------ seam
    def _PBM(self, forcing, Ac, Elevation, states, phy_dy_params_dict, phy_static_params_dict,
             outlet_topo=None, areas=None, distr_params_dict=None):
        """Reference-compatible seam (hbv_2.py:392-400, hbv_2_hourly.py:451-462): DESCALED
        parameter dicts in (dynamic [T, B, nmul], static [B, nmul]); returns
        ``(flux_dict, state_series)``.  The dicts are packed once and run through the same kernels
        with an identity descale."""
        names = list(self.parameter_bounds.keys())
        dyn_names = [n for n in names if n in phy_dy_params_dict]
        sta_names = [n for n in names if n not in phy_dy_params_dict]
        dyn = (torch.cat([phy_dy_params_dict[k] for k in dyn_names], dim=-1).contiguous()
               if dyn_names else None)
        sta = torch.cat([phy_static_params_dict[k] for k in sta_names], dim=-1).contiguous()
        keep = (self.dynamic_params, self.dy_drop)
        self.dynamic_params, self.dy_drop = dyn_names, 0.0
        try:
            spec = self._spec(self.routing)
        finally:
            self.dynamic_params, self.dy_drop = keep
        n = len(names)
        spec.par_lo, spec.par_hi = [0.0] * n, [1.0] * n
        long_uh = None
        if spec.routing:
            ra = self.routing_param_dict['route_a'].view(-1, 1)
            rb = self.routing_param_dict['route_b'].view(-1, 1)
            if self.lenF > 16 and not self.initialize:
                long_uh = torch.cat([ra, rb], dim=1)          # already descaled: identity bounds
                spec.routing = False
            else:
                sta = torch.cat([sta, ra, rb], dim=1).contiguous()
                spec.route_bounds = ((0.0, 1.0), (0.0, 1.0))
        attrs = torch.stack([Ac.reshape(Ac.shape[0], -1)[:, 0], Elevation.reshape(Elevation.shape[0], -1)[:, 0]])
        attrs = attrs.to(self.device, dtype=torch.float32).contiguous()
        current = torch.stack(tuple(states))
        x = forcing.contiguous()
        if self.initialize:
            refuse_forward_ad('`initialize=True` (its states are detached)', x, dyn, sta, current)
            with torch.no_grad():
                spec.state_series = False
                out = hbv_states_only(spec, x, None if dyn is None else dyn.detach(), sta.detach(),
                                      current, attrs=attrs)
            return {}, tuple(out[i].unsqueeze(0) for i in range(5))
        res = hbv_run(spec, x, dyn, sta, current, attrs=attrs, muwts=self.muwts)
        if long_uh is not None:
            self._apply_long_uh(res, x.shape[0], long_uh, ((0.0, 1.0), (0.0, 1.0)))
        series = (tuple(res['series'][i] for i in range(5)) if res['series'] is not None
                  else tuple(res['state_out'][i].unsqueeze(0) for i in range(5)))
        return self._flux_from_run(res, x, outlet_topo, areas, distr_params_dict), series
