"""HBV 2.0 hourly — B200-native drop-in for ``hydrodl2/models/hbv/hbv_2_hourly.py:14-897``."""

from __future__ import annotations

import torch

from ... import _cabi as A
from ._split import SplitHbv


class Hbv_2_hourly(SplitHbv):
    """HBV 2.0 at dt = 1/24 day: rates x dt store updates, state guard rails, Hortonian
    infiltration (parF0, parFMIN, parALPHA), lenF = 72, optional distributed (gage, unit)
    pair routing with a fractional lag (hbv_2_hourly.py:376-449,800-897).

    Returns ``{'Qs': unit runoff x dt, 'streamflow': gage flow}`` like the reference
    (hbv_2_hourly.py:740-796)."""

    _variant = A.VARIANT_HOURLY
    _name = 'HBV 2.0 Hourly'
    _lenF = 72

    def __init__(self, config=None, device=None) -> None:
        self.dt = 1.0 / 24
        self._dt = self.dt
        self.use_distr_routing = True
        self.infiltration = True
        self.lag_uh = True
        self._qs_buffer = []
        self._max_history = 100
        super().__init__(config, device)

    def _extend_bounds(self) -> None:
        self.parameter_bounds.update({
            'parF0': [5.0 / self.dt, 120.0 / self.dt],
            'parFMIN': [0.0, 1.0],
            'parALPHA': [0.5, 5.0],
        })
        self.routing_parameter_bounds = {'route_a': [0, 5.0], 'route_b': [0, 12.0]}
        self.distr_parameter_bounds = {
            'route_a': [0, 5.0], 'route_b': [0, 12.0], 'route_tau': [0, 48.0],
        }

    def get_states(self):
        # hbv_2_hourly.py:170 returns `_states_cache`; the reference never sets it (its forward
        # writes `_state_cache`, SURVEY.md §5) — here both names hold the series.
        return self._states_cache

    def _set_parameters(self) -> None:
        super()._set_parameters()
        self.learnable_param_count3 = len(self.distr_parameter_bounds)
        self.learnable_param_count = (
            self.learnable_param_count1 + self.learnable_param_count2 + self.learnable_param_count3
        )

    def _descale_distr_parameters(self, distr_params: torch.Tensor) -> dict[str, torch.Tensor]:
        """hbv_2_hourly.py:350-374."""
        out = {}
        for i, name in enumerate(self.distr_parameter_bounds.keys()):
            lo, hi = self.distr_parameter_bounds[name]
            out[name] = distr_params[:, i] * (hi - lo) + lo
        return out

    def forward(self, x_dict: dict[str, torch.Tensor], parameters, states=None) -> dict[str, torch.Tensor]:
        """hbv_2_hourly.py:376-449.  `states` (optional tuple of 5 [B, nmul] tensors) overrides the
        initial storages — used by Hbv_2_mts, which hands over the daily model's final states."""
        x, dyn, sta, current, ngrid = self._prep(x_dict, parameters, states)
        attrs = self._attrs(x_dict)
        drop = self._draw_drop(ngrid)
        res = self._run(x, dyn, sta, current, attrs, drop, self.routing)
        self._store_states(res)
        if self.initialize:
            return {}
        distr = parameters[2] if len(parameters) > 2 else None
        return self._flux_from_run(res, x, x_dict.get('outlet_topo'), x_dict.get('areas'), distr)

    def _flux_from_run(self, res, x, outlet_topo=None, areas=None, distr=None):
        """hbv_2_hourly.py:740-796.  `distr`: [n_pairs, 3] in [0, 1], or the reference's descaled
        dict {'route_a', 'route_b', 'route_tau'} (from `_descale_distr_parameters`)."""
        qs = (res['routed'][0] if res['routed'] is not None else res['flux'][A.F_QSIM])
        out = {'Qs': qs.unsqueeze(-1) * self.dt}
        if not self.warm_up_states:
            # hbv_2_hourly.py:761-764: `pred_cutoff` is never set by the hourly model (stays 0)
            out['Qs'] = out['Qs'][self.pred_cutoff:, :, :]
        if self.use_distr_routing:
            from ...routing import distr_routing
            bounds = tuple(tuple(v) for v in self.distr_parameter_bounds.values())
            if isinstance(distr, dict):
                distr = torch.stack([distr[k] for k in self.distr_parameter_bounds.keys()], dim=1)
                bounds = tuple((0.0, 1.0) for _ in bounds)
            if self.cache_states:   # streaming: keep <= _max_history steps of runoff history
                from ...ops import refuse_forward_ad
                refuse_forward_ad('the streaming runoff history of `cache_states` (it is detached)', out['Qs'])
                self._qs_buffer.append(out['Qs'].detach())
                if len(self._qs_buffer) > self._max_history:
                    self._qs_buffer.pop(0)
                qs_history = torch.cat(self._qs_buffer, dim=0)
            else:
                qs_history = out['Qs']
            # (the caller's own tensors key the topology cache; the index is built on the device)
            rout = distr_routing(qs_history, distr, outlet_topo, areas, lenF=self.lenF,
                                 lag_uh=self.lag_uh, bounds=bounds)
            out['streamflow'] = rout[-1:] if self.cache_states else rout
        return out

    def distr_routing(self, Qs, distr_params_dict, outlet_topo, areas):
        """Same signature and result as the reference method (hbv_2_hourly.py:800-855):
        DESCALED pair parameters in, ``{'Qs_rout': [T, n_gages, 1]}`` out."""
        from ...routing import distr_routing
        names = list(self.distr_parameter_bounds.keys())
        par = torch.stack([distr_params_dict[k] for k in names], dim=1)
        rout = distr_routing(Qs, par, outlet_topo, areas, lenF=self.lenF,
                             lag_uh=self.lag_uh, bounds=tuple((0.0, 1.0) for _ in names))
        return {'Qs_rout': rout}
