"""HBV 2.0 multi-timescale — drop-in for ``hydrodl2/models/hbv/hbv_2_mts.py:14-377``.

Orchestration only: a daily `Hbv_2` run warms the storages up (initialize=True, no gradient),
the states are handed over unchanged (identity state transfer, hbv_2_mts.py:343-349), the
low-frequency static parameters are re-used for the hourly run with the three hourly-only
infiltration parameters appended (param_transfer, hbv_2_mts.py:292-341), then `Hbv_2_hourly`
runs — all arithmetic is in the CUDA kernels the two sub-models use.  Spatial chunking of the
runoff generation and temporal chunking of the pair routing (hbv_2_mts.py:204-279) are kept; the
reference's chunked branch calls two methods that do not exist (`unpack_parameters`,
`_descale_rout_parameters`; SURVEY.md §8 c1) — here it works.
"""

from __future__ import annotations

from typing import Any, Optional

import torch

from .hbv_2 import Hbv_2
from .hbv_2_hourly import Hbv_2_hourly


class Hbv_2_mts(torch.nn.Module):
    """Daily warm-up -> hourly simulation with distributed routing."""

    def __init__(
        self,
        low_freq_config: Optional[dict[str, Any]] = None,
        high_freq_config: Optional[dict[str, Any]] = None,
        device: Optional[torch.device] = None,
    ) -> None:
        super().__init__()
        self.device = device if device is not None else torch.device('cpu')
        self.dtype = torch.float32
        self.low_freq_model = Hbv_2(low_freq_config, device=device)
        self.low_freq_model.initialize = True
        self.high_freq_model = Hbv_2_hourly(high_freq_config, device=device)
        self._state_cache = [None, None]
        self.states = (None, None)
        self.load_from_cache = False
        self.use_from_cache = False
        self.state_transfer_model = torch.nn.ModuleDict(
            {name: torch.nn.Identity() for name in self.high_freq_model.state_names}
        )
        self.train_spatial_chunk_size = high_freq_config['train_spatial_chunk_size']
        self.simulate_spatial_chunk_size = high_freq_config['simulate_spatial_chunk_size']
        self.simulate_temporal_chunk_size = high_freq_config['simulate_temporal_chunk_size']
        self.spatial_chunk_size = self.train_spatial_chunk_size
        self.simulate_mode = False
        self.train_warmup = high_freq_config['train_warmup']

    # ------------------------------------------------------------------ state API
    def get_states(self):
        return (self.low_freq_model.get_states(), self.high_freq_model.get_states())

    def load_states(self, state_tuple) -> None:
        if not isinstance(state_tuple, tuple) or len(state_tuple) != 2:
            raise ValueError("`states` must be a tuple of two tuples of tensors.")
        self._state_cache = tuple(
            tuple(s[-1].detach().to(self.device, dtype=self.dtype) for s in states)
            for states in state_tuple
        )
        if self.load_from_cache:
            self.low_freq_model.load_states(state_tuple[0])

    def set_mode(self, is_simulate: bool):
        if is_simulate:
            self.spatial_chunk_size = self.simulate_spatial_chunk_size
            self.simulate_mode = True
        else:
            self.spatial_chunk_size = self.train_spatial_chunk_size
            self.simulate_mode = False

    def state_transfer(self, states):
        d = dict(zip(self.high_freq_model.state_names, states))
        return [self.state_transfer_model[k](d[k]) for k in d.keys()]

    def param_transfer(self, low_freq_parameters, high_freq_parameters):
        """-> (hourly dynamic tensor, merged static tensor, distr tensor), all still in [0, 1]."""
        low, high = self.low_freq_model, self.high_freq_model
        nmul = high.nmul
        hi_names = [n for n in high.phy_param_names if n not in high.dynamic_params]
        lo_names = [n for n in low.phy_param_names if n not in low.dynamic_params]
        lo_sta = low_freq_parameters[1][:, :len(lo_names) * nmul]
        hi_sta = high_freq_parameters[1][:, :len(hi_names) * nmul].view(-1, len(hi_names), nmul)
        extra = [i for i, n in enumerate(hi_names) if n not in lo_names]
        merged = torch.cat([lo_sta, hi_sta[:, extra].reshape(hi_sta.shape[0], -1)], dim=1)
        if high.routing:
            merged = torch.cat([merged, high_freq_parameters[1][:, len(hi_names) * nmul:]], dim=1)
        distr = high_freq_parameters[2] if len(high_freq_parameters) > 2 else None
        return high_freq_parameters[0], merged, distr

    # ------------------------------------------------------------------ forward
    def _forward(self, x_dict, parameters):
        low_p, high_p = parameters
        low, high = self.low_freq_model, self.high_freq_model
        if self.use_from_cache and (self._state_cache[1] is not None):
            states = self.states[1]
        else:
            low.states = None
            keep = low.cache_states
            low.cache_states = True       # the hand-over needs `low.states` (hbv_2_mts.py:119-131)
            try:
                low({'x_phy': x_dict['x_phy_low_freq'], 'ac_all': x_dict['ac_all'],
                     'elev_all': x_dict['elev_all'], 'muwts': x_dict.get('muwts', None)}, low_p)
            finally:
                low.cache_states = keep
            self._state_cache[0] = low.states
            states = self.state_transfer(low.states)
            low.states = None
        dyn, sta, distr = self.param_transfer(low_p, high_p)
        xd = {'x_phy': x_dict['x_phy_high_freq'], 'ac_all': x_dict['ac_all'],
              'elev_all': x_dict['elev_all'], 'outlet_topo': x_dict.get('outlet_topo'),
              'areas': x_dict.get('areas'), 'muwts': x_dict.get('muwts', None)}
        params = [dyn, sta] + ([distr] if distr is not None else [])
        predictions = high(xd, params, states=tuple(states))
        hif = high._state_cache
        self._state_cache[1] = tuple(s.detach() for s in hif)
        if self.load_from_cache:
            self.states = (self._state_cache[0], tuple(s[-1] for s in hif))
        return predictions

    def forward(self, x_dict, parameters):
        from ...ops import refuse_forward_ad
        flat = [t for p in parameters for t in (p if isinstance(p, (tuple, list)) else (p,))]
        refuse_forward_ad('Hbv_2_mts (its daily warm-up states are detached)',
                          *flat, *(v for v in x_dict.values() if isinstance(v, torch.Tensor)))
        device = self.device
        n_units = x_dict['areas'].shape[0]
        high = self.high_freq_model
        if (not self.simulate_mode) and (n_units <= self.spatial_chunk_size):
            high.use_distr_routing = False
            return self._forward(x_dict, parameters)

        high.use_distr_routing = False
        preds = []
        topo = x_dict['outlet_topo']
        pair_cols = (topo == 1).nonzero(as_tuple=False)[:, 1]
        for i in range(0, n_units, self.spatial_chunk_size):
            j = min(i + self.spatial_chunk_size, n_units)
            in_chunk = (pair_cols >= i) & (pair_cols < j)
            cx = {
                'x_phy_low_freq': x_dict['x_phy_low_freq'][:, i:j].to(device),
                'x_phy_high_freq': x_dict['x_phy_high_freq'][:, i:j].to(device),
                'ac_all': x_dict['ac_all'][i:j].to(device),
                'elev_all': x_dict['elev_all'][i:j].to(device),
                'areas': x_dict['areas'][i:j].to(device),
                'outlet_topo': topo[:, i:j].to(device),
            }
            cp = ([parameters[0][0][:, i:j].to(device), parameters[0][1][i:j].to(device)],
                  [parameters[1][0][:, i:j].to(device), parameters[1][1][i:j].to(device),
                   parameters[1][2][in_chunk.to(parameters[1][2].device)].to(device)])
            preds.append(self._forward(cx, cp))
        predictions = self.concat_spatial_chunks(preds)
        runoff = predictions['Qs']
        n_t = runoff.shape[0]

        from ...routing import distr_routing
        bounds = tuple(tuple(v) for v in high.distr_parameter_bounds.values())
        distr = parameters[1][2].to(device)
        # the caller's own tensors key the topology cache (routing.pair_index); the index arrays
        # are built on the device once and reused by every temporal chunk and every later call
        topo_d, areas_d = topo, x_dict['areas']
        w = self.train_warmup
        routed = []
        for t in range(w, n_t, self.simulate_temporal_chunk_size):
            e = min(t + self.simulate_temporal_chunk_size, n_t)
            r = distr_routing(runoff[t - w:e], distr, topo_d, areas_d, lenF=high.lenF,
                              lag_uh=high.lag_uh, bounds=bounds)
            routed.append(r if t == w else r[w:])   # drop the routing warm-up of later chunks
        predictions['streamflow'] = torch.cat(routed, dim=0)
        return predictions

    @staticmethod
    def concat_spatial_chunks(pred_list):
        out = {}
        for key in pred_list[0].keys():
            dim = 1 if pred_list[0][key].ndim == 3 else 0
            out[key] = torch.cat([p[key] for p in pred_list], dim=dim)
        return out

    @staticmethod
    def concat_temporal_chunks(pred_list):
        out = {}
        for key in pred_list[0].keys():
            if pred_list[0][key].ndim == 3:
                out[key] = torch.cat([p[key] for p in pred_list], dim=0)
            else:
                out[key] = pred_list[0][key]
        return out
