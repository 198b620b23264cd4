"""HBV adjoint (implicit scheme) — B200-native drop-in for ``hydrodl2/models/hbv/hbv_adj.py``.

Same constructor, attributes and ``forward(x_dict, parameters) -> {'flow_sim': [T-warm_up, B, 1]}``
contract as ``HbvAdj`` (hbv_adj.py:15-330).  The reference class cannot be imported (encrypted
``batch_jacobian.pye``) and has fatal defects (SURVEY.md §8 c2), so behaviour is defined by the
algorithm as written there, restated in ``oracle/hbv_adj_oracle.py``:

* backward-Euler step ``G(x) = (x - xt)/dt - f(x, theta_t, t) = 0`` with the 12-flux right-hand
  side of hbv_adj.py:341-498, solved by Newton per (basin, component) lane in one CUDA kernel
  (csrc/hbv_adj.cu) — analytic block-triangular Jacobian instead of ``batchJacobian`` +
  ``torch.linalg.solve`` + three host syncs per iteration (hbv_adj.py:531-581);
* gradients by the adjoint the reference intends (hbv_adj.py:620-633), analytic dG/dp instead
  of the float64 forward difference of core/calc/fdj.py;
* differentiable warm-up with static parameters from row ``warm_up-1`` (hbv_adj.py:257-274),
  states start at zero (:254), flux read at the end-of-step state (:309-313), nmul mean
  (:315-317), gamma-UH routing with lenF 15 (:319-325).

Extensions (not in the reference; the explicit models have them too):

* gradient w.r.t. the forcings: when ``x_dict['x_phy']`` requires grad, backward fills
  ``x_phy.grad`` — columns prcp / tmean / pet, warm-up rows included (the warm-up is
  differentiable here), other columns 0 — from the same adjoint sweep (lambda^T df/d(P, T, Ep)).
  If ``parameters`` does not require grad (variational precipitation data assimilation), no
  parameter-gradient tensor is allocated;
* state carry-over between calls: ``cache_states`` (the next call starts from the last call's
  final states instead of zeros, its warm-up included), ``get_states()``, ``load_states()``, and
  ``uh_carry_over`` (with ``cache_states`` and routing: the last lenF - 1 steps of the un-routed
  flow are routed together with the next call, so a run stepped chunk by chunk gives the routed
  flow of the one-shot run; inference only).

Deviations (documented in DESIGN.md §4 K3): per-lane stopping rule (the reference's is a
whole-batch max, :539-544); ``rout_params_name`` typo (:282) fixed; without ``parBETAET`` in
``dynamic_params`` the reference indexes a 13th parameter that does not exist (:380-383) — here
the evaporation exponent is then 1.
"""

from __future__ import annotations

from typing import Any, Optional, Union

import torch

from ... import _cabi as A
from ...ops import RunSpec, hbv_adj_run, route_with_history


class HbvAdj(torch.nn.Module):
    """Multi-component HBV with an implicit numerical scheme and adjoint gradients."""

    def __init__(
        self,
        config: Optional[dict[str, Any]] = None,
        device: Optional[torch.device] = None,
    ) -> None:
        super().__init__()
        self.name = 'HBV Adjoint'
        self.config = config
        self.initialize = False
        self.warm_up = 0
        self.dynamic_params = []
        self.dy_drop = 0.0
        self.variables = ['prcp', 'tmean', 'pet']
        self.routing = True
        self.comprout = False
        self.nearzero = 1e-5
        self.nmul = 1
        self.ad_efficient = True
        self.device = device
        self.cache_states = False
        self.uh_carry_over = False
        self._uh_hist = None
        self.states, self._states_cache = None, None
        self.state_names = ['SNOWPACK', 'MELTWATER', 'SM', 'SUZ', 'SLZ']
        # Newton controls (extension): reference gtol = 1e-3, <= 4 updates (hbv_adj.py:518-519)
        self.newton_tol = 1e-3
        self.newton_max_updates = 8
        self.parameter_bounds = {
            'parBETA': [1.0, 6.0], 'parFC': [50, 1000], 'parK0': [0.05, 0.9],
            'parK1': [0.01, 0.5], 'parK2': [0.001, 0.2], 'parLP': [0.2, 1],
            'parPERC': [0, 10], 'parUZL': [0, 100], 'parTT': [-2.5, 2.5],
            'parCFMAX': [0.5, 10], 'parCFR': [0, 0.1], 'parCWH': [0, 0.2],
        }
        self.routing_parameter_bounds = {'rout_a': [0, 2.9], 'rout_b': [0, 6.5]}

        if not device:
            self.device = torch.device('cuda' if torch.cuda.is_available() else 'cpu')

        if config is not None:
            self.warm_up = config.get('warm_up', self.warm_up)
            self.dy_drop = config.get('dy_drop', self.dy_drop)
            self.dynamic_params = config['dynamic_params'].get(
                self.__class__.__name__, self.dynamic_params
            )
            self.variables = config.get('variables', self.variables)
            self.routing = config.get('routing', self.routing)
            self.comprout = config.get('comprout', self.comprout)
            self.nearzero = config.get('nearzero', self.nearzero)
            self.nmul = config.get('nmul', self.nmul)
            self.ad_efficient = config.get('ad_efficient', self.ad_efficient)
            self.newton_tol = config.get('newton_tol', self.newton_tol)
            self.newton_max_updates = config.get('newton_max_updates', self.newton_max_updates)
            self.cache_states = config.get('cache_states', self.cache_states)
            self.uh_carry_over = config.get('uh_carry_over', self.uh_carry_over)
            if 'parBETAET' in self.dynamic_params:
                self.parameter_bounds['parBETAET'] = [0.3, 5]

        self.set_parameters()
        self.newton_stats = None

    def get_states(self) -> Optional[tuple[torch.Tensor, ...]]:
        """Final states of the last forward (SNOWPACK, MELTWATER, SM, SUZ, SLZ), each [B, nmul] —
        a tuple, so that ``load_states(get_states())`` round-trips."""
        return self._states_cache

    def load_states(self, states: tuple[torch.Tensor, ...]) -> None:
        """Start the next forward (with ``cache_states``) from `states` (hbv.py:148-168: same
        checks, same errors; stored detached)."""
        for state in states:
            if not isinstance(state, torch.Tensor):
                raise ValueError("Each element in `states` must be a tensor.")
        nstates = len(self.state_names)
        if not (isinstance(states, tuple) and len(states) == nstates):
            raise ValueError(f"`states` must be a tuple of {nstates} tensors.")
        self.states = tuple(s.detach().to(self.device, dtype=torch.float32) for s in states)
        self._uh_hist = None         # a new starting point: no runoff history to route

    def set_parameters(self) -> None:
        """hbv_adj.py:99-111."""
        self.phy_param_names = self.parameter_bounds.keys()
        if self.routing:
            self.routing_param_names = self.routing_parameter_bounds.keys()
        else:
            self.routing_param_names = []
        self.learnable_param_count = len(self.phy_param_names) * self.nmul + len(
            self.routing_param_names
        )

    def _spec(self, dyn_names, routing: bool) -> RunSpec:
        names = list(self.parameter_bounds.keys())
        n = len(names)
        src = [A.SRC_DYN_T if nm in dyn_names else A.SRC_DYN_LAST for nm in names]
        return RunSpec(
            variant=A.VARIANT_ADJ, n_par=n, betaet='parBETAET' in self.parameter_bounds,
            apply_sigmoid=True, par_src=src, par_col=[i * self.nmul for i in range(n)],
            par_lo=[self.parameter_bounds[k][0] for k in names],
            par_hi=[self.parameter_bounds[k][1] for k in names],
            nmul=self.nmul, nflux=1, nearzero=self.nearzero,
            var_index=tuple(self.variables.index(v) for v in ('prcp', 'tmean', 'pet')),
            routing=routing, route_src='dyn_last', route_col=n * self.nmul,
            route_bounds=tuple(tuple(v) for v in self.routing_parameter_bounds.values()),
            lenF=15, n_routed=1, bfi=False,
        )

    def _draw_drop(self, ngrid: int) -> Optional[torch.Tensor]:
        """One CPU bernoulli draw per dynamic parameter, in bounds order (hbv_adj.py:186-191).
        The reference draws per (component, basin) lane ([1, B*nmul], component-major);
        the kernel applies one mask per basin, so dropout > 0 uses a per-basin draw here."""
        if self.dy_drop <= 0 or not self.dynamic_params:
            return None
        names = list(self.parameter_bounds.keys())
        pmat = torch.ones([1, ngrid]) * self.dy_drop
        mask = torch.zeros(len(names), ngrid, dtype=torch.uint8)
        for i, nm in enumerate(names):
            if nm in self.dynamic_params:
                mask[i] = torch.bernoulli(pmat).view(ngrid).to(torch.uint8)
        return mask.to(self.device) if bool(mask.any()) else None

    def forward(
        self,
        x_dict: dict[str, torch.Tensor],
        parameters: torch.Tensor,
    ) -> Union[tuple, dict[str, torch.Tensor]]:
        """hbv_adj.py:227-330."""
        x = x_dict['x_phy']
        n_steps, bs, _ = x.size()
        need = len(self.parameter_bounds) * self.nmul + (2 if self.routing else 0)
        if parameters.shape[-1] < need:
            raise ValueError(f'parameters last dim {parameters.shape[-1]} < {need}')
        if (not self.states) or (not self.cache_states):
            y_init = torch.zeros((5, bs, self.nmul), dtype=torch.float32, device=self.device)   # :254
            self._uh_hist = None
        else:
            y_init = torch.stack(tuple(self.states))
            if tuple(y_init.shape) != (5, bs, self.nmul):
                raise ValueError(f'cached states have shape {tuple(y_init.shape[1:])}, this call needs '
                                 f'{(bs, self.nmul)} (basins, nmul)')
        carry = self.uh_carry_over and self.cache_states and self.routing
        if carry and torch.is_grad_enabled() and (parameters.requires_grad or x.requires_grad):
            raise RuntimeError('uh_carry_over is a streaming-inference option: call the model under '
                               'torch.no_grad() (the routed history of earlier calls carries no gradient)')
        spec_w = self._spec((), routing=False)
        spec = self._spec(self.dynamic_params, routing=self.routing and not carry)
        res = hbv_adj_run(spec_w, spec, x, parameters, y_init, drop=self._draw_drop(bs),
                          warm_up=self.warm_up, tol=self.newton_tol,
                          max_updates=self.newton_max_updates)
        self.newton_stats = res['stats']     # int32[2]: max updates, unconverged lane-steps
        if carry:
            # route [history of the previous calls ; this run] and keep this run's part
            n_phy = len(self.parameter_bounds) * self.nmul
            hist = self._uh_hist
            if hist is not None and hist.shape[2] != bs:
                hist = None
            routed, self._uh_hist = route_with_history(
                spec, parameters[parameters.shape[0] - 1, :, n_phy:].detach(), parameters.shape[-1],
                res['qsim'].unsqueeze(0), hist)
            flow = routed[0]
        else:
            flow = res['routed'] if self.routing else res['qsim']
        self._states_cache = tuple(res['state_out'][i].detach() for i in range(5))
        if self.cache_states:
            self.states = self._states_cache
        return {'flow_sim': flow.unsqueeze(-1)}
