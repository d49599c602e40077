"""Ensemble controller with the reference's API (marl/controllers/ensemble_agent_controller.py:10-152): a fixed-policy
league opponent whose agents infer either with the native (shared) network or with a per-agent network of the ensemble.

Inference only, as in the reference ("can only be used as a fixed policy opponent within league training").  The
native pass is BasicMAC's fused launch over all agents; every ensemble agent adds one dense-input launch of the same
kernel over its own rows, whose Q-values replace the native ones.  The reference builds the per-agent inputs with
`x.reshape(n_agents, -1)` (`:78`), which is only meaningful for batch size 1 (its steppers assert that); here the rows
of agent `aid` are taken for every batch element, which is the same thing at batch size 1.
"""
from __future__ import annotations

from typing import Dict

import torch as th

from .._native import MalError
from ..exceptions import HiddenStateNotInitialized
from .basic_controller import BasicMAC


class EnsembleMAC(BasicMAC):
    def __init__(self, scheme, groups, args):
        super().__init__(scheme, groups, args)
        self.ensemble: Dict[int, object] = dict()      # agent id -> AgentNetwork
        self.native_hidden_states = None
        self.ensemble_hidden_states = None
        self._all_ids = set(range(self.n_agents))

    # ------------------------------------------------------------------ inference
    def select_actions(self, ep_batch, t_ep, t_env, bs=slice(None), test_mode=False, u=None, e=None):
        if not self.ensemble:                            # nothing replaced: the fully fused path
            self.hidden_states = self.native_hidden_states
            out = super().select_actions(ep_batch, t_ep, t_env, bs=bs, test_mode=test_mode, u=u, e=e)
            self.native_hidden_states = self.hidden_states
            return out
        avail_actions = ep_batch["avail_actions"][:, t_ep]
        with self._no_recording():
            agent_outs = self.forward(ep_batch, t_ep, test_mode=test_mode)
        return self.action_selector.select(agent_outs[bs], avail_actions[bs], t_env, test_mode, u=u, e=e)

    def forward(self, ep_batch, t, test_mode=False):
        if self.native_hidden_states is None:
            raise HiddenStateNotInitialized()
        if self.ensemble and self._pool is not None:
            raise MalError("per-match policies do not run ensemble agents")
        if self.ensemble and getattr(self.args, "autograd_forward", False) and th.is_grad_enabled():
            raise MalError("EnsembleMAC.forward does not record autograd nodes for ensemble agents (a fixed-policy opponent); "
                           "call it under torch.no_grad() or switch args.autograd_forward off")
        self.hidden_states = self.native_hidden_states
        agent_outs = super().forward(ep_batch, t, test_mode=test_mode)          # [B, N, A], native net for everyone
        self.native_hidden_states = self.hidden_states
        if self.ensemble:
            B = ep_batch.batch_size
            inputs = self._build_inputs(ep_batch, t).view(B, self.n_agents, -1)
            for aid, agent in self.ensemble.items():
                q, h = agent(inputs[:, aid].contiguous(), self.ensemble_hidden_states[aid])
                agent_outs[:, aid, :] = q
                self.ensemble_hidden_states[aid] = h
        return agent_outs

    def init_hidden(self, batch_size):
        self._check_pool_batch(batch_size)
        self.native_hidden_states = self.agent.init_hidden().unsqueeze(0).expand(batch_size, self.n_agents, -1)
        self.hidden_states = self.native_hidden_states
        self.ensemble_hidden_states = {aid: agent.init_hidden().unsqueeze(0).expand(batch_size, 1, -1)
                                       for aid, agent in self.ensemble.items()}

    # ------------------------------------------------------------------ state handling
    def load_state(self, other_mac: "EnsembleMAC"):
        self.agent.load_state_dict(other_mac.agent.state_dict())
        for aid, agent in getattr(other_mac, "ensemble", {}).items():
            self._merge(aid, agent.state_dict())

    def load_state_dict(self, agent=None, ensemble=None):
        if agent is not None:
            self.agent.load_state_dict(agent)
        if ensemble is not None:
            for aid, state in ensemble.items():
                self._merge(aid, state)

    def _merge(self, aid, state):
        """Load into the ensemble member `aid`, building it first if needed.  (The reference's `load_state` inserts
        the OTHER controller's module object instead of the freshly built copy, SURVEY.md appendix A; the copy is used
        here, which is what `load_state_dict` does in the reference too.)"""
        if aid not in self.ensemble:
            self.ensemble[aid] = self._build_agent(self.input_shape)
        self.ensemble[aid].load_state_dict(state)

    def parameters(self):
        return list(self.agent.parameters())     # the reference's list arithmetic discards the ensemble's (appendix A)

    def update_trained_steps(self, update):
        super().update_trained_steps(update)

    def save_models(self, path, name):
        th.save(self.agent.state_dict(), f"{path}/{name}agent.th")
        for aid, agent in self.ensemble.items():
            th.save(agent.state_dict(), f"{path}/{name}ensemble_agent{aid}.th")

    def load_models(self, path, name):
        self.agent.load_state_dict(th.load("{}/{}agent.th".format(path, name), map_location=lambda storage, loc: storage))

    @property
    def n_specific_agents(self):
        return len(self.ensemble)

    @property
    def n_native_agents(self):
        return self.n_agents - self.n_specific_agents

    @property
    def ensemble_ids(self):
        return list(self.ensemble.keys())

    @property
    def native_agents_ids(self):
        return list(self._all_ids.difference(self.ensemble_ids))
