"""Reference computations for agent inputs with `obs_last_action` / `obs_agent_id` switched off (test infrastructure).

The agent input is [obs | one-hot(a_{t-1}) | one-hot(agent id)] with the last two blocks optional
(basic_controller.py:80-101).  The numpy oracle assembles the full layout; an input without some of the blocks is
the full input with those columns removed, so a network over it is the full-layout network whose fc1 weight is zero
on the removed columns.  The learner reference therefore embeds fc1.weight into the full layout, runs
np_oracle.learner_forward_backward unchanged and reads the fc1 gradient back on the kept columns.  The torch functions
below assemble the reduced input directly (th.cat, as the reference does) and differentiate with autograd: they
check that embedding on CPU.
"""
from __future__ import annotations

from collections import OrderedDict

import numpy as np
import torch as th
import torch.nn.functional as F

from oracle import np_oracle as O
from oracle import rollout_oracle as RO
from oracle import torch_port as TP

LAYOUTS = [(True, True), (False, True), (True, False), (False, False)]   # (last_action, agent_id)


def input_columns(OBS, A, N, last_action=True, agent_id=True):
    """Columns of the full [OBS + A + N] layout that the switched layout keeps, in order."""
    cols = list(range(OBS))
    if last_action:
        cols += range(OBS, OBS + A)
    if agent_id:
        cols += range(OBS + A, OBS + A + N)
    return np.asarray(cols, dtype=np.int64)


def d_in(OBS, A, N, last_action=True, agent_id=True):
    return OBS + A * bool(last_action) + N * bool(agent_id)


def build_inputs(obs, actions_onehot, t, last_action=True, agent_id=True):
    """np_oracle.build_inputs for the switched layout: [B*N, d_in]."""
    _, _, N, OBS = obs.shape
    full = O.build_inputs(obs, actions_onehot, t)
    return full[:, input_columns(OBS, actions_onehot.shape[-1], N, last_action, agent_id)]


def embed_agent(p, cols, d_full):
    """Agent parameters over the full layout: fc1.weight zero on the columns the switched layout leaves out."""
    out = OrderedDict(p)
    w = p["fc1.weight"]
    full = np.zeros((w.shape[0], d_full), dtype=w.dtype)
    full[:, cols] = w
    out["fc1.weight"] = full
    return out


def learner_forward_backward(agent_p, target_agent_p, mixer_p, target_mixer_p, batch, *, last_action=True,
                             agent_id=True, **kw):
    """np_oracle.learner_forward_backward for the switched layout (see the module docstring)."""
    _, _, N, OBS = batch["obs"].shape
    A = batch["actions_onehot"].shape[-1]
    cols = input_columns(OBS, A, N, last_action, agent_id)
    d_full = OBS + A + N
    ref = O.learner_forward_backward(embed_agent(agent_p, cols, d_full), embed_agent(target_agent_p, cols, d_full),
                                     mixer_p, target_mixer_p, batch, **kw)
    ref["agent_grads"]["fc1.weight"] = np.ascontiguousarray(ref["agent_grads"]["fc1.weight"][:, cols])
    return ref


# ---------------------------------------------------------------------------------------------- torch, autograd
def torch_agent_step(p, batch, t, h, last_action=True, agent_id=True):
    """torch_port.agent_step with the switched _build_inputs (basic_controller.py:80-92)."""
    obs, onehot = batch["obs"], batch["actions_onehot"]
    B, _, N, _ = obs.shape
    parts = [obs[:, t]]
    if last_action:
        parts.append(th.zeros_like(onehot[:, t]) if t == 0 else onehot[:, t - 1])
    if agent_id:
        parts.append(th.eye(N, device=obs.device).unsqueeze(0).expand(B, -1, -1))
    inp = th.cat([x.reshape(B * N, -1) for x in parts], dim=1)
    x = F.relu(F.linear(inp, p["fc1.weight"], p["fc1.bias"]))
    if "gru.weight_ih" not in p:
        return F.linear(x, p["fc2.weight"], p["fc2.bias"]).view(B, N, -1), h
    h = th.gru_cell(x, h.reshape(-1, x.shape[1]), p["gru.weight_ih"], p["gru.weight_hh"], p["gru.bias_ih"],
                    p["gru.bias_hh"])
    return F.linear(h, p["fc2.weight"], p["fc2.bias"]).view(B, N, -1), h


def torch_loss_grads(agent_p, target_agent_p, mixer_p, target_mixer_p, batch, *, mixer, double_q, gamma,
                     last_action=True, agent_id=True):
    """loss.backward() of QLearner.train (q_learner.py:34-103, as torch_port.TorchPortLearner.train) in float64 on CPU.
    Returns (loss, agent grads, mixer grads) as numpy."""
    dt = th.float64
    ap = OrderedDict((k, th.tensor(v, dtype=dt, requires_grad=True)) for k, v in agent_p.items())
    tp = OrderedDict((k, th.tensor(v, dtype=dt)) for k, v in target_agent_p.items())
    mp = OrderedDict((k, th.tensor(v, dtype=dt, requires_grad=True)) for k, v in (mixer_p or {}).items())
    tmp = OrderedDict((k, th.tensor(v, dtype=dt)) for k, v in (target_mixer_p or {}).items())
    b = {k: th.tensor(v) for k, v in batch.items()}
    for k in ("obs", "actions_onehot", "state", "reward"):
        b[k] = b[k].to(dt)
    B, TT, N, _ = b["obs"].shape

    def unroll(p):
        h = th.zeros(B * N, O.H_DEFAULT, dtype=dt)
        outs = []
        for t in range(TT):
            q, h = torch_agent_step(p, b, t, h, last_action, agent_id)
            outs.append(q)
        return th.stack(outs, dim=1)

    rewards, actions = b["reward"][:, :-1], b["actions"][:, :-1]
    terminated = b["terminated"][:, :-1].to(dt)
    mask = b["filled"][:, :-1].to(dt)
    mask[:, 1:] = mask[:, 1:] * (1 - terminated[:, :-1])
    avail = b["avail_actions"]
    mac_out = unroll(ap)
    chosen = th.gather(mac_out[:, :-1], dim=3, index=actions).squeeze(3)
    target_out = unroll(tp)[:, 1:].detach()
    target_out[avail[:, 1:] == 0] = -9999999
    if double_q:
        det = mac_out.clone().detach()
        det[avail == 0] = -9999999
        tmax = th.gather(target_out, 3, det[:, 1:].max(dim=3, keepdim=True)[1]).squeeze(3)
    else:
        tmax = target_out.max(dim=3)[0]
    if mixer == "qmix":
        q_tot, tq_tot = TP.qmix(mp, chosen, b["state"][:, :-1]), TP.qmix(tmp, tmax, b["state"][:, 1:])
    else:
        q_tot, tq_tot = chosen.sum(dim=2, keepdim=True), tmax.sum(dim=2, keepdim=True)
    targets = rewards + gamma * (1 - terminated) * tq_tot
    masked = (q_tot - targets.detach()) * mask
    loss = (masked ** 2).sum() / mask.sum()
    loss.backward()
    return (float(loss.detach()), OrderedDict((k, v.grad.numpy()) for k, v in ap.items()),
            OrderedDict((k, v.grad.numpy()) for k, v in mp.items()))


# ---------------------------------------------------------------------------------------------- rollout
class OracleMAC(RO.OracleMAC):
    """rollout_oracle.OracleMAC over the switched input layout."""

    def __init__(self, params, n_agents, n_actions, draws, last_action=True, agent_id=True, **kw):
        super().__init__(params, n_agents, n_actions, draws, **kw)
        self.last_action, self.agent_id = last_action, agent_id

    def select_actions(self, batch, t_ep, t_env, test_mode):
        inp = build_inputs(batch["obs"][None].astype(self.dtype), batch["actions_onehot"][None].astype(self.dtype), t_ep,
                           self.last_action, self.agent_id)
        q, self.h, _ = O.drqn_step(self.p, inp, self.h)
        eps = 0.0 if test_mode else O.epsilon_linear(*self.sched, t_env)
        u, e = self.draws(t_ep)
        self.q_log.append(q.copy())
        a, g = O.eps_greedy_select(q.reshape(1, self.N, self.A), batch["avail_actions"][t_ep][None], eps,
                                   np.asarray(u, np.float32).reshape(1, self.N), np.asarray(e, np.float32).reshape(self.N, self.A))
        return a[0], g[0]
