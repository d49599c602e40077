"""Reference computations for independent Q-learners (`mixer: None`), test infrastructure.

IQL is `QLearner.train` (q_learner.py:34-125) with self.mixer = None: the mixing lines (:81-83) are skipped, so
`chosen_action_qvals` [B,T,N] and `target_max_qvals` [B,T,N] meet the [B,T,1] reward directly, every agent has its
own TD error and the mask is expanded to [B,T,N] (:92).  Both functions are built from the unchanged shared modules:

* `learner_forward_backward`: the fp64 numpy reference, np_oracle's unroll / masked target max / td_loss /
  agent_backward without a mixer in between (hand-derived backward, no autograd).  Switched agent inputs go through the
  embedded layout of tests/input_layout_ref.py.
* `torch_port_train`: torch_port's ATen sequence (per-timestep unroll, gather, masked max, autograd backward,
  clip_grad_norm_, stock RMSprop) without the mixer, with the optimiser over the agent's parameters.

The torch port's autograd is the independent check of the hand-derived reference (tests/test_iql.py).
"""
from __future__ import annotations

from collections import OrderedDict

import numpy as np
import torch as th

from oracle import np_oracle as O
from oracle import torch_port as TP
from tests import input_layout_ref as IL


def learner_forward_backward(agent_p, target_agent_p, batch, *, double_q, gamma, dtype=np.float64,
                             argmax_override=None, discrete=None, last_action=True, agent_id=True):
    """Everything QLearner.train computes up to loss.backward() for IQL; the keys of np_oracle.learner_forward_backward.
    q_tot / target_q_tot are chosen / target_max ([B,T,N]); the statistics follow q_learner.py:117-124 literally on the
    expanded mask: mask_elems = N * mask.sum(), and N enters q_taken_mean / target_mean a second time through the
    `mask_elems * n_agents` denominator.  ``argmax_override`` / ``discrete`` as in np_oracle (only ``x_mask`` applies)."""
    _, _, N, OBS = batch["obs"].shape
    A = batch["actions_onehot"].shape[-1]
    cols = IL.input_columns(OBS, A, N, last_action, agent_id)
    cast = lambda d: OrderedDict((k, v.astype(dtype)) for k, v in d.items())
    ap = cast(IL.embed_agent(agent_p, cols, OBS + A + N))
    tp = cast(IL.embed_agent(target_agent_p, cols, OBS + A + N))
    obs = batch["obs"].astype(dtype)
    onehot = batch["actions_onehot"].astype(dtype)
    rewards = batch["reward"][:, :-1].astype(dtype)
    actions = batch["actions"][:, :-1]
    mask, term = O.make_mask(batch["filled"], batch["terminated"])
    mask, term = mask.astype(dtype), term.astype(dtype)

    mac_out, caches = O.unroll(ap, obs, onehot)
    chosen = np.take_along_axis(mac_out[:, :-1], actions, axis=3)[..., 0]                   # :55
    target_full, _ = O.unroll(tp, obs, onehot)
    tmax, amax = O.masked_target_max(mac_out, target_full, batch["avail_actions"], double_q, argmax_override)
    loss, td, mtd, targets, g = O.td_loss(chosen, tmax, rewards, term, mask, gamma)          # :86-98, no mixer
    dmac = np.zeros_like(mac_out)
    np.put_along_axis(dmac[:, :-1], actions, g[..., None], axis=3)
    agent_grads = O.agent_backward(ap, caches, dmac, (discrete or {}).get("x_mask"))
    agent_grads["fc1.weight"] = np.ascontiguousarray(agent_grads["fc1.weight"][:, cols])
    m = np.broadcast_to(mask, td.shape)
    elems = m.sum(dtype=dtype)
    stats = dict(loss=loss, td_error_abs=np.abs(mtd).sum(dtype=dtype) / elems,
                 q_taken_mean=(chosen * m).sum(dtype=dtype) / (elems * N),
                 target_mean=(targets * m).sum(dtype=dtype) / (elems * N),
                 mask_sum=elems, trained_steps=int(np.count_nonzero(m)))
    return dict(pre=dict(x=np.stack([c["x_pre"] for c in caches], axis=0)), mac_out=mac_out,
                target_mac_out=target_full, hout=np.stack([c["h"] for c in caches], axis=0), chosen=chosen,
                target_max=tmax, argmax=amax, q_tot=chosen, target_q_tot=tmax, targets=targets, td=td, mask=mask,
                loss=loss, dq_tot=g, dchosen=g, agent_grads=agent_grads, mixer_grads=OrderedDict(), stats=stats)


def torch_port_train(agent_p, target_agent_p, batch, *, double_q, gamma, lr, alpha, eps, clip):
    """One IQL step in torch_port's op sequence (fp32, CPU).  Returns the loss, the clipped gradients, the parameters
    after RMSprop, the optimiser, and the statistics of :112-124 computed literally on the port's tensors."""
    ap, tp = TP.to_params(agent_p), TP.to_params(target_agent_p)
    params = list(ap.values())
    opt = th.optim.RMSprop(params, lr=lr, alpha=alpha, eps=eps)
    rewards = batch["reward"][:, :-1]
    actions = batch["actions"][:, :-1]
    terminated = batch["terminated"][:, :-1].float()
    mask = batch["filled"][:, :-1].float()
    mask[:, 1:] = mask[:, 1:] * (1 - terminated[:, :-1])
    avail = batch["avail_actions"]
    mac_out = TP.unroll(ap, batch)
    chosen = th.gather(mac_out[:, :-1], dim=3, index=actions).squeeze(3)
    target_out = TP.unroll(tp, batch)[:, 1:]
    target_out[avail[:, 1:] == 0] = -9999999
    if double_q:
        det = mac_out.clone().detach()
        det[avail == 0] = -9999999
        tmax = th.gather(target_out, 3, det[:, 1:].max(dim=3, keepdim=True)[1]).squeeze(3)
    else:
        tmax = target_out.max(dim=3)[0]
    targets = rewards + gamma * (1 - terminated) * tmax            # [B,T,1] + [B,T,N]: one target per agent
    td = chosen - targets.detach()
    mask = mask.expand_as(td)
    masked = td * mask
    loss = (masked ** 2).sum() / mask.sum()
    opt.zero_grad()
    loss.backward()
    grad_norm = th.nn.utils.clip_grad_norm_(params, clip)
    grads = OrderedDict((k, p.grad.detach().clone()) for k, p in ap.items())
    opt.step()
    N = chosen.shape[2]
    mask_elems = mask.sum().item()
    stats = dict(td_error_abs=masked.abs().sum().item() / mask_elems,
                 q_taken_mean=(chosen * mask).sum().item() / (mask_elems * N),
                 target_mean=(targets * mask).sum().item() / (mask_elems * N),
                 mask_sum=mask_elems, trained_steps=int(th.count_nonzero(mask).item()))
    return dict(loss=float(loss.item()), grad_norm=float(grad_norm), grads=grads, params=ap, opt=opt, stats=stats)
