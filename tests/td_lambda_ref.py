"""Reference computations for TD(lambda) targets in the learner step (`args.td_lambda`), test infrastructure.

The lambda-return of the reference's `build_td_lambda_targets` (coma_learner.py:10-21), written over the learner's
[B,T] target array: tq[:, t] = target_q_tot of row t (the target mixer on state[:, t+1] and the masked target max at
t+1), which is the reference function's target_qs[:, t+1].

    R[b,T] = tq[b,T-1] (1 - sum_{t<T} term[b,t])
    R[b,t] = lambda gamma R[b,t+1] + m[b,t] (r[b,t] + (1 - lambda) gamma (1 - term[b,t]) tq[b,t])      t = T-1 .. 0
    targets = R[:, 0:T],  td = q_tot - targets

Everything else is QLearner.train unchanged: loss sum_b w_b sum (td m)^2 / sum m, seed 2 w_b td m^2 / sum m.

* `learner_forward_backward`: fp64 numpy, composed from the unchanged oracle (unroll, masked_target_max, qmix_forward /
  vdn_forward or none (IQL), agent_backward / qmix_backward; switched agent inputs through tests/input_layout_ref's
  embedding), with the recursion above; the keys of np_oracle.learner_forward_backward.
* `torch_loss_grads`: the reference learner's op sequence in torch with a restatement of build_td_lambda_targets, the
  targets detached, autograd in fp64 on CPU: the independent check of the above (tests/test_td_lambda.py).
"""
from __future__ import annotations

from collections import OrderedDict

import numpy as np
import torch as th

from oracle import np_oracle as O
from oracle import torch_port as TP
from tests import input_layout_ref as IL


def lambda_returns(tq, rewards, term, mask, gamma, td_lambda):
    """targets [B,T,Q] (fp64) from tq [B,T,Q] and rewards / term / mask [B,T,1] (broadcast over Q)."""
    tq = np.asarray(tq, dtype=np.float64)
    r, te, m = (np.asarray(x, dtype=np.float64) for x in (rewards, term, mask))
    B, T, Q = tq.shape
    R = np.zeros((B, T + 1, Q))
    R[:, T] = tq[:, T - 1] * (1.0 - te.sum(axis=1))
    for t in range(T - 1, -1, -1):
        R[:, t] = td_lambda * gamma * R[:, t + 1] + m[:, t] * (r[:, t] + (1.0 - td_lambda) * gamma * (1.0 - te[:, t]) * tq[:, t])
    return R[:, :T]


def learner_forward_backward(agent_p, target_agent_p, mixer_p, target_mixer_p, batch, *, mixer, double_q, gamma,
                             td_lambda, weights=None, dtype=np.float64, argmax_override=None, discrete=None,
                             last_action=True, agent_id=True):
    """QLearner.train up to loss.backward() with lambda-return targets.  mixer in {"qmix", "vdn", None}; ``weights`` [B]
    are prioritized replay's importance weights (None: unweighted).  ``argmax_override`` / ``discrete`` as in np_oracle.
    Statistics follow q_learner.py:117-124 over the mask expanded to the TD array (N times the mask for IQL)."""
    _, _, N, OBS = batch["obs"].shape
    A = batch["actions_onehot"].shape[-1]
    cols = IL.input_columns(OBS, A, N, last_action, agent_id)
    cast = lambda d: OrderedDict((k, v.astype(dtype)) for k, v in d.items()) if d is not None else None
    ap = cast(IL.embed_agent(agent_p, cols, OBS + A + N))
    tp = cast(IL.embed_agent(target_agent_p, cols, OBS + A + N))
    mp, tmp = cast(mixer_p), cast(target_mixer_p)
    obs = batch["obs"].astype(dtype)
    onehot = batch["actions_onehot"].astype(dtype)
    state = batch["state"].astype(dtype)
    rewards = batch["reward"][:, :-1].astype(dtype)
    actions = batch["actions"][:, :-1]
    mask, term = O.make_mask(batch["filled"], batch["terminated"])
    mask, term = mask.astype(dtype), term.astype(dtype)

    mac_out, caches = O.unroll(ap, obs, onehot)
    chosen = np.take_along_axis(mac_out[:, :-1], actions, axis=3)[..., 0]
    target_full, _ = O.unroll(tp, obs, onehot)
    tmax, amax = O.masked_target_max(mac_out, target_full, batch["avail_actions"], double_q, argmax_override)
    mc = None
    if mixer == "qmix":
        q_tot, mc = O.qmix_forward(mp, chosen, state[:, :-1])
        tq_tot, _ = O.qmix_forward(tmp, tmax, state[:, 1:])
    elif mixer == "vdn":
        q_tot, tq_tot = O.vdn_forward(chosen), O.vdn_forward(tmax)
    elif mixer is None:
        q_tot, tq_tot = chosen, tmax
    else:
        raise ValueError("Mixer {} not recognised.".format(mixer))

    targets = lambda_returns(tq_tot, rewards, term, mask, gamma, td_lambda).astype(dtype)
    td = q_tot - targets
    m = np.broadcast_to(mask, td.shape)
    mtd = td * m
    elems = m.sum(dtype=dtype)
    w = np.ones((td.shape[0], 1, 1), dtype=dtype) if weights is None else \
        np.asarray(weights, dtype=dtype).reshape(-1, 1, 1)
    loss = (w * mtd ** 2).sum(dtype=dtype) / elems
    g = 2.0 * w * mtd * m / elems

    if mixer == "qmix":
        mixer_grads, dchosen = O.qmix_backward(mp, mc, g, discrete)
        dchosen = dchosen.reshape(chosen.shape)
    elif mixer == "vdn":
        mixer_grads, dchosen = OrderedDict(), np.broadcast_to(g, chosen.shape).copy()
    else:
        mixer_grads, dchosen = OrderedDict(), g
    dmac = np.zeros_like(mac_out)
    np.put_along_axis(dmac[:, :-1], actions, dchosen[..., None], axis=3)
    agent_grads = O.agent_backward(ap, caches, dmac, (discrete or {}).get("x_mask"))
    agent_grads["fc1.weight"] = np.ascontiguousarray(agent_grads["fc1.weight"][:, cols])
    stats = dict(loss=loss, td_error_abs=np.abs(mtd).sum(dtype=dtype) / elems,
                 q_taken_mean=(q_tot * m).sum(dtype=dtype) / (elems * N),
                 target_mean=(targets * m).sum(dtype=dtype) / (elems * N),
                 mask_sum=elems, trained_steps=int(np.count_nonzero(m)))
    pre = dict(x=np.stack([c["x_pre"] for c in caches], axis=0))
    if mc is not None:
        pre.update(a1=mc["a1"], af=mc["af"], h1=mc["h1_pre"], hf=mc["hf_pre"], v1=mc["v1_pre"])
    return dict(pre=pre, mac_out=mac_out, target_mac_out=target_full, hout=np.stack([c["h"] for c in caches], axis=0),
                chosen=chosen, target_max=tmax, argmax=amax, q_tot=q_tot, target_q_tot=tq_tot, targets=targets, td=td,
                mask=mask, loss=loss, dq_tot=g, dchosen=dchosen, agent_grads=agent_grads, mixer_grads=mixer_grads,
                stats=stats)


# ---------------------------------------------------------------------------------------------- torch, autograd
def build_td_lambda_targets(rewards, terminated, mask, target_qs, n_agents, gamma, td_lambda):
    """coma_learner.py:10-21 restated: target_qs [B,T+1,Q] over every stored step, rewards / terminated / mask [B,T,1]."""
    ret = target_qs.new_zeros(*target_qs.shape)
    ret[:, -1] = target_qs[:, -1] * (1 - th.sum(terminated, dim=1))
    for t in range(ret.shape[1] - 2, -1, -1):
        ret[:, t] = td_lambda * gamma * ret[:, t + 1] + mask[:, t] * (
            rewards[:, t] + (1 - td_lambda) * gamma * target_qs[:, t + 1] * (1 - terminated[:, t]))
    return ret[:, 0:-1]


def torch_loss_grads(agent_p, target_agent_p, mixer_p, target_mixer_p, batch, *, mixer, double_q, gamma, td_lambda,
                     weights=None, last_action=True, agent_id=True):
    """The reference learner's loss with build_td_lambda_targets in torch (fp64, CPU, autograd).
    Returns (loss, agent grads, mixer grads, targets) as numpy."""
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
            q, h = IL.torch_agent_step(p, b, t, h, last_action, agent_id)
            outs.append(q)
        return th.stack(outs, dim=1)

    rewards, actions = b["reward"][:, :-1], b["actions"][:, :-1]
    terminated = b["terminated"][:, :-1].to(dt)
    mask = b["filled"][:, :-1].to(dt)
    mask[:, 1:] = mask[:, 1:] * (1 - terminated[:, :-1])
    avail = b["avail_actions"]
    mac_out = unroll(ap)
    chosen = th.gather(mac_out[:, :-1], dim=3, index=actions).squeeze(3)
    target_out = unroll(tp).detach()
    target_out[avail == 0] = -9999999
    if double_q:
        det = mac_out.clone().detach()
        det[avail == 0] = -9999999
        tmax = th.gather(target_out, 3, det.max(dim=3, keepdim=True)[1]).squeeze(3)     # every stored step
    else:
        tmax = target_out.max(dim=3)[0]
    if mixer == "qmix":
        q_tot, target_qs = TP.qmix(mp, chosen, b["state"][:, :-1]), TP.qmix(tmp, tmax, b["state"])
    elif mixer == "vdn":
        q_tot, target_qs = chosen.sum(dim=2, keepdim=True), tmax.sum(dim=2, keepdim=True)
    else:
        q_tot, target_qs = chosen, tmax
    targets = build_td_lambda_targets(rewards, terminated, mask, target_qs, N, gamma, td_lambda)
    masked = (q_tot - targets.detach()) * mask
    mask = mask.expand_as(masked)
    wt = th.ones(B, 1, 1, dtype=dt) if weights is None else th.tensor(np.asarray(weights, dtype=np.float64)).view(B, 1, 1)
    loss = (wt * masked ** 2).sum() / mask.sum()
    loss.backward()
    return (float(loss.detach()), OrderedDict((k, v.grad.numpy()) for k, v in ap.items()),
            OrderedDict((k, v.grad.numpy()) for k, v in mp.items()), targets.detach().numpy())
