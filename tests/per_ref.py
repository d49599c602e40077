"""Reference computations for prioritized episode replay (proportional PER over episodes), test infrastructure.

* `sample`: stratified draws from the fp64 prefix sums of the fp32 priorities, given the uniforms, and the importance
  weights w_j = (p_min / p_{id_j})^beta.
* `update`: new priorities (sum |td*m| / sum m + eps)^alpha of the sampled slots, the highest batch index winning for a
  slot drawn twice, and the running maximum over the written priorities.
* `weighted_learner`: the importance-weighted loss and gradient from the unchanged oracle.  Episodes are independent
  through forward and backward, and the normaliser is the global sum of the mask, so
  grad = sum_b w_b * (sum_t m_b / sum m) * oracle_grad(episode b alone), and likewise for the loss.
* `torch_weighted`: torch_port's op sequence with the weighted loss, autograd in fp64 (the independent check of the above).
"""
from __future__ import annotations

from collections import OrderedDict

import numpy as np
import torch as th

from oracle import np_oracle as O
from oracle import torch_port as TP
from tests import iql_ref as IQ
from tests import input_layout_ref as IL

NEAR = 1e-6


def sample(p, n, u, beta):
    """(ids int64 [B], weights fp64 [B], near bool [B]) for priorities p (fp32, >= n entries) and uniforms u [B].
    `near` flags draws whose point lies within NEAR * total of a prefix-sum boundary (their slot may legitimately differ)."""
    p = np.asarray(p, dtype=np.float32)[:n].astype(np.float64)
    u = np.asarray(u, dtype=np.float32).astype(np.float64)
    B = u.shape[0]
    cum = np.cumsum(p)
    total = cum[-1]
    x = (np.arange(B, dtype=np.float64) + u) * total / B
    ids = np.searchsorted(cum, x, side="right")                    # first slot whose inclusive prefix exceeds x
    pos = np.nonzero(p > 0)[0]
    last = pos[-1] if pos.size else n - 1
    ids = np.where(ids >= n, last, ids).astype(np.int64)
    dist = np.min(np.abs(cum[None, :] - x[:, None]), axis=1) if n <= 20000 else \
        np.minimum(np.abs(cum[np.clip(ids, 0, n - 1)] - x), np.abs(cum[np.clip(ids - 1, 0, n - 1)] - x))
    near = dist <= NEAR * max(total, 1e-300)
    pmin = p.min()
    pid = p[ids]
    w = np.where(pid > 0, (pmin / np.where(pid > 0, pid, 1.0)) ** beta, 1.0)
    return ids, w, near


def update(p, maxp, ids, td, mask, alpha, eps):
    """(new priorities fp64, new running maximum) after one step.  td [B,T,Q], mask [B,T]."""
    p = np.asarray(p, dtype=np.float64).copy()
    td = np.asarray(td, dtype=np.float64)
    m = np.asarray(mask, dtype=np.float64).reshape(td.shape[0], td.shape[1], 1)
    num = np.abs(td * m).sum(axis=(1, 2))
    den = np.broadcast_to(m, td.shape).sum(axis=(1, 2))
    new = (np.where(den > 0, num / np.where(den > 0, den, 1.0), 0.0) + eps) ** alpha
    written = {}
    for b, i in enumerate(np.asarray(ids)):          # ascending batch index: the last occurrence wins
        written[int(i)] = new[b]
    for i, v in written.items():
        p[i] = v
    return p, max([float(maxp)] + list(written.values()))


def _episode(batch, b):
    return {k: v[b:b + 1] for k, v in batch.items()}


def weighted_learner(agent_p, tagent_p, mixer_p, tmixer_p, batch, w, *, mixer, double_q, gamma, last_action=True,
                     agent_id=True):
    """(weighted loss, agent grads, mixer grads) in fp64, from the oracle run on one episode at a time."""
    mask, _ = O.make_mask(batch["filled"], batch["terminated"])
    msum = mask.reshape(mask.shape[0], -1).sum(axis=1).astype(np.float64)
    total = msum.sum()
    loss, ag, mg = 0.0, None, None
    for b in range(batch["obs"].shape[0]):
        if msum[b] == 0:
            continue
        eb = _episode(batch, b)
        if mixer is None:
            r = IQ.learner_forward_backward(agent_p, tagent_p, eb, double_q=double_q, gamma=gamma, dtype=np.float64,
                                            last_action=last_action, agent_id=agent_id)
        else:
            r = IL.learner_forward_backward(agent_p, tagent_p, mixer_p, tmixer_p, eb, mixer=mixer, double_q=double_q,
                                            gamma=gamma, dtype=np.float64, last_action=last_action, agent_id=agent_id)
        f = float(w[b]) * msum[b] / total
        loss += f * float(r["loss"])
        ag = OrderedDict((k, f * v) for k, v in r["agent_grads"].items()) if ag is None else \
            OrderedDict((k, ag[k] + f * v) for k, v in r["agent_grads"].items())
        mg = OrderedDict((k, f * v) for k, v in r["mixer_grads"].items()) if mg is None else \
            OrderedDict((k, mg[k] + f * v) for k, v in r["mixer_grads"].items())
    return loss, ag, mg


def torch_weighted(agent_p, tagent_p, mixer_p, tmixer_p, batch, w, *, mixer, double_q, gamma, last_action=True,
                   agent_id=True):
    """The weighted loss sum_b w_b sum (td*m)^2 / sum m in torch_port's op sequence, autograd in fp64 on CPU."""
    dt = th.float64
    ap = OrderedDict((k, th.tensor(v, dtype=dt, requires_grad=True)) for k, v in agent_p.items())
    tp = OrderedDict((k, th.tensor(v, dtype=dt)) for k, v in tagent_p.items())
    mp = OrderedDict((k, th.tensor(v, dtype=dt, requires_grad=True)) for k, v in (mixer_p or {}).items())
    tmp = OrderedDict((k, th.tensor(v, dtype=dt)) for k, v in (tmixer_p or {}).items())
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
    elif mixer == "vdn":
        q_tot, tq_tot = chosen.sum(dim=2, keepdim=True), tmax.sum(dim=2, keepdim=True)
    else:
        q_tot, tq_tot = chosen, tmax
    targets = rewards + gamma * (1 - terminated) * tq_tot
    masked = (q_tot - targets.detach()) * mask
    mask = mask.expand_as(masked)
    wt = th.tensor(np.asarray(w, dtype=np.float64)).view(B, 1, 1)
    loss = (wt * masked ** 2).sum() / mask.sum()
    loss.backward()
    return (float(loss.detach()), OrderedDict((k, v.grad.numpy()) for k, v in ap.items()),
            OrderedDict((k, v.grad.numpy()) for k, v in mp.items()))
