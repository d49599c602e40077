"""The reference learner's op sequence over callables (test infrastructure).

`reference_loss` restates `QLearner.train` of marl/learners/q_learner.py:36-105 up to `loss.backward()`: a loop of
`mac.forward`, the chosen-action gather, the masked (double-Q) target max, the mixer, the TD loss.  It takes the agent /
mixer calls as callables, so the same code drives torch_port's functions in fp64 on the CPU (pinned against the fp64
oracle) and BasicMAC + QMixer / VDNMixer with `args.autograd_forward` on the GPU.
"""
from __future__ import annotations

import torch as th

NEG_MASK = -9999999.0   # q_learner.py:68,73


def reference_loss(batch, mac_forward, target_forward, mixer=None, target_mixer=None, *, double_q, gamma):
    """batch: dict of tensors with the scheme's keys over TT stored steps.  mac_forward(t) / target_forward(t) -> [B,N,A]
    (hidden states are the callables' business, like mac.init_hidden + mac.forward); mixer(qs [B,T,N], states [B,T,S])
    -> [B,T,1] or None for independent learners.  Returns (loss, dict of intermediates)."""
    rewards = batch["reward"][:, :-1]
    actions = batch["actions"][:, :-1]
    terminated = batch["terminated"][:, :-1].to(rewards.dtype)
    mask = batch["filled"][:, :-1].to(rewards.dtype)
    mask[:, 1:] = mask[:, 1:] * (1 - terminated[:, :-1])
    avail_actions = batch["avail_actions"]
    TT = batch["obs"].shape[1]

    mac_out = th.stack([mac_forward(t) for t in range(TT)], dim=1)                          # :46-52
    chosen_action_qvals = th.gather(mac_out[:, :-1], dim=3, index=actions).squeeze(3)       # :55
    target_mac_out = th.stack([target_forward(t) for t in range(TT)], dim=1)[:, 1:]         # :58-65
    target_mac_out[avail_actions[:, 1:] == 0] = NEG_MASK                                    # :68
    if double_q:                                                                            # :71-75
        mac_out_detach = mac_out.clone().detach()
        mac_out_detach[avail_actions == 0] = NEG_MASK
        cur_max_actions = mac_out_detach[:, 1:].max(dim=3, keepdim=True)[1]
        target_max_qvals = th.gather(target_mac_out, 3, cur_max_actions).squeeze(3)
    else:
        target_max_qvals = target_mac_out.max(dim=3)[0]                                     # :77
    if mixer is not None:                                                                   # :81-83
        chosen_action_qvals = mixer(chosen_action_qvals, batch["state"][:, :-1])
        target_max_qvals = target_mixer(target_max_qvals, batch["state"][:, 1:])
    targets = rewards + gamma * (1 - terminated) * target_max_qvals                          # :86
    td_error = chosen_action_qvals - targets.detach()                                       # :89
    mask = mask.expand_as(td_error)                                                         # :92
    masked_td_error = td_error * mask                                                       # :95
    loss = (masked_td_error ** 2).sum() / mask.sum()                                        # :98
    return loss, dict(mac_out=mac_out, chosen=chosen_action_qvals, targets=targets, td=td_error, mask=mask)
