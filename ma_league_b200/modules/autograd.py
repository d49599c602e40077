"""torch.autograd Functions over the module kernels, for callers that train through `BasicMAC.forward`, the agent networks
and the mixers (the reference's `q_learner.py:46-105` op sequence, a user's own loss) instead of `QLearner.train`.

Opt-in through `args.autograd_forward` (default False): only then, with grad mode on and an input or parameter that
requires grad, does a forward record a node.  The forward runs the same kernel launch as without the switch (outputs are
bit-identical); the backward is `mal_agent_step_backward` / `mal_mixer_backward` (VDN: d q_tot broadcast over agents).
Parameter gradients are views of one flat per-call buffer in state_dict order, which torch accumulates into `p.grad`.
Parameters, `h_in` and the batch views a forward read are saved for backward, so an in-place change of any of them
between forward and backward (an optimiser step, a write into the batch) raises torch's version error.
"""
from __future__ import annotations

import torch as th
from torch.autograd.function import once_differentiable

from .. import _native as nat
from ..flat import flat_views


def recording(switch_owner, *tensors) -> bool:
    """True when a forward of `switch_owner` (anything with `.args`, or a mixer carrying `autograd_forward`) records a node."""
    args = getattr(switch_owner, "args", None)
    on = getattr(args, "autograd_forward", False) if args is not None else getattr(switch_owner, "autograd_forward", False)
    if not on or not th.is_grad_enabled():
        return False
    return any(t is not None and t.requires_grad for t in tensors)


def _reject_input_grad(x, what):
    if x is not None and x.requires_grad:
        raise nat.MalError("%s requires grad: gradients with respect to agent inputs / states are not computed" % what)


def _param_grads(ctx, first, params, flat_grad):
    """Gradient tuple entries for `params` (input positions first..): views of flat_grad, None where none is needed."""
    if flat_grad is None:
        return (None,) * len(params)
    views = flat_views(flat_grad, params)
    return tuple(v if ctx.needs_input_grad[first + i] else None for i, v in enumerate(views))


class AgentStep(th.autograd.Function):
    """One step of the agent: (q [rows,A], h_out [rows,64]) for the recurrent agent, q for the feed-forward one.

    `cfg`: dict(kind, flat, rows, N, OBS, A, dense_input, obs_ptr, obs_sb, last_ptr, last_sb).  `obs` / `onehot` are the
    tensors behind obs_ptr / last_ptr (saved for the version check only; no gradient flows into them), `h_in` is None for
    the zero initial state."""

    @staticmethod
    def forward(ctx, cfg, obs, onehot, h_in, *params):
        rows, A = cfg["rows"], cfg["A"]
        dev = cfg["flat"].device
        rnn = cfg["kind"] == nat.AGENT_RNN
        q = th.empty(rows, A, dtype=th.float32, device=dev)
        h_out = th.empty(rows, nat.HID, dtype=th.float32, device=dev) if rnn else None
        with nat.on_device(dev):
            st = nat.current_stream(dev)
            if rnn:
                nat.check(nat.lib().mal_agent_step(
                    nat.ptr(cfg["flat"]), rows, cfg["N"], cfg["OBS"], A, cfg["dense_input"], cfg["obs_ptr"], cfg["obs_sb"],
                    cfg["last_ptr"], cfg["last_sb"], nat.ptr(h_in), nat.ptr(h_out), nat.ptr(q), None, st), "mal_agent_step")
            else:
                nat.check(nat.lib().mal_dqn_step(
                    nat.ptr(cfg["flat"]), rows, cfg["N"], cfg["OBS"], A, cfg["dense_input"], cfg["obs_ptr"], cfg["obs_sb"],
                    cfg["last_ptr"], cfg["last_sb"], nat.ptr(q), None, st), "mal_dqn_step")
        ctx.set_materialize_grads(False)
        ctx.cfg = cfg
        ctx.n_params = len(params)
        ctx.save_for_backward(obs, onehot, h_in, *params)
        return (q, h_out) if rnn else q

    @staticmethod
    @once_differentiable
    def backward(ctx, d_q, d_h_out=None):
        cfg = ctx.cfg
        obs, onehot, h_in, *params = ctx.saved_tensors     # version check of everything the forward read
        rows, A = cfg["rows"], cfg["A"]
        dev = cfg["flat"].device
        rnn = cfg["kind"] == nat.AGENT_RNN
        want_h = rnn and h_in is not None and ctx.needs_input_grad[3]
        want_p = any(ctx.needs_input_grad[4:])
        if not want_h and not want_p:
            return (None,) * (4 + ctx.n_params)
        d_q = d_q.reshape(rows, A).float().contiguous() if d_q is not None else None
        d_h_out = d_h_out.reshape(rows, nat.HID).float().contiguous() if (rnn and d_h_out is not None) else None
        lib = nat.lib()
        ws_bytes = lib.mal_agent_step_backward_workspace(cfg["kind"], rows, cfg["N"], cfg["OBS"], A, cfg["dense_input"])
        if ws_bytes < 0:
            raise nat.MalError("mal_agent_step_backward_workspace: " + lib.mal_last_error().decode())
        ws = th.empty(max(ws_bytes, 1), dtype=th.uint8, device=dev)
        d_h_in = th.empty(rows, nat.HID, dtype=th.float32, device=dev) if want_h else None
        d_flat = th.empty(cfg["flat"].numel(), dtype=th.float32, device=dev) if want_p else None
        with nat.on_device(dev):
            nat.check(lib.mal_agent_step_backward(
                cfg["kind"], nat.ptr(cfg["flat"]), rows, cfg["N"], cfg["OBS"], A, cfg["dense_input"], cfg["obs_ptr"],
                cfg["obs_sb"], cfg["last_ptr"], cfg["last_sb"], nat.ptr(h_in) if rnn else None, nat.ptr(d_q),
                nat.ptr(d_h_out), nat.ptr(d_h_in), nat.ptr(d_flat), nat.ptr(ws), nat.current_stream(dev)),
                "mal_agent_step_backward")
        return (None, None, None, d_h_in) + _param_grads(ctx, 4, params, d_flat)


def agent_step(agent, cfg, obs, onehot, h_in):
    """Record one agent step of `agent` (DRQNAgentNetwork / DQNAgentNetwork) on the kernel described by `cfg`."""
    params = list(agent.parameters())
    cfg = dict(cfg, kind=agent.mal_kind, flat=agent.flat_params())
    return AgentStep.apply(cfg, obs, onehot, h_in, *params)


class QMix(th.autograd.Function):
    """QMixer.forward: q [B,T,N] contiguous, states [B,T,S] (inner dim contiguous) -> q_tot [B,T,1]."""

    @staticmethod
    def forward(ctx, mixer, q, s, *params):
        B, T, N = q.shape
        E, HE = mixer.embed_dim, mixer.hypernet_embed
        ld = (2 * HE + 2 * E if mixer.hypernet_layers == 2 else 2 * E) + E * N + E
        scratch = th.empty(B * T * ld, dtype=th.float32, device=q.device)
        out = th.empty(B, T, 1, dtype=th.float32, device=q.device)
        flat = mixer.flat_params()
        with nat.on_device(q.device):
            nat.check(nat.lib().mal_mixer_forward(mixer.mal_kind, B, T, N, mixer.state_dim, E, HE, nat.ptr(flat), nat.ptr(q),
                                                  nat.ptr(s), s.stride(0), s.stride(1), nat.ptr(scratch), nat.ptr(out),
                                                  nat.current_stream(q.device)), "mal_mixer_forward")
        ctx.set_materialize_grads(False)
        ctx.meta = (mixer.mal_kind, mixer.state_dim, E, HE, flat)
        ctx.scratch = scratch                         # raw hypernet outputs of this call, read by the backward
        ctx.n_params = len(params)
        ctx.save_for_backward(q, s, *params)
        return out

    @staticmethod
    @once_differentiable
    def backward(ctx, g):
        q, s, *params = ctx.saved_tensors
        if g is None:
            return (None,) * (3 + ctx.n_params)
        kind, S, E, HE, flat = ctx.meta
        B, T, N = q.shape
        dev = q.device
        g = g.reshape(B * T).float().contiguous()
        lib = nat.lib()
        ws_bytes = lib.mal_mixer_backward_workspace(kind, B, T, N, S, E, HE)
        if ws_bytes < 0:
            raise nat.MalError("mal_mixer_backward_workspace: " + lib.mal_last_error().decode())
        ws = th.empty(ws_bytes, dtype=th.uint8, device=dev)
        d_q = th.empty(B, T, N, dtype=th.float32, device=dev)
        d_flat = th.empty(flat.numel(), dtype=th.float32, device=dev)
        with nat.on_device(dev):
            nat.check(lib.mal_mixer_backward(kind, B, T, N, S, E, HE, nat.ptr(flat), nat.ptr(q), nat.ptr(s), s.stride(0),
                                             s.stride(1), nat.ptr(ctx.scratch), nat.ptr(g), nat.ptr(d_q), nat.ptr(d_flat),
                                             nat.ptr(ws), nat.current_stream(dev)), "mal_mixer_backward")
        ctx.scratch = None
        return (None, d_q if ctx.needs_input_grad[1] else None, None) + _param_grads(ctx, 3, params, d_flat)


class VDN(th.autograd.Function):
    """VDNMixer.forward: q [B,T,N] contiguous -> q_tot [B,T,1]; the backward broadcasts d q_tot over the agents."""

    @staticmethod
    def forward(ctx, q):
        B, T, N = q.shape
        out = th.empty(B, T, 1, dtype=th.float32, device=q.device)
        with nat.on_device(q.device):
            nat.check(nat.lib().mal_mixer_forward(nat.MIXER_VDN, B, T, N, 0, 0, 0, None, nat.ptr(q), None, 0, 0, None,
                                                  nat.ptr(out), nat.current_stream(q.device)), "mal_mixer_forward")
        ctx.n = N
        return out

    @staticmethod
    @once_differentiable
    def backward(ctx, g):
        return g.expand(g.shape[0], g.shape[1], ctx.n)

