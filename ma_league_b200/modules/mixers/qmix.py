"""QMIX monotonic mixing network (reference: marl/modules/mixers/qmix.py:7-59).

Same constructor arguments and state_dict keys (hyper_w_1.{0,2}.*, hyper_w_final.{0,2}.*, hyper_b_1.*, V.{0,2}.*, or the
single-Linear hypernets when hypernet_layers == 1); parameters alias one flat fp32 buffer read by the kernels.
"""
import numpy as np
import torch as th
import torch.nn as nn

from ... import _native as nat
from ...flat import ensure_flat
from .. import autograd as ag


class QMixer(nn.Module):
    def __init__(self, args):
        super().__init__()
        self.args = args
        self.n_agents = args.n_agents
        self.state_dim = int(np.prod(args.state_shape))
        self.embed_dim = args.mixing_embed_dim
        if self.embed_dim > nat.MAX_EMBED:
            raise nat.MalError("mixing_embed_dim must be <= %d" % nat.MAX_EMBED)
        dev = args.device
        layers = getattr(args, "hypernet_layers", 1)
        if layers == 1:
            self.hyper_w_1 = nn.Linear(self.state_dim, self.embed_dim * self.n_agents, device=dev)
            self.hyper_w_final = nn.Linear(self.state_dim, self.embed_dim, device=dev)
            self.hypernet_embed = 0
        elif layers == 2:
            he = args.hypernet_embed
            self.hypernet_embed = he
            self.hyper_w_1 = nn.Sequential(nn.Linear(self.state_dim, he, device=dev), nn.ReLU(),
                                           nn.Linear(he, self.embed_dim * self.n_agents, device=dev))
            self.hyper_w_final = nn.Sequential(nn.Linear(self.state_dim, he, device=dev), nn.ReLU(),
                                               nn.Linear(he, self.embed_dim, device=dev))
        elif layers > 2:
            raise Exception("Sorry >2 hypernet layers is not implemented!")
        else:
            raise Exception("Error setting number of hypernet layers.")
        self.hypernet_layers = layers
        self.hyper_b_1 = nn.Linear(self.state_dim, self.embed_dim, device=dev)
        self.V = nn.Sequential(nn.Linear(self.state_dim, self.embed_dim, device=dev), nn.ReLU(),
                               nn.Linear(self.embed_dim, 1, device=dev))

    @property
    def mal_kind(self):
        return nat.MIXER_QMIX2 if self.hypernet_layers == 2 else nat.MIXER_QMIX1

    def flat_params(self):
        return ensure_flat(self)

    def forward(self, agent_qs, states):
        """agent_qs [B,T,N], states [B,T,S] -> q_tot [B,T,1].  Records an autograd node under `args.autograd_forward`
        (modules/autograd.py); the learner uses its fused path."""
        if ag.recording(self, agent_qs, states, *self.parameters()):
            ag._reject_input_grad(states, "states")
            q = nat.require_cuda(agent_qs, "agent_qs").float().contiguous()
            s = states if (states.dtype == th.float32 and states.stride(-1) == 1) else states.float().contiguous()
            return ag.QMix.apply(self, q, s, *self.parameters())
        q = nat.require_cuda(agent_qs, "agent_qs").float().contiguous()
        B, T, N = q.shape
        s = states
        if s.dtype != th.float32 or s.stride(-1) != 1:
            s = s.float().contiguous()
        E, HE = self.embed_dim, self.hypernet_embed
        ld = (2 * HE + 2 * E if self.hypernet_layers == 2 else 2 * E) + E * N + E
        scratch = th.empty(B * T * ld, dtype=th.float32, device=q.device)
        out = th.empty(B, T, 1, dtype=th.float32, device=q.device)
        flat = self.flat_params()
        with th.cuda.device(q.device):
            nat.check(nat.lib().mal_mixer_forward(self.mal_kind, B, T, N, self.state_dim, E, HE, nat.ptr(flat),
                                                  nat.ptr(q), nat.ptr(s), s.stride(0), s.stride(1), nat.ptr(scratch),
                                                  nat.ptr(out), nat.current_stream(q.device)), "mal_mixer_forward")
        return out
