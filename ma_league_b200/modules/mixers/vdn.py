"""VDN mixer: q_tot = sum over agents (reference: marl/modules/mixers/vdn.py:5-10)."""
import torch as th
import torch.nn as nn

from ... import _native as nat
from .. import autograd as ag


class VDNMixer(nn.Module):
    def __init__(self, args=None):
        super().__init__()
        self.args = args          # only `autograd_forward` is read (the reference's VDNMixer takes no arguments)

    def forward(self, agent_qs, batch):
        if ag.recording(self, agent_qs):
            return ag.VDN.apply(nat.require_cuda(agent_qs, "agent_qs").float().contiguous())
        q = nat.require_cuda(agent_qs, "agent_qs")
        B, T, N = q.shape
        q = q.float().contiguous()
        out = th.empty(B, T, 1, dtype=th.float32, device=q.device)
        with th.cuda.device(q.device):
            nat.check(nat.lib().mal_mixer_forward(nat.MIXER_VDN, B, T, N, 0, 0, 0, None, nat.ptr(q), None, 0, 0, None,
                                                  nat.ptr(out), nat.current_stream(q.device)), "mal_mixer_forward")
        return out
