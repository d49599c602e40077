"""Recurrent Q-network fc1 -> ReLU -> GRUCell -> fc2 (reference: marl/modules/agents/drqn_agent.py:7-35).

Parameters are ordinary nn.Linear / nn.GRUCell parameters (same state_dict keys: fc1.*, gru.weight_ih, gru.weight_hh,
gru.bias_ih, gru.bias_hh, fc2.*) aliased onto one flat fp32 buffer; the arithmetic runs in libmal_b200's kernels.
"""
import torch as th
import torch.nn as nn

from ... import _native as nat
from ...flat import ensure_flat
from .. import autograd as ag
from .agent_network import AgentNetwork


class DRQNAgentNetwork(AgentNetwork):
    mal_kind = nat.AGENT_RNN

    def __init__(self, input_shape, args):
        super().__init__(input_shape, args)
        if args.rnn_hidden_dim != nat.HID:
            raise nat.MalError("the B200 kernels are built for rnn_hidden_dim == %d" % nat.HID)
        if args.n_actions > nat.MAX_ACTIONS:
            raise nat.MalError("n_actions must be <= %d" % nat.MAX_ACTIONS)
        dev = args.device
        self.fc1 = nn.Linear(input_shape, args.rnn_hidden_dim, device=dev)
        self.gru = nn.GRUCell(args.rnn_hidden_dim, args.rnn_hidden_dim, device=dev)
        self.fc2 = nn.Linear(args.rnn_hidden_dim, args.n_actions, device=dev)

    def flat_params(self):
        return ensure_flat(self)

    def init_hidden(self):
        return self.fc1.weight.new_zeros(1, self.args.rnn_hidden_dim)

    def forward(self, inputs, hidden_state):
        """inputs [rows, input_shape] (already assembled), hidden_state [..., 64] -> (q [rows, A], h' [rows, 64]).
        Records an autograd node under `args.autograd_forward` (modules/autograd.py); the learner differentiates through
        its own fused path, not through this call."""
        x = nat.require_cuda(inputs, "inputs")
        if ag.recording(self, x, hidden_state, *self.parameters()):
            ag._reject_input_grad(x, "agent input")
            x = x.detach().float().contiguous()
            h = hidden_state.reshape(-1, nat.HID)
            if h.shape[0] != x.shape[0]:
                h = h.expand(x.shape[0], nat.HID)
            h = h.float().contiguous()
            cfg = dict(rows=x.shape[0], N=1, OBS=self.input_shape, A=self.args.n_actions, dense_input=nat.STEP_DENSE,
                       obs_ptr=x.data_ptr(), obs_sb=x.stride(0), last_ptr=None, last_sb=0)
            with th.cuda.device(x.device):
                return ag.agent_step(self, cfg, x, None, h)
        if x.dtype != th.float32 or x.stride(-1) != 1:
            x = x.float().contiguous()
        rows = x.shape[0]
        h = hidden_state.reshape(-1, nat.HID)
        if h.shape[0] != rows or not h.is_contiguous():
            h = h.expand(rows, nat.HID).contiguous()
        flat = self.flat_params()
        q = th.empty(rows, self.args.n_actions, dtype=th.float32, device=x.device)
        h_out = th.empty(rows, nat.HID, dtype=th.float32, device=x.device)
        with th.cuda.device(x.device):
            nat.check(nat.lib().mal_agent_step(nat.ptr(flat), rows, 1, self.input_shape, self.args.n_actions, 1,
                                               nat.ptr(x), x.stride(0), None, 0, nat.ptr(h), nat.ptr(h_out),
                                               nat.ptr(q), None, nat.current_stream(x.device)), "mal_agent_step")
        return q, h_out
