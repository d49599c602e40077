"""Feed-forward Q-network fc1 -> ReLU -> fc2 (reference: marl/modules/agents/dqn_agent.py:9-37), registry key "dqn".

Same state_dict keys as the reference (fc1.weight, fc1.bias, fc2.weight, fc2.bias) on one flat fp32 buffer; the
arithmetic runs in libmal_b200 (`mal_dqn_step`; inside the learner the agent path is fc1 GEMM -> Q head with h := relu(fc1)).
The model has no hidden state; like the reference it "pretends otherwise for consistency" and passes the placeholder through.
"""
import torch as th
import torch.nn as nn

from ... import _native as nat
from ...flat import ensure_flat
from .. import autograd as ag
from .agent_network import AgentNetwork


class DQNAgentNetwork(AgentNetwork):
    mal_kind = nat.AGENT_DQN

    def __init__(self, input_shape, args):
        super().__init__(input_shape, args)
        if args.rnn_hidden_dim != nat.HID:
            raise nat.MalError("the B200 kernels are built for rnn_hidden_dim == %d" % nat.HID)
        if args.n_actions > nat.MAX_ACTIONS:
            raise nat.MalError("n_actions must be <= %d" % nat.MAX_ACTIONS)
        dev = args.device
        self.fc1 = nn.Linear(input_shape, args.rnn_hidden_dim, device=dev)
        self.fc2 = nn.Linear(args.rnn_hidden_dim, args.n_actions, device=dev)

    def flat_params(self):
        return ensure_flat(self)

    def init_hidden(self):
        # dqn_agent.py:27-32: "model has no hidden state, but we will pretend otherwise for consistency"
        return th.zeros(self.args.batch_size, 1, 1, device=self.args.device)

    def forward(self, inputs, hidden_states):
        """inputs [rows, input_shape] -> (q [rows, A], hidden_states unchanged).  Records an autograd node under
        `args.autograd_forward` (modules/autograd.py)."""
        x = nat.require_cuda(inputs, "inputs")
        if ag.recording(self, x, *self.parameters()):
            ag._reject_input_grad(x, "agent input")
            x = x.detach().float().contiguous()
            cfg = dict(rows=x.shape[0], N=1, OBS=self.input_shape, A=self.args.n_actions, dense_input=nat.STEP_DENSE,
                       obs_ptr=x.data_ptr(), obs_sb=x.stride(0), last_ptr=None, last_sb=0)
            with th.cuda.device(x.device):
                return ag.agent_step(self, cfg, x, None, None), hidden_states
        if x.dtype != th.float32 or x.stride(-1) != 1:
            x = x.float().contiguous()
        rows = x.shape[0]
        flat = self.flat_params()
        q = th.empty(rows, self.args.n_actions, dtype=th.float32, device=x.device)
        with th.cuda.device(x.device):
            nat.check(nat.lib().mal_dqn_step(nat.ptr(flat), rows, 1, self.input_shape, self.args.n_actions, 1, nat.ptr(x),
                                             x.stride(0), None, 0, nat.ptr(q), None, nat.current_stream(x.device)),
                      "mal_dqn_step")
        return q, hidden_states
