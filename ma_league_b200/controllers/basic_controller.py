"""Shared-parameter multi-agent controller with the reference's API (marl/controllers/basic_controller.py:12-101).

`select_actions` is ONE kernel launch (input assembly + fc1 + GRU step + fc2 + avail mask + epsilon-greedy with
Philox), `forward` the same kernel without the selection tail.  The reference's hooks (`_build_inputs`,
`_compute_agent_outputs`, `_build_agent`, `_get_input_shape`) are kept: a subclass that overrides the first two is
served through them (dense-input kernel) instead of the fused path.

`set_match_policies(table, ids)` makes match b of the batch play row ids[b] of a [K, P] table of flat agent buffers
(league opponents, cross-play pairings) instead of the controller's own agent: still one launch per step.
"""
from __future__ import annotations

import contextlib
import ctypes as C

import torch as th

from .. import _native as nat
from ..components.action_selectors import make_select_struct
from ..exceptions import HiddenStateNotInitialized
from ..flat import ensure_flat
from ..modules import autograd as ag
from ..modules.agents import REGISTRY as agent_REGISTRY
from ..modules.agents.drqn_agent import DRQNAgentNetwork
from ..modules.agents.dqn_agent import DQNAgentNetwork
from .multi_agent_controller import MultiAgentController


class BasicMAC(MultiAgentController):
    def __init__(self, scheme, groups, args):
        super().__init__(scheme, groups, args)
        self._obs_dim = scheme["obs"]["vshape"] if isinstance(scheme["obs"]["vshape"], int) else scheme["obs"]["vshape"][0]
        self._pool = None           # set_match_policies: (table, ids on the device, schedule buffer)

    # ------------------------------------------------------------------ per-match policies
    def set_match_policies(self, table, ids=None):
        """Make match b play with the agent in row `ids[b]` of `table` instead of `self.agent`; `set_match_policies(None)`
        goes back to the controller's own agent.

        `table` is a [K, P] float32 CUDA tensor whose rows are flat agent buffers in state_dict order (e.g.
        `DeviceAgentPool.pool`, rows of `agent.flat_params()`), P = this agent's parameter count; `ids` holds one policy
        per match (a sequence, CPU or CUDA tensor).  The ids are checked and bucketed by policy here, once per assignment
        (one launch); the table itself is read at every step and never copied, so a `pool.sync()` (or any in-place write
        to the table) between steps takes effect at the next step.  While policies are set, `select_actions`,
        `rollout_step` and `forward` run the pooled kernels (still one launch per step), `init_hidden` must be called with
        `len(ids)` matches, and nothing records an autograd node: the pooled path reads no parameter of `self.agent`.
        Recurrent agent only."""
        if table is None:
            self._pool = None
            return
        if not isinstance(table, th.Tensor) or not table.is_cuda:
            raise nat.MalError("the policy table must be a CUDA tensor: the B200 path has no CPU fallback")
        if not self._rollout_fusable():
            raise nat.MalError("per-match policies need the fused recurrent agent path (not the dqn agent or a subclass "
                               "that overrides the input hooks)")
        if getattr(self, "ensemble", None):
            raise nat.MalError("per-match policies do not run ensemble agents")
        if table.dim() != 2 or table.dtype != th.float32 or table.stride(1) != 1:
            raise nat.MalError("the policy table must be a [K, P] float32 tensor with contiguous rows")
        n_params = ensure_flat(self.agent).numel()
        if table.shape[1] != n_params:
            raise ValueError("agent architectures differ: %d vs %d parameters" % (table.shape[1], n_params))
        K = table.shape[0]
        if not 1 <= K <= nat.MAX_POLICIES:
            raise ValueError("the policy table must have between 1 and %d rows, got %d" % (nat.MAX_POLICIES, K))
        ids = th.as_tensor(ids).reshape(-1)
        if ids.numel() == 0 or ids.is_floating_point() or ids.dtype == th.bool:
            raise ValueError("ids must hold one integer policy per match")
        if int(ids.min()) < 0 or int(ids.max()) >= K:
            raise ValueError("policy ids must be in [0, %d)" % K)
        dev = table.device
        bs = ids.numel()
        ids_dev = ids.to(device=dev, dtype=th.int32)
        lib = nat.lib()
        nbytes = lib.mal_policy_schedule_bytes(bs, self.n_agents, K)
        if nbytes < 0:
            raise nat.MalError(lib.mal_last_error().decode())
        sched = th.empty((nbytes + 3) // 4, dtype=th.int32, device=dev)
        with nat.on_device(dev):
            nat.check(lib.mal_policy_schedule(ids_dev.data_ptr(), bs, self.n_agents, K, sched.data_ptr(), None,
                                              nat.current_stream(dev)), "mal_policy_schedule")
        self._pool = (table, ids_dev, sched)

    @property
    def match_policies(self):
        """The per-match policy ids set by `set_match_policies` (int32 device tensor), or None."""
        return None if self._pool is None else self._pool[1]

    def _pool_args(self, dev, B):
        """(table ptr, table_ld, K, schedule ptr) of the pooled launches for a batch of B matches on `dev`."""
        table, ids, sched = self._pool
        if table.device != dev:
            raise nat.MalError("the policy table lives on %s, the batch on %s" % (table.device, dev))
        if B != ids.numel():
            raise nat.MalError("per-match policies were set for %d matches, the batch has %d" % (ids.numel(), B))
        return table.data_ptr(), table.stride(0), table.shape[0], sched.data_ptr()

    # ------------------------------------------------------------------ public API
    def select_actions(self, ep_batch, t_ep, t_env, bs=slice(None), test_mode=False, u=None, e=None):
        if self._fusable() and isinstance(bs, slice) and bs == slice(None):
            sel = self.action_selector
            eps = sel._epsilon(t_env, test_mode)
            avail_actions = ep_batch["avail_actions"][:, t_ep]
            B = ep_batch.batch_size
            dev = avail_actions.device
            out = th.empty(2, B, self.n_agents, dtype=th.long, device=dev)     # actions | greedy, one allocation
            status = th.zeros(1, dtype=th.int32, device=dev) if sel.validate else None
            s, keep = make_select_struct(avail_actions, eps, out[0], out[1], status, u, e)
            self._step(ep_batch, t_ep, s)
            if status is not None and int(status.item()) != 0:
                raise ValueError("Expected at least one available action per agent (Categorical probs are all zero)")
            return out[0], out[1]
        avail_actions = ep_batch["avail_actions"][:, t_ep]
        with self._no_recording():    # acting never records an autograd node, whatever args.autograd_forward says
            agent_outs = self.forward(ep_batch, t_ep, test_mode=test_mode)
        return self.action_selector.select(agent_outs[bs], avail_actions[bs], t_env, test_mode, u=u, e=e)

    def rollout_step(self, ep_batch, t_ep, t_env, pre, prev=None, alive=None, test_mode=False, u=None, e=None):
        """One timestep of the rollout loop around `select_actions` in ONE launch (steppers/episode_stepper.py:110-142,
        177-186): `ep_batch.update(pre, ts=t_ep)` (state / avail_actions / obs from the environment, device tensors
        [bs, ...]), `ep_batch.update({"reward", "terminated"}, ts=t_ep-1)` for `prev = (reward [bs] f32, done [bs] bool)`,
        `select_actions(ep_batch, t_ep, t_env)` and `ep_batch.update({"actions": ...}, ts=t_ep)` incl. the one-hot.
        `alive` [bs] bool: matches that have ended select on a dummy avail row.  Returns (actions, is_greedy) like
        `select_actions`.  Needs a packed device batch and the fused agent (`_fusable()`); callers fall back to the
        separate calls otherwise."""
        if not self._rollout_fusable():
            raise nat.MalError("rollout_step needs the fused recurrent agent path")
        if self.hidden_states is None:
            raise HiddenStateNotInitialized()
        tv = ep_batch.data.transition_data
        obs_all = nat.require_cuda(tv["obs"], "ep_batch")
        B, TT, N, OBS = obs_all.shape
        A = self.n_actions
        dev = obs_all.device
        state, avail, obs = pre["state"], pre["avail_actions"], pre["obs"]
        if state.dtype != th.float32 or obs.dtype != th.float32 or avail.dtype != th.int32:
            raise nat.MalError("pre-transition data must be float32 state / obs and int32 avail_actions")
        if state.stride(-1) != 1 or not obs[0].is_contiguous() or not avail[0].is_contiguous():
            raise nat.MalError("pre-transition rows must be contiguous")
        sel = self.action_selector
        eps = sel._epsilon(t_env, test_mode)
        out = th.empty(2, B, N, dtype=th.long, device=dev)                       # actions | greedy
        status = th.zeros(1, dtype=th.int32, device=dev) if sel.validate else None
        s, keep = make_select_struct(avail, eps, out[0], out[1], status, u, e)
        io = nat.RolloutIO()
        io.agent_input = self._input_flags()
        io.state_dim = state.shape[-1]
        io.env_state, io.env_state_sb = state.data_ptr(), state.stride(0)
        io.env_avail, io.env_avail_sb = avail.data_ptr(), avail.stride(0)
        io.env_obs, io.env_obs_sb = obs.data_ptr(), obs.stride(0)
        if alive is not None:
            alive = alive if alive.dtype == th.bool else alive != 0
            io.alive = alive.data_ptr()
        fld = {}
        for key in ("state", "avail_actions", "obs", "filled", "actions", "actions_onehot", "reward", "terminated"):
            v = tv[key]
            fld[key] = (v.data_ptr(), v.element_size(), v.stride(0), v.stride(1))

        def at(key, t):
            p, es, sb, st = fld[key]
            return p + es * st * t, sb
        io.state_t, io.state_sb = at("state", t_ep)
        io.avail_t, io.avail_sb = at("avail_actions", t_ep)
        io.obs_t, io.obs_sb = at("obs", t_ep)
        io.filled_t, io.filled_sb = at("filled", t_ep)
        io.actions_t, io.actions_sb = at("actions", t_ep)
        io.onehot_t, io.onehot_sb = at("actions_onehot", t_ep)
        if t_ep > 0:
            io.onehot_tm1, io.onehot_tm1_sb = at("actions_onehot", t_ep - 1)
        if prev is not None:
            if t_ep == 0:
                raise nat.MalError("there is no previous step at t_ep = 0")
            reward, done = prev
            reward = reward if reward.dtype == th.float32 else reward.float()
            done = done if done.dtype == th.bool else done != 0
            io.prev_reward, io.prev_done = reward.data_ptr(), done.data_ptr()
            io.reward_tm1, io.reward_sb = at("reward", t_ep - 1)
            io.term_tm1, io.term_sb = at("terminated", t_ep - 1)
            keep += [reward, done]
        rows = B * N
        h_in = self.hidden_states
        if h_in.dim() == 3 and h_in.stride(0) == 0 and h_in.stride(1) == 0:      # fresh init_hidden(): zeros
            h_ptr = None
        else:
            h_in = h_in.reshape(rows, nat.HID)
            if not h_in.is_contiguous():
                h_in = h_in.contiguous()
            h_ptr = h_in.data_ptr()
        buf = th.empty(rows * (A + nat.HID), dtype=th.float32, device=dev)       # q | h_out, one allocation
        q = buf[:rows * A].view(B, N, A)
        h_out = buf[rows * A:].view(rows, nat.HID)
        with nat.on_device(dev):
            if self._pool is not None:
                nat.check(nat.lib().mal_rollout_step_pool(*self._pool_args(dev, B), B, N, OBS, A, C.byref(io), h_ptr,
                                                          h_out.data_ptr(), q.data_ptr(), C.byref(s), nat.current_stream(dev)),
                          "mal_rollout_step_pool")
            else:
                flat = self.agent.flat_params()
                nat.check(nat.lib().mal_rollout_step(flat.data_ptr(), B, N, OBS, A, C.byref(io), h_ptr, h_out.data_ptr(),
                                                     q.data_ptr(), C.byref(s), nat.current_stream(dev)), "mal_rollout_step")
        self.hidden_states = h_out
        if status is not None and int(status.item()) != 0:
            raise ValueError("Expected at least one available action per agent (Categorical probs are all zero)")
        return out[0], out[1]

    def forward(self, ep_batch, t, test_mode=False):
        """Q-values [bs, N, A] of timestep t.  Under `args.autograd_forward` (grad mode on, agent parameters or the hidden
        state requiring grad) the step records an autograd node (modules/autograd.py), so that a loss over the outputs can
        be back-propagated into the agent's parameters through time."""
        if self._pool is not None:
            if getattr(self.args, "autograd_forward", False) and th.is_grad_enabled():
                raise nat.MalError("forward with per-match policies records no autograd node (it reads no parameter of "
                                   "the agent); call it under torch.no_grad() or clear the policies")
            return self._step(ep_batch, t, None)
        if self._fusable():
            if self.hidden_states is not None and ag.recording(self, self.hidden_states, *self.agent.parameters()):
                return self._step_recorded(ep_batch, t)
            return self._step(ep_batch, t, None)
        agent_inputs = self._build_inputs(ep_batch, t)
        if self.hidden_states is None:
            raise HiddenStateNotInitialized()
        agent_outs = self._compute_agent_outputs(agent_inputs)
        return agent_outs.view(ep_batch.batch_size, self.n_agents, -1)

    def init_hidden(self, batch_size):
        self._check_pool_batch(batch_size)
        if isinstance(self.agent, DQNAgentNetwork):
            # The reference's expand() of the 3-D placeholder (basic_controller.py:59-60 on dqn_agent.py:27-32) raises a
            # RuntimeError, i.e. the "dqn" agent cannot be rolled out or trained there; here the placeholder is a
            # [bs, N, 1] zero tensor that nothing reads (dqn_agent.py:34-37 passes it through).
            self.hidden_states = th.zeros(batch_size, self.n_agents, 1, device=self.args.device)
            return
        self.hidden_states = self.agent.init_hidden().unsqueeze(0).expand(batch_size, self.n_agents, -1)

    def _check_pool_batch(self, batch_size):
        if self._pool is not None and batch_size != self._pool[1].numel():
            raise nat.MalError("per-match policies were set for %d matches, init_hidden(%d)" % (self._pool[1].numel(), batch_size))

    def update_trained_steps(self, update):
        if isinstance(update, th.Tensor):   # device-side count: accumulate without a host sync
            a = self.agent
            if a._trained_steps_dev is None:
                a._trained_steps_dev = th.zeros((), dtype=th.long, device=update.device)
            a._trained_steps_dev += update.reshape(()).to(th.long)
        else:
            self.agent._trained_steps_host += int(update)

    def parameters(self):
        return self.agent.parameters()

    def load_state(self, other_mac: "BasicMAC"):
        self.agent.load_state_dict(other_mac.agent.state_dict())

    def load_state_dict(self, agent):
        self.agent.load_state_dict(agent)

    def save_models(self, path, name):
        th.save(self.agent.state_dict(), "{}/{}agent.th".format(path, name))

    def load_models(self, path, name):
        self.agent.load_state_dict(th.load("{}/{}agent.th".format(path, name), map_location=lambda storage, loc: storage))

    # ------------------------------------------------------------------ hooks (kept for subclasses)
    def _build_agent(self, input_shape):
        return agent_REGISTRY[self.args.agent](input_shape, self.args)

    def _build_inputs(self, batch, t):
        """[obs_t | one-hot(a_{t-1}) | agent id], row order b-major (basic_controller.py:80-92).  Only used by
        subclasses / the non-fused path; the kernels never materialise this tensor."""
        bs = batch.batch_size
        parts = [batch["obs"][:, t]]
        if self.args.obs_last_action:
            parts.append(th.zeros_like(batch["actions_onehot"][:, t]) if t == 0 else batch["actions_onehot"][:, t - 1])
        if self.args.obs_agent_id:
            parts.append(th.eye(self.n_agents, device=batch.device).unsqueeze(0).expand(bs, -1, -1))
        return th.cat([x.reshape(bs * self.n_agents, -1) for x in parts], dim=1)

    def _compute_agent_outputs(self, agent_inputs):
        agent_outs, self.hidden_states = self.agent(agent_inputs, self.hidden_states)
        return agent_outs

    def _get_input_shape(self, scheme):
        input_shape = scheme["obs"]["vshape"]
        if self.args.obs_last_action:
            input_shape += scheme["actions_onehot"]["vshape"][0]
        if self.args.obs_agent_id:
            input_shape += self.n_agents
        return input_shape

    # ------------------------------------------------------------------ fused path
    def _fusable(self):
        cls = type(self)
        return (cls._build_inputs is BasicMAC._build_inputs and cls._compute_agent_outputs is BasicMAC._compute_agent_outputs
                and isinstance(self.agent, (DRQNAgentNetwork, DQNAgentNetwork)) and self.agent_output_type == "q")

    def _input_flags(self):
        """IN_* bits of the agent input the kernels assemble (obs_last_action / obs_agent_id, basic_controller.py:80-101)."""
        return nat.agent_input_flags(self.args.obs_last_action, self.args.obs_agent_id)

    def _rollout_fusable(self):
        return self._fusable() and isinstance(self.agent, DRQNAgentNetwork)

    def _no_recording(self):
        return th.no_grad() if getattr(self.args, "autograd_forward", False) else contextlib.nullcontext()

    def _step_inputs(self, ep_batch, t):
        """Pointers of the fused input assembly at timestep t: (obs [B, T+1, N, OBS], obs_ptr, last-action one-hot
        [B, T+1, N, A] or None, last_ptr, last_sb)."""
        obs_all = nat.require_cuda(ep_batch["obs"], "ep_batch")        # [B, T+1, N, OBS] (strided view of the records)
        OBS = obs_all.shape[3]
        A = self.n_actions
        if obs_all.stride(3) != 1 or obs_all.stride(2) != OBS or obs_all.dtype != th.float32:
            raise nat.MalError("obs must be float32 with contiguous [N, OBS] rows")
        obs_ptr = obs_all.data_ptr() + 4 * t * obs_all.stride(1)
        oh, last_ptr, last_sb = None, None, 0
        if t > 0 and self.args.obs_last_action:
            oh = ep_batch["actions_onehot"]
            if oh.stride(3) != 1 or oh.stride(2) != A or oh.dtype != th.float32:
                raise nat.MalError("actions_onehot must be float32 with contiguous [N, A] rows")
            last_ptr, last_sb = oh.data_ptr() + 4 * (t - 1) * oh.stride(1), oh.stride(0)
        return obs_all, obs_ptr, oh, last_ptr, last_sb

    def _step_recorded(self, ep_batch, t):
        """`_step` without selection as an autograd node: the same kernel launch, plus the backward of
        modules/autograd.py.  The obs / one-hot views it reads and h_in are saved for the version check."""
        obs_all, obs_ptr, oh, last_ptr, last_sb = self._step_inputs(ep_batch, t)
        B, _, N, OBS = obs_all.shape
        A = self.n_actions
        rows = B * N
        cfg = dict(rows=rows, N=N, OBS=OBS, A=A, dense_input=self._input_flags() << 1, obs_ptr=obs_ptr,
                   obs_sb=obs_all.stride(0), last_ptr=last_ptr, last_sb=last_sb)
        obs_v = obs_all[:, t]
        oh_v = oh[:, t - 1] if oh is not None else None
        with nat.on_device(obs_all.device):
            if isinstance(self.agent, DQNAgentNetwork):
                return ag.agent_step(self.agent, cfg, obs_v, oh_v, None).view(B, N, A)
            h_in = self.hidden_states
            if h_in.dim() == 3 and h_in.stride(0) == 0 and h_in.stride(1) == 0 and not h_in.requires_grad:
                h_in = None                                                # fresh init_hidden(): zeros
            else:
                h_in = h_in.reshape(rows, nat.HID).contiguous()
            q, h_out = ag.agent_step(self.agent, cfg, obs_v, oh_v, h_in)
        self.hidden_states = h_out
        return q.view(B, N, A)

    def _step(self, ep_batch, t, select_struct):
        if self.hidden_states is None:
            raise HiddenStateNotInitialized()
        obs_all, obs_ptr, _, last_ptr, last_sb = self._step_inputs(ep_batch, t)
        B, _, N, OBS = obs_all.shape
        A = self.n_actions
        flags = self._input_flags()
        rows = B * N
        dev = obs_all.device
        if isinstance(self.agent, DQNAgentNetwork):      # feed-forward agent: no hidden state to read or write
            q = th.empty(B, N, A, dtype=th.float32, device=dev)
            flat = self.agent.flat_params()
            with nat.on_device(dev):
                nat.check(nat.lib().mal_dqn_step(
                    flat.data_ptr(), rows, N, OBS, A, flags << 1, obs_ptr, obs_all.stride(0), last_ptr, last_sb, q.data_ptr(),
                    C.byref(select_struct) if select_struct is not None else None, nat.current_stream(dev)), "mal_dqn_step")
            return q
        h_in = self.hidden_states
        if h_in.dim() == 3 and h_in.stride(0) == 0 and h_in.stride(1) == 0:   # fresh init_hidden(): zeros
            h_ptr = None
        else:
            h_in = h_in.reshape(rows, nat.HID)
            if not h_in.is_contiguous():
                h_in = h_in.contiguous()
            h_ptr = h_in.data_ptr()
        buf = th.empty(rows * (A + nat.HID), dtype=th.float32, device=dev)      # q | h_out, one allocation
        q = buf[:rows * A].view(B, N, A)
        h_out = buf[rows * A:].view(rows, nat.HID)
        sel = C.byref(select_struct) if select_struct is not None else None
        with nat.on_device(dev):
            if self._pool is not None:
                nat.check(nat.lib().mal_agent_step_pool(
                    *self._pool_args(dev, B), rows, N, OBS, A, flags << 1, obs_ptr, obs_all.stride(0), last_ptr, last_sb,
                    h_ptr, h_out.data_ptr(), q.data_ptr(), sel, nat.current_stream(dev)), "mal_agent_step_pool")
            else:
                flat = self.agent.flat_params()
                nat.check(nat.lib().mal_agent_step(
                    flat.data_ptr(), rows, N, OBS, A, flags << 1, obs_ptr, obs_all.stride(0), last_ptr, last_sb, h_ptr,
                    h_out.data_ptr(), q.data_ptr(), sel, nat.current_stream(dev)), "mal_agent_step")
        self.hidden_states = h_out
        return q
