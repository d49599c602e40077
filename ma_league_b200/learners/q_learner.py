"""Q-learning learner for VDN / QMIX / independent Q-learners (`mixer: None`) with the reference's API
(marl/learners/q_learner.py:11-147).

`train()` is one call into libmal_b200 (`mal_learner_step`): online + target RNN unroll, chosen-Q gather, masked
double-Q target max, mixers, TD loss, full backward (mixer + BPTT), clip_grad_norm_ and RMSprop, or Adam with
`args.optimizer: "adam"` (`mal_learner_step_adam`).  The TD targets are
the 1-step targets of q_learner.py:86, or lambda-returns when `args.td_lambda` is a number in [0, 1] (INTEGRATION.md).  Nothing is read
back to the host except on log steps (the reference syncs every step through `.item()`, q_learner.py:113).
`args.target_update_interval_or_tau` (EPyMARL) <= 1 blends the target networks softly inside the optimiser kernel.
"""
import copy
import ctypes as C
import math
import numbers

import torch as th

from .. import _native as nat
from ..flat import ensure_flat, flat_views
from ..modules.mixers.qmix import QMixer
from ..modules.mixers.vdn import VDNMixer
from .learner import FusedAdam, Learner


DP_RAW = 6     # raw sums written by k_stats_finalize at scalars[SC_RAW0:]: sum mtd^2, sum|mtd|, sum q_tot*m,
DP_TAIL = 8    # sum targets*m, sum m, count(m != 0); the tail is padded to 8 floats


def global_stats(raw, n_agents, scalars=None):
    """Logged statistics of q_learner.py:117-124 from the all-reduced raw sums (host tensor of >= DP_RAW floats)."""
    out = th.zeros(8) if scalars is None else scalars.clone()
    msum = float(raw[4])
    out[nat.SC_MASK_SUM] = msum
    out[nat.SC_LOSS] = float(raw[0]) / msum
    out[nat.SC_TD_ABS] = float(raw[1]) / msum
    out[nat.SC_Q_TAKEN] = float(raw[2]) / (msum * n_agents)
    out[nat.SC_TARGET] = float(raw[3]) / (msum * n_agents)
    return out


class QLearner(Learner):
    def __init__(self, mac, scheme, logger, args, name=None):
        super().__init__(mac, scheme, logger, args, name)
        self.last_target_update_episode = 0
        self.mixer = None
        if args.mixer is not None:
            if args.mixer == "vdn":
                self.mixer = VDNMixer(args)
            elif args.mixer == "qmix":
                self.mixer = QMixer(args)
            else:
                raise ValueError("Mixer {} not recognised.".format(args.mixer))
            self.target_mixer = copy.deepcopy(self.mixer)
        else:
            # IQL: every agent learns from its own TD error; there is no mixer and no target mixer
            self.target_mixer = None
        self.target_mac = copy.deepcopy(mac)
        self._ws = None
        self._ws_key = None
        self._plan = nat.Plan()
        self._grad = None
        self._grad_views = None
        self.save_q = False      # tests: also materialise mac_out / target_mac_out
        # CUDA graphs: the ~18 launches + fork/join events of one step are captured once per (batch storage, shape,
        # hyper-parameter) key and replayed; a step on a batch whose tensors live at addresses seen before costs one
        # graph launch on the host.  `args.cuda_graphs = False` (or `learner.use_graphs = False`) keeps eager launches.
        self.use_graphs = bool(getattr(args, "cuda_graphs", True))
        self._graphs = {}        # key -> (CUDAGraph, kernels per replay) ; key -> None after the first (eager) sighting
        self._graph_cap = 32
        self._graph_captures_left = 64   # a capture costs ~10 ms: batches whose addresses never repeat stay eager
        self._bs_cache = {}
        self.n_graph_replays = self.n_graph_captures = self.n_eager_steps = 0   # accounting (bench.py reports them)
        self.dp_profile = None   # set to [] to collect (start, end) CUDA events around the data-parallel exchange

    def build_optimizer(self):
        if self.mixer is None:
            self._agent_frozen()           # a frozen agent without a mixer leaves nothing to train: raise here already
        super().build_optimizer()

    def parameters(self):
        # q_learner.py:30-32 returns [] without a mixer (an operator-precedence slip); the agent's parameters are meant
        if self.mixer is None:
            return list(self.mac.parameters())
        return list(self.mac.parameters()) + list(self.mixer.parameters())

    # ------------------------------------------------------------------ ABI marshalling
    def _mixer_kind(self):
        if self.mixer is None:
            return nat.MIXER_NONE
        return self.mixer.mal_kind if isinstance(self.mixer, QMixer) else nat.MIXER_VDN

    def _cfg(self):
        a = self.args
        qm = isinstance(self.mixer, QMixer)
        return nat.LearnerCfg(self._mixer_kind(), int(bool(a.double_q)), self.mixer.embed_dim if qm else 0,
                              self.mixer.hypernet_embed if qm else 0, a.gamma, a.lr, a.optim_alpha, a.optim_eps,
                              a.grad_norm_clip, int(self.save_q), int(self._dp_world() > 1), int(self._agent_frozen()),
                              getattr(self.mac.agent, "mal_kind", nat.AGENT_RNN),
                              nat.agent_input_flags(getattr(a, "obs_last_action", True), getattr(a, "obs_agent_id", True)),
                              *self._returns(), self._target_update()[2])

    def _returns(self):
        """(mal_learner_cfg_t.returns, td_lambda) from `args.td_lambda`: absent or None is the 1-step target of
        q_learner.py:86; a number in [0, 1] selects TD(lambda) targets (build_td_lambda_targets, coma_learner.py:10-21)."""
        lam = getattr(self.args, "td_lambda", None)
        if lam is None:
            return nat.RETURNS_ONE_STEP, 0.0
        if isinstance(lam, bool) or not isinstance(lam, numbers.Real) or not 0.0 <= float(lam) <= 1.0:
            raise nat.MalError("args.td_lambda must be None or a number in [0, 1], got %r" % (lam,))
        return nat.RETURNS_TD_LAMBDA, float(lam)

    def _target_update(self):
        """(mode, interval, tau) from EPyMARL's `args.target_update_interval_or_tau`:
        - absent or None: ("hard", None, 0.0), hard copies every `args.target_update_interval` episodes
          (the reference rule; the interval is read where train() checks it, as the reference reads it);
        - a number > 1: ("hard", that number, 0.0), the same rule with this interval;
        - tau in (0, 1]: ("soft", None, tau), target = (1 - tau) target + tau param after every optimiser step, in the
          optimiser kernel (mal_learner_cfg_t.target_tau, the *_soft entries), and no hard copy."""
        v = getattr(self.args, "target_update_interval_or_tau", None)
        if v is None:
            return "hard", None, 0.0
        if isinstance(v, bool) or not isinstance(v, numbers.Real) or not math.isfinite(v) or not v > 0:
            raise nat.MalError("args.target_update_interval_or_tau must be None, an interval > 1 or a tau in (0, 1], "
                               "got %r" % (v,))
        return ("hard", v, 0.0) if v > 1 else ("soft", None, float(v))

    def _agent_frozen(self):
        """`freeze_agent_weights()` (multi_agent_controller.py:74-76, `args.freeze_native`): in the reference a frozen
        agent gets no gradient, stays out of the clip norm and is skipped by RMSprop, so only the mixer trains
        (q_learner.py:101-105).  Supported as all-or-nothing per network, like the reference's own switch."""
        ap = getattr(self.mac.agent, "_mal_params", None) or list(self.mac.parameters())   # cached list (flat.py)
        n_req = sum(1 for p in ap if p.requires_grad)
        if 0 < n_req < len(ap):
            raise nat.MalError("partially frozen agents are not supported: freeze all agent parameters or none")
        if self.mixer is None:
            if len(ap) > 0 and n_req == 0:
                raise nat.MalError("the agent is frozen (args.freeze_native) and there is no mixer: "
                                   "independent Q-learners (mixer=None) would have no parameter to train")
            return False
        mp = getattr(self.mixer, "_mal_params", None) or list(self.mixer.parameters())
        if not all(p.requires_grad for p in mp):
            raise nat.MalError("frozen mixer parameters are not supported by the fused learner step")
        return len(ap) > 0 and n_req == 0

    def _dp_world(self):
        """>1 when `args.data_parallel` is set and a process group exists: the batch given to train() is this rank's
        shard of the global batch (SURVEY.md 8e, config 5)."""
        if not getattr(self.args, "data_parallel", False):
            return 1
        import torch.distributed as dist
        return dist.get_world_size() if dist.is_available() and dist.is_initialized() else 1

    def _batch_struct(self, batch):
        obs = nat.require_cuda(batch["obs"], "batch")
        # the marshalled struct only depends on where the batch's tensors live: reuse it for a batch seen before
        # (unpacked batches keep one tensor per key, so every key's address is part of the identity)
        ck = (obs.data_ptr(), obs.shape, obs.stride()) + tuple(
            (batch[k].data_ptr(), batch[k].stride(0), batch[k].stride(1)) for k in
            ("actions_onehot", "actions", "avail_actions", "state", "reward", "terminated", "filled"))
        hit = self._bs_cache.get(ck)
        if hit is not None:
            return hit
        if len(self._bs_cache) >= 64:
            self._bs_cache.clear()
        bs = self._batch_struct_build(batch, obs)
        self._bs_cache[ck] = bs
        return bs

    def _batch_struct_build(self, batch, obs):
        B, TT, N, OBS = obs.shape
        A = self.args.n_actions
        state = batch["state"]
        S = state.shape[-1]
        b = nat.Batch(B, TT, N, A, OBS, S)
        b.obs = nat.field_of(obs, N * OBS)
        b.onehot = nat.field_of(batch["actions_onehot"], N * A)
        b.actions = nat.field_of(batch["actions"], N)
        b.avail = nat.field_of(batch["avail_actions"], N * A)
        b.state = nat.field_of(state, S)
        b.reward = nat.field_of(batch["reward"], 1)
        b.terminated = nat.field_of(batch["terminated"], 1)
        b.filled = nat.field_of(batch["filled"], 1)
        for key, dt in (("obs", th.float32), ("actions_onehot", th.float32), ("actions", th.long),
                        ("avail_actions", th.int32), ("state", th.float32), ("reward", th.float32),
                        ("terminated", th.uint8), ("filled", th.long)):
            if batch[key].dtype != dt:
                raise nat.MalError("scheme field %s must be %s (ma_experiment.py:99-118)" % (key, dt))
        return b

    def _prepare(self, batch):
        """Flat buffers, plan and workspace for this batch shape."""
        dev = batch["obs"].device
        bs = self._batch_struct(batch)
        if bs.weight.ptr:                # the cached struct may carry the weights of an earlier train() call
            bs.weight = nat.Field()
        cfg = self._cfg()
        key = (bs.B, bs.TT, bs.N, bs.A, bs.OBS, bs.S, cfg.mixer, cfg.save_q, str(dev))
        if key != self._ws_key:
            with nat.on_device(dev):     # the chunk layout is sized from the SM count of the learner's device
                nat.check(nat.lib().mal_learner_plan(C.byref(bs), C.byref(cfg), C.byref(self._plan)),
                          "mal_learner_plan")
            if self._ws is None or self._ws.numel() < self._plan.total_bytes or self._ws.device != dev:
                self._ws = th.empty(self._plan.total_bytes, dtype=th.uint8, device=dev)
            self._ws_key = key
        no_mixer = self.mixer is None
        flats = dict(agent=ensure_flat(self.mac.agent), tagent=ensure_flat(self.target_mac.agent),
                     mixer=None if no_mixer else ensure_flat(self.mixer),
                     tmixer=None if no_mixer else ensure_flat(self.target_mixer))
        n_total = self._plan.n_agent_params + self._plan.n_mixer_params
        if flats["agent"].numel() != self._plan.n_agent_params or \
                (flats["mixer"].numel() if flats["mixer"] is not None else 0) != self._plan.n_mixer_params:
            raise nat.MalError("parameter count mismatch between the modules and the kernel layout")
        if self._grad is None or self._grad.numel() != n_total or self._grad.device != dev:
            # + DP_TAIL floats: the rank's raw statistic sums ride in the same all-reduce as the gradient
            self._grad_store = th.zeros(n_total + DP_TAIL, dtype=th.float32, device=dev)
            self._grad = self._grad_store[:n_total]
            self._dp_scratch = th.empty((n_total + 255) // 256, dtype=th.float32, device=dev)
            self._grad_views = None
        return bs, cfg, flats

    def _ws_f32(self, offset, numel):
        return self._ws[offset:offset + 4 * numel].view(th.float32)

    def scalars(self):
        return self._ws_f32(self._plan.scalars, 64)

    # ------------------------------------------------------------------ training
    def train(self, batch, t_env: int, episode_num: int, weights=None):
        """`weights`: optional importance weights [B] (f32, on the batch's device) of prioritized replay: the loss becomes
        sum_b w_b sum_t (td*m)^2 / sum m.  None is the unweighted step, bit for bit."""
        bs, cfg, f = self._prepare(batch)
        if self.optimiser is None:
            raise nat.MalError("call build_optimizer() before train() (ma_experiment.py:61)")
        dev = batch["obs"].device
        dp = cfg.unnormalized != 0
        self._set_weights(bs, weights, dev, dp)
        adam = self._adam()
        counted = False                          # True: the trained-steps counter was advanced inside the replayed graph
        if dp:
            self._train_data_parallel(bs, cfg, f, dev, adam)
        elif self.use_graphs and not self.save_q:
            counted = self._step_graphed(bs, cfg, f, dev, adam)
        else:
            self._step_eager(bs, cfg, f, dev, adam)
        self.optimiser._steps += 1
        if getattr(self, "_grad_views", None) is None:   # p.grad = views of the flat (clipped) gradient, bound once
            params = self.parameters()
            self._grad_views = list(zip(params, flat_views(self._grad, params)))
        frozen = cfg.freeze_agent != 0
        for p, g in self._grad_views:
            if frozen and not p.requires_grad:
                continue                                  # a frozen parameter keeps p.grad = None, as in the reference
            if p.grad is not g:
                p.grad = g

        mode, interval, _ = self._target_update()
        if mode == "hard":
            if interval is None:
                interval = self.args.target_update_interval
            if (episode_num - self.last_target_update_episode) / interval >= 1.0:
                self.update_targets()
                self.last_target_update_episode = episode_num

        sc = self.scalars()
        if dp:
            n_total = self._grad.numel()
            self.mac.update_trained_steps(self._grad_store[n_total + 5:n_total + 6].round())   # global count
        elif not counted:
            self.mac.update_trained_steps(sc[nat.SC_MASK_COUNT:nat.SC_MASK_COUNT + 1].view(th.int32))

        if t_env - self.log_stats_t >= self.args.learner_log_interval:
            h = sc[:8].cpu()                            # the only device->host sync of the step
            if dp:
                h = global_stats(self._grad_store[self._grad.numel():].cpu(), self.args.n_agents, h)
            self.logger.log_stat(self.name + "loss", float(h[nat.SC_LOSS]), t_env)
            self.logger.log_stat(self.name + "grad_norm", h[nat.SC_GRAD_NORM].numpy(), t_env)
            self.logger.log_stat(self.name + "td_error_abs", float(h[nat.SC_TD_ABS]), t_env)
            self.logger.log_stat(self.name + "q_taken_mean", float(h[nat.SC_Q_TAKEN]), t_env)
            self.logger.log_stat(self.name + "target_mean", float(h[nat.SC_TARGET]), t_env)
            self.log_stats_t = t_env

    def _set_weights(self, bs, weights, dev, dp):
        if weights is None:
            return
        if dp or getattr(self.args, "data_parallel", False):
            raise nat.MalError("importance weights (prioritized replay) are not supported with data_parallel: "
                               "sharded sampling would need a sampler per rank and a global normaliser")
        if not isinstance(weights, th.Tensor) or weights.device != dev or weights.dtype != th.float32 or \
                weights.dim() != 1 or weights.numel() != bs.B:
            raise nat.MalError("weights must be a float32 [B] tensor on the batch's device")
        bs.weight = nat.Field(weights.data_ptr(), weights.stride(0), 0)

    def _adam(self):
        """The optimiser kernel of every training path: None selects clip + RMSprop (FusedRMSprop), a mal_adam_t
        clip + Adam (FusedAdam, lr and clip read from the args like the RMSprop path reads them)."""
        opt = self.optimiser
        return opt.hyper(self.args.lr, self.args.grad_norm_clip) if isinstance(opt, FusedAdam) else None

    def _step_eager(self, bs, cfg, f, dev, adam):
        if adam is not None:
            with nat.on_device(dev):
                nat.check(nat.lib().mal_learner_step_adam(
                    C.byref(bs), C.byref(cfg), C.byref(self._plan), nat.ptr(f["agent"]), nat.ptr(f["tagent"]),
                    nat.ptr(f["mixer"]), nat.ptr(f["tmixer"]), nat.ptr(self._ws), nat.ptr(self._grad), C.byref(adam),
                    nat.ptr(self.optimiser.flat_state), nat.current_stream(dev)), "mal_learner_step_adam")
            return
        with nat.on_device(dev):
            nat.check(nat.lib().mal_learner_step(C.byref(bs), C.byref(cfg), C.byref(self._plan),
                                                 nat.ptr(f["agent"]), nat.ptr(f["tagent"]), nat.ptr(f["mixer"]),
                                                 nat.ptr(f["tmixer"]), nat.ptr(self._ws), nat.ptr(self._grad),
                                                 nat.ptr(self.optimiser.flat_sq), nat.current_stream(dev)),
                      "mal_learner_step")

    def _step_graphed(self, bs, cfg, f, dev, adam):
        """Replay the captured step when this exact set of device addresses / shapes / hyper-parameters was seen
        before; first sighting runs eagerly (it also warms the library's streams and kernel attributes), the second
        one captures."""
        fields = (bs.obs, bs.onehot, bs.actions, bs.avail, bs.state, bs.reward, bs.terminated, bs.filled, bs.weight)
        key = (tuple((x.ptr, x.sb, x.st) for x in fields), bs.B, bs.TT, bs.N, bs.A, bs.OBS, bs.S,
               tuple(getattr(cfg, n) for n, _ in cfg._fields_),
               tuple(0 if v is None else v.data_ptr() for v in f.values()), self._ws.data_ptr(), self._grad.data_ptr(),
               self.optimiser.flat_sq.data_ptr() if adam is None else
               (self.optimiser.flat_state.data_ptr(),) + tuple(getattr(adam, n) for n, _ in adam._fields_), str(dev))
        entry = self._graphs.get(key, False)
        if entry:
            graph, n_kernels = entry
            graph.replay()
            nat.lib().mal_count_launches(n_kernels)
            self.n_graph_replays += 1
            return True
        if entry is False:                      # first sighting: eager
            if len(self._graphs) >= self._graph_cap:
                self._graphs.pop(next(iter(self._graphs)))
            self._graphs[key] = None
            self._step_eager(bs, cfg, f, dev, adam)
            self.n_eager_steps += 1
            return False
        if self._graph_captures_left <= 0:
            self._step_eager(bs, cfg, f, dev, adam)
            self.n_eager_steps += 1
            return False
        self._graph_captures_left -= 1
        self.n_graph_captures += 1
        # second sighting: capture (the capture stream becomes torch's current stream, which the C ABI call reads)
        lib = nat.lib()
        graph = th.cuda.CUDAGraph()
        th.cuda.synchronize(dev)
        n0 = lib.mal_launch_count()
        sc = self.scalars()
        self.mac.update_trained_steps(th.zeros(1, dtype=th.int32, device=dev))      # the device counter exists before capture
        with th.cuda.graph(graph, capture_error_mode="thread_local"):   # other threads may keep using CUDA meanwhile
            self._step_eager(bs, cfg, f, dev, adam)
            self.mac.update_trained_steps(sc[nat.SC_MASK_COUNT:nat.SC_MASK_COUNT + 1].view(th.int32))
        n_kernels = lib.mal_launch_count() - n0
        self._graphs[key] = (graph, n_kernels)
        graph.replay()                          # capture only records: this performs the step
        return True

    def _train_data_parallel(self, bs, cfg, f, dev, adam):
        """Config 5 (SURVEY.md 8e): every rank back-propagates the UN-normalised sum over its batch shard, one
        all-reduce(sum) carries the flat gradient plus the raw statistic sums (incl. mask.sum()), then every rank
        divides by the global mask sum and applies the identical clip + RMSprop (or Adam), which reproduces
        `loss = sum(masked_td^2) / mask.sum()` of q_learner.py:98 over the global batch."""
        import torch.distributed as dist
        sym = self._dp_symmetric(self._grad.numel(), dev)
        if sym is not None:
            return self._train_data_parallel_fused(bs, cfg, f, dev, sym, adam)
        lib, st = nat.lib(), nat.current_stream(dev)
        n_total = self._grad.numel()
        with nat.on_device(dev):
            nat.check(lib.mal_learner_forward(C.byref(bs), C.byref(cfg), C.byref(self._plan), nat.ptr(f["agent"]),
                                              nat.ptr(f["tagent"]), nat.ptr(f["mixer"]), nat.ptr(f["tmixer"]),
                                              nat.ptr(self._ws), st), "mal_learner_forward")
            nat.check(lib.mal_learner_backward(C.byref(bs), C.byref(cfg), C.byref(self._plan), nat.ptr(f["agent"]),
                                               nat.ptr(f["mixer"]), nat.ptr(self._ws), nat.ptr(self._grad), st),
                      "mal_learner_backward")
        self._grad_store[n_total:n_total + DP_RAW].copy_(self.scalars()[nat.SC_RAW0:nat.SC_RAW0 + DP_RAW])
        if self.dp_profile is not None:
            ev0 = th.cuda.Event(enable_timing=True)
            ev0.record()
        dist.all_reduce(self._grad_store, op=dist.ReduceOp.SUM)
        denom = self._grad_store[n_total + 4:]            # global mask.sum()
        a = self.args
        n_frozen = self._plan.n_agent_params if cfg.freeze_agent else 0
        soft = self._soft_target(cfg, f)
        with nat.on_device(dev):
            if adam is not None:
                args = (nat.ptr(f["agent"]), self._plan.n_agent_params, nat.ptr(f["mixer"]), self._plan.n_mixer_params,
                        nat.ptr(self._grad), nat.ptr(self.optimiser.flat_state), C.byref(adam), nat.ptr(self.scalars()),
                        nat.ptr(self._dp_scratch), nat.ptr(denom), n_frozen)
                if soft is None:
                    nat.check(lib.mal_clip_adam(*args, st), "mal_clip_adam")
                else:
                    nat.check(lib.mal_clip_adam_soft(*args, C.byref(soft), st), "mal_clip_adam_soft")
            else:
                args = (nat.ptr(f["agent"]), self._plan.n_agent_params, nat.ptr(f["mixer"]), self._plan.n_mixer_params,
                        nat.ptr(self._grad), nat.ptr(self.optimiser.flat_sq), a.lr, a.optim_alpha, a.optim_eps,
                        a.grad_norm_clip, nat.ptr(self.scalars()), nat.ptr(self._dp_scratch), nat.ptr(denom), n_frozen)
                if soft is None:
                    nat.check(lib.mal_clip_rmsprop(*args, st), "mal_clip_rmsprop")
                else:
                    nat.check(lib.mal_clip_rmsprop_soft(*args, C.byref(soft), st), "mal_clip_rmsprop_soft")
        if self.dp_profile is not None:
            ev1 = th.cuda.Event(enable_timing=True)
            ev1.record()
            self.dp_profile.append((ev0, ev1))

    @staticmethod
    def _soft_target(cfg, f):
        """The mal_soft_target_t of the data-parallel optimiser entries, or None without a soft target update (the
        single-process step reads tau from the cfg)."""
        if cfg.target_tau == 0.0:
            return None
        return nat.SoftTarget(cfg.target_tau, nat.ptr(f["tagent"]), nat.ptr(f["tmixer"]))

    # ---- fused exchange: peer-memory all-reduce inside the optimiser prologue (no NCCL call on the path)
    def _dp_symmetric(self, n_total, dev):
        """Two symmetric (peer-mapped) halves of [n_total + DP_TAIL] floats, rendezvoused over the default group.
        Returns None when the platform cannot provide them (then the NCCL all-reduce path is used)."""
        st = getattr(self, "_dp_sym", None)
        if st is not None and (st is False or st[0].shape[1] == n_total + DP_TAIL):
            return st or None
        self._dp_sym = False
        if not getattr(self.args, "dp_fused", True):
            return None
        try:
            import torch.distributed as dist
            import torch.distributed._symmetric_memory as symm_mem
            if dist.get_backend() != "nccl":
                return None
            buf = symm_mem.empty(2, n_total + DP_TAIL, dtype=th.float32, device=dev)
            hdl = symm_mem.rendezvous(buf, dist.group.WORLD)
            if hdl.world_size > 16:
                return None
            buf.zero_()
            ptrs = [(C.c_void_p * hdl.world_size)(*[int(p) + 4 * h * (n_total + DP_TAIL) for p in hdl.buffer_ptrs])
                    for h in range(2)]
            hdl.barrier(channel=0)
            self._dp_sym = (buf, hdl, ptrs)
            self._dp_step = 0
        except Exception as ex:                         # no peer access / symmetric memory on this platform
            self._dp_sym_error = repr(ex)
            return None
        return self._dp_sym

    def _train_data_parallel_fused(self, bs, cfg, f, dev, sym, adam):
        buf, hdl, ptrs = sym
        lib, st = nat.lib(), nat.current_stream(dev)
        n_total = self._grad.numel()
        h = self._dp_step & 1                            # double-buffered: ONE cross-rank barrier per step is enough
        half = buf[h]
        with nat.on_device(dev):
            nat.check(lib.mal_learner_forward(C.byref(bs), C.byref(cfg), C.byref(self._plan), nat.ptr(f["agent"]),
                                              nat.ptr(f["tagent"]), nat.ptr(f["mixer"]), nat.ptr(f["tmixer"]),
                                              nat.ptr(self._ws), st), "mal_learner_forward")
            nat.check(lib.mal_learner_backward(C.byref(bs), C.byref(cfg), C.byref(self._plan), nat.ptr(f["agent"]),
                                               nat.ptr(f["mixer"]), nat.ptr(self._ws), nat.ptr(half), st),
                      "mal_learner_backward")
        half[n_total:n_total + DP_RAW].copy_(self.scalars()[nat.SC_RAW0:nat.SC_RAW0 + DP_RAW])
        if self.dp_profile is not None:
            ev0 = th.cuda.Event(enable_timing=True)
            ev0.record()
        hdl.barrier(channel=0)                           # every rank's half h is complete (and half h^1 is free again)
        a = self.args
        n_frozen = self._plan.n_agent_params if cfg.freeze_agent else 0
        soft = self._soft_target(cfg, f)
        head = (ptrs[h], hdl.world_size, nat.ptr(f["agent"]), self._plan.n_agent_params, nat.ptr(f["mixer"]),
                self._plan.n_mixer_params, nat.ptr(self._grad), nat.ptr(self._grad_store[n_total:]), DP_TAIL)
        with nat.on_device(dev):
            if adam is not None:
                args = head + (nat.ptr(self.optimiser.flat_state), C.byref(adam), nat.ptr(self.scalars()),
                               nat.ptr(self._dp_scratch), n_frozen)
                if soft is None:
                    nat.check(lib.mal_peer_allreduce_clip_adam(*args, st), "mal_peer_allreduce_clip_adam")
                else:
                    nat.check(lib.mal_peer_allreduce_clip_adam_soft(*args, C.byref(soft), st),
                              "mal_peer_allreduce_clip_adam_soft")
            else:
                args = head + (nat.ptr(self.optimiser.flat_sq), a.lr, a.optim_alpha, a.optim_eps, a.grad_norm_clip,
                               nat.ptr(self.scalars()), nat.ptr(self._dp_scratch), n_frozen)
                if soft is None:
                    nat.check(lib.mal_peer_allreduce_clip_rmsprop(*args, st), "mal_peer_allreduce_clip_rmsprop")
                else:
                    nat.check(lib.mal_peer_allreduce_clip_rmsprop_soft(*args, C.byref(soft), st),
                              "mal_peer_allreduce_clip_rmsprop_soft")
        if self.dp_profile is not None:
            ev1 = th.cuda.Event(enable_timing=True)
            ev1.record()
            self.dp_profile.append((ev0, ev1))
        self._dp_step += 1

    def train_from_buffer(self, buffer, batch_size: int, t_env: int, episode_num: int, truncate: bool = False):
        """The learner-side input pipeline of runs/train/ma_experiment.py:231-239 in one call:
        `sample(batch_size)` -> [`max_t_filled` -> truncate] -> `train`.

        The sampled records land in a persistent staging batch (one bulk record-copy launch, stable addresses, so the
        step replays its CUDA graph) and, by default, the padding is MASKED instead of truncated: the step runs over
        the buffer's full sequence length and transitions past an episode's end carry mask 0, which gives the same
        loss, gradients and update as the reference's truncation (steps after the longest episode's last one are
        unfilled) without the host sync that `max_t_filled` as a Python slice bound costs.  `truncate=True` keeps the
        reference's exact sequence (one device->host sync per step, less arithmetic when episodes are short).
        Precondition of the masked form, as in the reference's steppers: an episode shorter than the sequence length
        ends with `terminated = 1` on its last transition.

        A `PrioritizedReplayBuffer` runs sample (by priority, beta = `buffer.beta_at(t_env)`) -> record copy -> the
        importance-weighted step -> priority update of the sampled episodes from the step's TD errors: two launches more
        than the uniform step, and still no host sync in the masked form."""
        from ..components.replay_buffers.prioritized_replay_buffer import PrioritizedReplayBuffer
        per = isinstance(buffer, PrioritizedReplayBuffer)
        if per and getattr(self.args, "data_parallel", False):
            raise nat.MalError("prioritized replay is not supported with data_parallel")
        st = getattr(self, "_stage", None)
        if st is None or st.batch_size != batch_size or st.max_seq_length != buffer.max_seq_length or \
                st._storage.device != buffer._storage.device or not st._layout.same_as(buffer._layout):
            st = buffer._gather_records(th.zeros(batch_size, dtype=th.long))   # a packed batch with the buffer's layout
            self._stage = st
        if per:
            buffer.sample_into(st, buffer.beta_at(t_env))
        else:
            buffer.sample_into(st)
        batch = st
        if truncate:
            batch = st[:, :int(st.max_t_filled())]
        self.train(batch, t_env, episode_num, weights=st.weights if per else None)
        if per:
            B, T = batch.batch_size, batch.max_seq_length - 1
            Q = self.args.n_agents if self.mixer is None else 1
            buffer.update_priorities(st.ids, self._ws_f32(self._plan.td, B * T * Q).view(B, T, Q),
                                     self._ws_f32(self._plan.mask, B * T))
        return batch

    def forward_only(self, batch):
        """Forward half of train() (q_learner.py:36-98); intermediates stay in the workspace (tests, debugging)."""
        bs, cfg, f = self._prepare(batch)
        dev = batch["obs"].device
        with nat.on_device(dev):
            nat.check(nat.lib().mal_learner_forward(C.byref(bs), C.byref(cfg), C.byref(self._plan),
                                                    nat.ptr(f["agent"]), nat.ptr(f["tagent"]), nat.ptr(f["mixer"]),
                                                    nat.ptr(f["tmixer"]), nat.ptr(self._ws), nat.current_stream(dev)),
                      "mal_learner_forward")
        return bs, cfg, f

    def forward_backward(self, batch):
        """forward + loss.backward() without the optimiser step; returns the flat unclipped gradient."""
        bs, cfg, f = self.forward_only(batch)
        dev = batch["obs"].device
        with nat.on_device(dev):
            nat.check(nat.lib().mal_learner_backward(C.byref(bs), C.byref(cfg), C.byref(self._plan),
                                                     nat.ptr(f["agent"]), nat.ptr(f["mixer"]), nat.ptr(self._ws),
                                                     nat.ptr(self._grad), nat.current_stream(dev)),
                      "mal_learner_backward")
        return self._grad

    def intermediates(self, batch):
        """Views of the workspace arrays produced by the last forward for `batch`'s shape (q_tot / target_q_tot /
        targets / td are [B,T,N] without a mixer: one TD error per agent)."""
        p = self._plan
        B, TT = batch.batch_size, batch.max_seq_length
        N, A, T = self.args.n_agents, self.args.n_actions, TT - 1
        Q = N if self.mixer is None else 1
        out = dict(chosen=self._ws_f32(p.chosen, B * T * N).view(B, T, N),
                   target_max=self._ws_f32(p.target_max, B * T * N).view(B, T, N),
                   argmax=self._ws[p.argmax:p.argmax + 4 * B * T * N].view(th.int32).view(B, T, N),
                   mask=self._ws_f32(p.mask, B * T).view(B, T, 1),
                   q_tot=self._ws_f32(p.q_tot, B * T * Q).view(B, T, Q),
                   target_q_tot=self._ws_f32(p.target_q_tot, B * T * Q).view(B, T, Q),
                   targets=self._ws_f32(p.targets, B * T * Q).view(B, T, Q),
                   td=self._ws_f32(p.td, B * T * Q).view(B, T, Q),
                   hout=self._ws_f32(p.h_on, TT * B * N * nat.HID).view(TT, B * N, nat.HID),
                   # relu(fc1): its own array for the recurrent agent, the "hidden state" itself for the feed-forward one
                   x=self._ws_f32(p.h_on if getattr(self.mac.agent, "mal_kind", nat.AGENT_RNN) == nat.AGENT_DQN else p.x_on,
                                  TT * B * N * nat.HID).view(TT, B * N, nat.HID),
                   scalars=self.scalars())
        if isinstance(self.mixer, QMixer):
            E, HE = self.mixer.embed_dim, self.mixer.hypernet_embed
            two = self._mixer_kind() == nat.MIXER_QMIX2
            ld1, ld2 = (2 * HE + 2 * E) if two else 2 * E, E * N + E
            out["a2"] = self._ws_f32(p.a2_on, B * T * ld2).view(B * T, ld2)     # a1 | af (pre-abs)
            out["y1"] = self._ws_f32(p.y1_on, B * T * ld1).view(B * T, ld1)     # [h1 | hf |] b1 | v1
        if self.save_q:
            out["mac_out"] = self._ws_f32(p.mac_out, B * TT * N * A).view(B, TT, N, A)
            out["target_mac_out"] = self._ws_f32(p.target_mac_out, B * TT * N * A).view(B, TT, N, A)
        return out

    def update_targets(self):
        """q_learner.py:127-131: online -> target copy (one flat device copy per network).  train() calls it in hard
        mode; with a soft `target_update_interval_or_tau` it is only the public hard copy."""
        pairs = [(ensure_flat(self.target_mac.agent), ensure_flat(self.mac.agent))]
        if self.mixer is not None:
            pairs.append((ensure_flat(self.target_mixer), ensure_flat(self.mixer)))
        for dst, src in pairs:
            if dst is None:
                continue
            with nat.on_device(dst.device):
                nat.check(nat.lib().mal_copy_f32(nat.ptr(dst), nat.ptr(src), src.numel(),
                                                 nat.current_stream(dst.device)), "mal_copy_f32")
        self.logger.info("Updated {0}target network.".format(self.name))

    def save_models(self, path, name=None):
        self.mac.save_models(path, name=self.name)
        if self.mixer is not None:
            th.save(self.mixer.state_dict(), "{}/{}mixer.th".format(path, self.name))
        th.save(self.optimiser.state_dict(), "{}/{}opt.th".format(path, self.name))

    def load_models(self, path):
        self.mac.load_models(path, self.name)
        self.target_mac.load_models(path, self.name)   # "not quite right", as in q_learner.py:141-142
        if self.mixer is not None:
            self.mixer.load_state_dict(
                th.load("{}/{}mixer.th".format(path, self.name), map_location=lambda storage, loc: storage))
        self.optimiser.load_state_dict(
            th.load("{}/{}opt.th".format(path, self.name), map_location=lambda storage, loc: storage))
