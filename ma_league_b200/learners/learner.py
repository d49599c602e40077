"""Learner base (reference: marl/learners/learner.py:6-78): name prefix + optimiser construction (RMSprop, or Adam
with `args.optimizer: "adam"` as pymarl2's configs select it)."""
import torch as th
from torch.optim import Adam, RMSprop

from .. import _native as nat
from ..flat import flat_views


class FusedRMSprop(RMSprop):
    """torch.optim.RMSprop (lr/alpha/eps as in learner.py:25-31; no momentum, not centered) whose state lives in ONE
    flat square_avg buffer and whose step is the fused clip+RMSprop kernel.  state_dict()/load_state_dict() keep
    torch's format, so the reference's `..opt.th` checkpoints (q_learner.py:133-147) interoperate."""

    def __init__(self, params, lr, alpha, eps):
        params = list(params)
        super().__init__(params, lr=lr, alpha=alpha, eps=eps)
        self._plist = params
        self._steps = 0
        self.flat_sq = None
        self._bind(None)

    def _bind(self, loaded):
        total = sum(p.numel() for p in self._plist)
        dev = self._plist[0].device
        self.flat_sq = th.zeros(total, dtype=th.float32, device=dev)
        views = flat_views(self.flat_sq, self._plist)
        for p, v in zip(self._plist, views):
            st = self.state[p]
            if loaded and "square_avg" in st:
                v.copy_(st["square_avg"].to(dev))
                self._steps = max(self._steps, int(st.get("step", th.tensor(0.)).item()))
            st["square_avg"] = v
            st["step"] = th.tensor(float(self._steps))

    def state_dict(self):
        for p in self._plist:
            self.state[p]["step"] = th.tensor(float(self._steps))
        return super().state_dict()

    def load_state_dict(self, state_dict):
        if any("alpha" not in g or "betas" in g for g in state_dict["param_groups"]):
            raise nat.MalError("not a torch.optim.RMSprop state dict (an Adam checkpoint needs args.optimizer: adam)")
        super().load_state_dict(state_dict)
        self._bind(True)

    def step(self, closure=None):
        raise nat.MalError("FusedRMSprop is stepped by QLearner.train (clip + RMSprop run inside mal_learner_step)")


class FusedAdam(Adam):
    """torch.optim.Adam (amsgrad=False, maximize=False, L2 weight decay that is not decoupled; betas and eps at torch's
    defaults unless a loaded state dict brings its own) whose state lives in ONE flat device buffer
    `exp_avg[P] | exp_avg_sq[P] | step | ticket` (MAL_ADAM_STATE_FLOATS) and whose step is the fused clip+Adam kernel.
    `exp_avg`, `exp_avg_sq` and `step` of every parameter are views of that buffer; the step counter lives on the device
    so that a replayed CUDA graph advances it.  state_dict()/load_state_dict() keep torch's format (a CPU float32
    `step` per parameter), so checkpoints interoperate with a stock torch.optim.Adam."""

    def __init__(self, params, lr, weight_decay=0.0):
        params = list(params)
        super().__init__(params, lr=lr, weight_decay=weight_decay)
        self._plist = params
        self._steps = 0
        self.flat_state = None
        self._bind(None)

    def _bind(self, loaded):
        P = sum(p.numel() for p in self._plist)
        dev = self._plist[0].device
        self.flat_state = th.zeros(nat.adam_state_floats(P), dtype=th.float32, device=dev)
        steps = 0
        for p, m, v in zip(self._plist, flat_views(self.flat_state, self._plist), flat_views(self.flat_state, self._plist, P)):
            st = self.state[p]
            if loaded and "exp_avg" in st:
                m.copy_(st["exp_avg"].to(dev))
                v.copy_(st["exp_avg_sq"].to(dev))
                steps = max(steps, int(st["step"].item()))
            st["exp_avg"], st["exp_avg_sq"], st["step"] = m, v, self.flat_state[2 * P]
        self._steps = steps
        self.flat_state[2 * P] = float(steps)

    def hyper(self, lr, clip):
        """mal_adam_t of this optimiser: betas, eps and weight_decay from param_groups[0], lr and clip from the args."""
        g = self.param_groups[0]
        return nat.AdamHyper(lr, g["betas"][0], g["betas"][1], g["eps"], g["weight_decay"], clip)

    def state_dict(self):
        sd = super().state_dict()
        step = th.tensor(float(self._steps))           # the host count equals the device counter; no sync needed
        sd["state"] = {k: dict(v, step=step.clone()) for k, v in sd["state"].items()}
        return sd

    def load_state_dict(self, state_dict):
        for g in state_dict["param_groups"]:
            if "betas" not in g or "alpha" in g:
                raise nat.MalError("not a torch.optim.Adam state dict (a RMSprop checkpoint needs args.optimizer: rmsprop)")
            for k in ("amsgrad", "maximize", "decoupled_weight_decay"):
                if g.get(k, False):
                    raise nat.MalError("the fused Adam step does not support %s=True" % k)
        super().load_state_dict(state_dict)
        self._bind(True)

    def step(self, closure=None):
        raise nat.MalError("FusedAdam is stepped by QLearner.train (clip + Adam run inside mal_learner_step_adam)")


class Learner:
    def __init__(self, mac, scheme, logger, args, name=None):
        self.mac = mac
        self.scheme = scheme
        self.logger = logger
        self.args = args
        self.name = f'{"" if name is None else name}_{self.__class__.__name__.lower()}_'
        self.log_stats_t = -self.args.learner_log_interval - 1
        self.optimiser = None

    def build_optimizer(self):
        """`args.optimizer`: absent or "rmsprop" (learner.py:25-31), or "adam" (pymarl2's qmix configs)."""
        kind = getattr(self.args, "optimizer", None)
        if kind is None or kind == "rmsprop":
            self.optimiser = FusedRMSprop(params=self.parameters(), lr=self.args.lr, alpha=self.args.optim_alpha,
                                          eps=self.args.optim_eps)
        elif kind == "adam":
            self.optimiser = FusedAdam(params=self.parameters(), lr=self.args.lr,
                                       weight_decay=getattr(self.args, "weight_decay", 0.0))
        else:
            raise nat.MalError('args.optimizer must be "rmsprop" or "adam", got %r' % (kind,))

    def parameters(self):
        raise NotImplementedError()

    def train(self, batch, t_env: int, episode_num: int) -> None:
        raise NotImplementedError()

    def cuda(self) -> None:
        raise NotImplementedError()

    def save_models(self, path, name):
        raise NotImplementedError()

    def load_models(self, path):
        raise NotImplementedError()

    def update_targets(self):
        pass
