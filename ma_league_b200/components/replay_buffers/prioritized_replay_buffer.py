"""Proportional prioritized episode replay (Schaul et al., 2016) on the device, under the reference's class name
(marl/components/replay_buffers/prioritized_replay_buffer.py, which cannot run there: `tree.add` has the wrong arity).

Contract (INTEGRATION.md):
* slot i has priority p_i in a device f32 [buffer_size] tensor; a newly inserted episode gets the running maximum stored
  priority, which starts at 1.0 and stays on the device;
* sampling is with replacement and stratified: over the n = episodes_in_buffer live slots, draw j of B lands at
  (j + u_j) * total / B and takes the first slot whose inclusive prefix sum exceeds that point (one launch, mal_per_sample);
* importance weights w_j = (p_min / p_{id_j})^beta, i.e. (n P(j))^-beta normalised by the largest weight over the buffer;
* after a learner step the sampled slots get (sum_t |td*m| / sum_t m + eps)^alpha (over t and agents without a mixer);
  when a slot was drawn twice the occurrence with the highest batch index wins (one launch, mal_per_update).
"""
import ctypes as C
import math

import torch as th

from ... import _native as nat
from .replay_buffer import ReplayBuffer


def _hyper(name, v):
    if isinstance(v, bool) or not isinstance(v, (int, float)) or not math.isfinite(v) or v < 0:
        raise nat.MalError("prioritized replay: %s must be a finite number >= 0, got %r" % (name, v))
    return float(v)


class PrioritizedReplayBuffer(ReplayBuffer):
    def __init__(self, scheme, groups, buffer_size: int, max_seq_length: int, preprocess=None, device="cpu",
                 alpha: float = 0.6, beta: float = 0.4, eps: float = 1e-6, beta_anneal_t=None):
        """`beta_anneal_t`: when set, `beta_at(t_env)` grows beta linearly from `beta` to 1 over that many env steps
        (QLearner.train_from_buffer samples with it); None keeps beta fixed."""
        self.alpha, self.beta, self.eps = _hyper("alpha", alpha), _hyper("beta", beta), _hyper("eps", eps)
        if beta_anneal_t is not None and _hyper("beta_anneal_t", beta_anneal_t) <= 0:
            raise nat.MalError("prioritized replay: beta_anneal_t must be > 0 or None")
        self.beta_anneal_t = beta_anneal_t
        super().__init__(scheme, groups, buffer_size, max_seq_length, preprocess=preprocess, device=device)
        if self._layout is None or self._storage.device.type != "cuda":
            raise nat.MalError("prioritized replay needs a device-resident buffer: host-resident buffers "
                               "(buffer_cpu_only) and wire records are not supported")
        dev = self._storage.device
        self.priorities = th.zeros(buffer_size, dtype=th.float32, device=dev)
        self.max_priority = th.ones(1, dtype=th.float32, device=dev)

    def beta_at(self, t_env: int) -> float:
        if self.beta_anneal_t is None or self.beta >= 1.0:
            return self.beta
        return min(1.0, self.beta + (1.0 - self.beta) * max(0, t_env) / self.beta_anneal_t)

    def insert_episode_batch(self, ep_batch):
        """The parent's ring insert; every new slot gets the running maximum priority (a device copy, no sync)."""
        n = ep_batch.batch_size
        if self.buffer_index + n <= self.buffer_size:
            self.priorities[self.buffer_index:self.buffer_index + n].copy_(self.max_priority.expand(n))
        super().insert_episode_batch(ep_batch)

    # ------------------------------------------------------------------ sampling
    def sample_ids(self, batch_size: int, beta=None, ids=None, weights=None, u=None):
        """Episode ids [B] int64 and importance weights [B] f32 on the device, drawn by priority (mal_per_sample).
        `u`: optional device uniforms [B] (tests); without them the draw takes Philox from torch's default CUDA generator
        in th.rand(B)'s layout and advances it the same way, so torch.manual_seed reproduces it."""
        beta = self.beta if beta is None else _hyper("beta", beta)
        dev = self.priorities.device
        if ids is None:
            ids = th.empty(batch_size, dtype=th.long, device=dev)
        if weights is None:
            weights = th.empty(batch_size, dtype=th.float32, device=dev)
        lib = nat.lib()
        nat.check(lib.mal_per_sample_check(self.episodes_in_buffer, batch_size, beta), "mal_per_sample")
        adv = C.c_uint64(0)
        with nat.on_device(dev):
            if u is None:
                gen = th.cuda.default_generators[dev.index if dev.index is not None else th.cuda.current_device()]
                seed, off = gen.initial_seed(), gen.get_offset()
            else:
                seed, off = 0, 0
            nat.check(lib.mal_per_sample(nat.ptr(self.priorities), self.episodes_in_buffer, batch_size, beta,
                                         nat.ptr(u), seed, off, nat.ptr(ids), nat.ptr(weights), C.byref(adv),
                                         nat.current_stream(dev)), "mal_per_sample")
            if u is None:
                gen.set_offset(off + adv.value)
        return ids, weights

    def sample(self, batch_size: int, beta=None):
        """A gathered batch of `batch_size` episodes drawn by priority; `.ids` / `.weights` hold the draw."""
        ids, w = self.sample_ids(batch_size, beta)
        out = self._gather_records(ids)
        out.ids, out.weights = ids, w
        return out

    def sample_into(self, out, beta=None):
        """`sample(out.batch_size, beta)` into the caller's packed staging batch `out` (stable addresses, so the learner's
        CUDA graph replays); the ids and weights land in tensors kept on `out` from call to call."""
        n = out.batch_size
        if self._layout is None or out._layout is None or not self._layout.same_as(out._layout):
            raise nat.MalError("sample_into needs packed batches with the buffer's record layout")
        if out._storage.device != self._storage.device:
            raise nat.MalError("sample_into: the buffer and the output batch must live on the same CUDA device")
        ids, w = getattr(out, "ids", None), getattr(out, "weights", None)
        if ids is None or ids.numel() != n or ids.device != self.priorities.device:
            ids = th.empty(n, dtype=th.long, device=self.priorities.device)
            w = th.empty(n, dtype=th.float32, device=self.priorities.device)
        self.sample_ids(n, beta, ids, w)
        dev = self._storage.device
        rb = self._layout.record_bytes
        with th.cuda.device(dev):
            nat.check(nat.lib().mal_record_copy(nat.ptr(out._storage), rb, None, nat.ptr(self._storage), rb,
                                                nat.ptr(ids), n, rb, nat.current_stream(dev)), "mal_record_copy")
        out.ids, out.weights = ids, w
        return out

    # ------------------------------------------------------------------ priority update
    def update_priorities(self, ids, td, mask):
        """New priorities of the sampled episodes `ids` [B] from a learner step's TD errors `td` [B,T,n_q] (n_q = 1 with a
        mixer, n_agents without) and mask `mask` [B,T(,1)]: (sum |td*m| / sum m + eps)^alpha; the highest batch index
        wins for a slot drawn twice, and the running maximum follows (mal_per_update, no sync)."""
        B = ids.numel()
        td = td.reshape(B, -1, td.shape[-1]) if td.dim() == 3 else td.reshape(B, -1, 1)
        T, nq = td.shape[1], td.shape[2]
        for t, what in ((ids, "ids"), (td, "td"), (mask, "mask")):
            if not t.is_cuda or t.device != self.priorities.device or not t.is_contiguous():
                raise nat.MalError("update_priorities: %s must be contiguous on the buffer's device" % what)
        if ids.dtype != th.long or td.dtype != th.float32 or mask.dtype != th.float32 or mask.numel() != B * T:
            raise nat.MalError("update_priorities: ids int64 [B], td f32 [B,T,n_q], mask f32 [B,T]")
        lib = nat.lib()
        nat.check(lib.mal_per_update_check(B, T, nq, self.alpha, self.eps), "mal_per_update")
        with nat.on_device(self.priorities.device):
            nat.check(lib.mal_per_update(nat.ptr(td), nat.ptr(mask), B, T, nq, nat.ptr(ids), self.alpha, self.eps,
                                         nat.ptr(self.priorities), self.buffer_size, nat.ptr(self.max_priority),
                                         nat.current_stream(self.priorities.device)), "mal_per_update")

    def __repr__(self):
        return "PrioritizedReplayBuffer. {}/{} episodes. Keys:{} Groups:{}".format(
            self.episodes_in_buffer, self.buffer_size, self.scheme.keys(), self.groups.keys())
