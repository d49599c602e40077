"""Soft target updates (`args.target_update_interval_or_tau` in (0, 1]) in the fused optimiser kernels, on the device.

The central check is a lock-step twin: learner S trains with tau, learner H is the same system in hard mode with an
interval that never fires, and after each of H's steps its target flats are overwritten with the reference blend of
tests/soft_target_ref.py (three fp32 torch ops) of its own post-step parameters.  After every chained `train()` step
S and H must be bit-identical in every parameter, every target parameter, the optimiser state, `p.grad` and the logged
statistics.  Also: tau = 1 copies; a frozen agent's target moves toward its frozen parameters; eager against graph
replay and re-capture when tau changes; `train_from_buffer` (uniform and prioritized) without a host sync; the launch
count; interval values > 1; the four stand-alone `*_soft` entries against their namesakes and numpy; two data-parallel
ranks against the full batch."""
import ctypes as C
import multiprocessing as mp
import os

import numpy as np
import pytest
import torch as th
import torch.distributed as dist

import ma_league_b200 as M
from ma_league_b200 import _native as nat
from ma_league_b200.learners.q_learner import DP_TAIL
from tests import soft_target_ref as R
from tests.gpu_helpers import np_params
from tests.helpers import rel_err
from tests.test_data_parallel import _free_port
from tests.test_gpu_td_lambda import _fill, _per_buffer, _system

pytestmark = pytest.mark.gpu
DEV = "cuda"
TOL = 1e-5


def _pair(N, B, TT, mixer, tau, layers=2, agent="rnn", optimizer="rmsprop", lam=None, seed=0, **kw):
    """(S, H): identical systems, S soft with tau, H in hard mode (target_update_interval 200, episode 0: no copy)."""
    lr = dict(lr=1e-3) if optimizer == "adam" else {}
    S = _system(N, B, TT, mixer, lam, layers, agent, seed=seed, optimizer=optimizer, target_update_interval_or_tau=tau,
                **lr, **kw)
    H = _system(N, B, TT, mixer, lam, layers, agent, seed=seed, optimizer=optimizer, **lr, **kw)
    return S, H


def _targets(s):
    L = s.learner
    return [L.target_mac.agent] + ([L.target_mixer] if L.mixer is not None else [])


def _onlines(s):
    L = s.learner
    return [s.mac.agent] + ([L.mixer] if L.mixer is not None else [])


def _opt_state(L):
    o = L.optimiser
    return o.flat_state if hasattr(o, "flat_state") else o.flat_sq


def _everything(s):
    """Parameters, target parameters, optimiser state, p.grad and the logged statistics (device tensors cloned)."""
    L = s.learner
    out = [p.detach().clone() for m in _onlines(s) + _targets(s) for p in m.parameters()]
    out.append(_opt_state(L).clone())
    out += [p.grad.clone() for p in L.parameters() if p.grad is not None]
    out.append(th.tensor([v for k, (v, _) in sorted(s.logger.stats.items())], dtype=th.float64))
    return out


def assert_identical(a, b, what):
    xa, xb = _everything(a), _everything(b)
    assert len(xa) == len(xb), what
    for i, (x, y) in enumerate(zip(xa, xb)):
        assert th.equal(x, y), "%s: item %d differs (max |diff| %g)" % (what, i, (x.double() - y.double()).abs().max())


def twin_steps(S, H, tau, steps=3, t0=0):
    for i in range(steps):
        S.learner.train(S.batch, t_env=t0 + i, episode_num=0)
        H.learner.train(H.batch, t_env=t0 + i, episode_num=0)
        R.blend_modules_(_targets(H), _onlines(H), tau)
        th.cuda.synchronize()
        assert_identical(S, H, "after step %d" % (t0 + i + 1))
    assert S.logger.infos == [] and S.learner.last_target_update_episode == 0


CASES = [  # N, B, TT, mixer, layers, agent, optimizer, lambda, tau
    (3, 32, 201, "qmix", 2, "rnn", "rmsprop", None, 0.005),
    (5, 32, 201, "qmix", 2, "rnn", "rmsprop", None, 0.3),
    (5, 32, 201, "qmix", 2, "rnn", "adam", None, 1.0),
    (5, 32, 201, "qmix", 2, "dqn", "adam", None, 0.005),
    (5, 32, 201, "qmix", 1, "rnn", "rmsprop", 0.6, 0.005),
    (5, 32, 201, "qmix", 1, "dqn", "adam", 0.6, 1.0),
    (3, 32, 201, "vdn", 2, "dqn", "rmsprop", None, 1.0),
    (5, 32, 201, "vdn", 2, "rnn", "adam", 0.6, 0.3),
    (5, 32, 201, None, 2, "rnn", "rmsprop", None, 0.3),
    (3, 32, 201, None, 2, "dqn", "adam", 0.6, 0.005),
    (20, 16, 24, "qmix", 2, "rnn", "adam", 0.6, 0.3),
    (20, 16, 24, "vdn", 2, "dqn", "rmsprop", 0.6, 0.005),
    (20, 16, 24, None, 2, "rnn", "rmsprop", None, 1.0),
]


@pytest.mark.parametrize("N,B,TT,mixer,layers,agent,optimizer,lam,tau", CASES)
def test_lock_step_twin(N, B, TT, mixer, layers, agent, optimizer, lam, tau):
    S, H = _pair(N, B, TT, mixer, tau, layers, agent, optimizer, lam, seed=500 + N + TT)
    twin_steps(S, H, tau)
    assert S.learner.n_graph_replays == 1 and S.learner.n_graph_captures == 1      # eager, capture, replay


@pytest.mark.parametrize("mixer", ["qmix", None])
def test_tau_one_copies(mixer):
    S, _ = _pair(5, 16, 61, mixer, 1.0, seed=8)
    for i in range(3):
        S.learner.train(S.batch, i, 0)
        th.cuda.synchronize()
        for tm, m in zip(_targets(S), _onlines(S)):
            for tp, p in zip(tm.parameters(), m.parameters()):
                assert th.equal(tp, p)


def test_frozen_agent_target_moves_toward_frozen_parameters():
    tau = 0.3
    S, H = _pair(5, 16, 61, "qmix", tau, seed=9)
    for s in (S, H):
        s.mac.freeze_agent_weights()
    agent0 = [p.detach().clone() for p in S.mac.agent.parameters()]
    gap0 = sum(float((tp.detach() - p).abs().sum()) for tp, p in zip(S.learner.target_mac.agent.parameters(), agent0))
    mixer0 = [p.detach().clone() for p in S.learner.mixer.parameters()]
    twin_steps(S, H, tau)
    for p, p0 in zip(S.mac.agent.parameters(), agent0):
        assert th.equal(p, p0)
    gap = sum(float((tp.detach() - p).abs().sum()) for tp, p in zip(S.learner.target_mac.agent.parameters(), agent0))
    assert abs(gap - gap0 * (1 - tau) ** 3) <= 1e-4 * gap0
    assert any(not th.equal(p, p0) for p, p0 in zip(S.learner.mixer.parameters(), mixer0))


@pytest.mark.parametrize("optimizer", ["rmsprop", "adam"])
def test_graph_replay_bit_identical_to_eager_and_recapture_on_tau_change(optimizer):
    Sg, H = _pair(5, 8, 61, "qmix", 0.3, optimizer=optimizer, seed=4)
    Se, _ = _pair(5, 8, 61, "qmix", 0.3, optimizer=optimizer, seed=4)
    Se.learner.use_graphs = False
    for i in range(4):                                       # eager, capture, replay, replay
        Sg.learner.train(Sg.batch, i, 0)
        Se.learner.train(Se.batch, i, 0)
        H.learner.train(H.batch, i, 0)
        R.blend_modules_(_targets(H), _onlines(H), 0.3)
    th.cuda.synchronize()
    assert Sg.learner.n_graph_captures == 1 and Sg.learner.n_graph_replays == 2 and Se.learner.n_graph_replays == 0
    assert_identical(Sg, Se, "graph replay against eager")
    assert_identical(Sg, H, "graph replay against the twin")
    captures, replays = Sg.learner.n_graph_captures, Sg.learner.n_graph_replays
    Sg.args.target_update_interval_or_tau = 0.01
    twin_steps(Sg, H, 0.01, t0=4)                            # its own key: eager, capture, replay with the new tau
    assert Sg.learner.n_graph_captures == captures + 1 and Sg.learner.n_graph_replays == replays + 1


@pytest.mark.parametrize("per", [False, True])
def test_train_from_buffer_equals_manual_loop(per):
    """Uniform and prioritized replay with a soft target update, graphs on, against the same steps by hand with eager
    launches: bit-identical; the prioritized steps run under `set_sync_debug_mode("error")`."""
    def system():
        s = _system(5, 8, 31, "qmix", 0.6, seed=9, open_ended=False, target_update_interval_or_tau=0.05)
        buf = _per_buffer(s, 64, 31) if per else M.ReplayBuffer(s.scheme, s.groups, 64, 31, preprocess=s.pre, device=DEV)
        _fill(s, buf, 8, 8, 31, 16, 5, short=20)
        s.learner.log_stats_t = 10 ** 9                      # no log step: nothing is read back
        return s, buf
    (s1, b1), (s2, b2) = system(), system()
    th.manual_seed(77)
    np.random.seed(77)
    for i in range(3):                                       # eager, capture, replay
        s1.learner.train_from_buffer(b1, 8, t_env=i, episode_num=0)
    th.cuda.synchronize()
    if per:                                                  # the uniform sampler draws its ids on the host
        th.cuda.set_sync_debug_mode("error")
    try:
        for i in range(3, 5):
            s1.learner.train_from_buffer(b1, 8, t_env=i, episode_num=0)
    finally:
        th.cuda.set_sync_debug_mode(0)
    th.manual_seed(77)
    np.random.seed(77)
    s2.learner.use_graphs = False
    for i in range(5):
        full = b2.sample(8)
        s2.learner.train(full, i, 0, weights=full.weights if per else None)
        if per:
            inter = s2.learner.intermediates(full)
            b2.update_priorities(full.ids, inter["td"].contiguous(), inter["mask"].reshape(8, -1).contiguous())
    th.cuda.synchronize()
    assert s1.learner.n_graph_replays >= 3
    assert_identical(s1, s2, "train_from_buffer against the loop by hand")
    if per:
        assert th.equal(b1.priorities, b2.priorities) and th.equal(b1.max_priority, b2.max_priority)


@pytest.mark.parametrize("optimizer", ["rmsprop", "adam"])
def test_launch_count_equals_hard_step_without_copy(optimizer):
    S, H = _pair(5, 8, 61, "qmix", 0.01, optimizer=optimizer, seed=5)
    counts = []
    for s in (S, H):
        s.learner.use_graphs = False
        s.learner.train(s.batch, 0, 0)
        th.cuda.synchronize()
        n0 = nat.lib().mal_launch_count()
        s.learner.train(s.batch, 1, 0)
        th.cuda.synchronize()
        counts.append(nat.lib().mal_launch_count() - n0)
    assert counts[0] == counts[1], counts


def test_interval_above_one_behaves_like_target_update_interval():
    new = _system(5, 8, 31, "qmix", None, seed=6, target_update_interval_or_tau=3)
    del new.args.target_update_interval
    old = _system(5, 8, 31, "qmix", None, seed=6, target_update_interval=3)
    episodes = [0, 1, 2, 3, 4, 5, 7, 8, 10]
    for i, ep in enumerate(episodes):
        for s in (new, old):
            s.learner.train(s.batch, t_env=i, episode_num=ep)
        th.cuda.synchronize()
        assert_identical(new, old, "episode %d" % ep)
        assert new.learner.last_target_update_episode == old.learner.last_target_update_episode
    assert new.learner.last_target_update_episode == 10
    assert len(new.logger.infos) == 3 and new.logger.infos == old.logger.infos


def test_update_targets_still_copies_in_soft_mode():
    S, _ = _pair(5, 8, 31, "qmix", 0.01, seed=7)
    S.learner.train(S.batch, 0, 0)
    S.learner.update_targets()
    th.cuda.synchronize()
    for tm, m in zip(_targets(S), _onlines(S)):
        assert all(th.equal(tp, p) for tp, p in zip(tm.parameters(), m.parameters()))


# ---------------------------------------------------------------------------------------------- stand-alone entry points
def _blend_check(tgt0, after, tau, got):
    """The soft entry's target against numpy's fp32 blend of the namesake's post-step parameters, bit for bit."""
    assert np.array_equal(got, R.blend_np(tgt0, after, tau))


def _buffers(P, n_agent, seed):
    rng = np.random.default_rng(seed)
    p = rng.standard_normal(P).astype(np.float32)
    t = (p + 0.1 * rng.standard_normal(P)).astype(np.float32)
    return rng, p, t


def _dev(x):
    return th.from_numpy(np.ascontiguousarray(x)).to(DEV)


@pytest.mark.parametrize("optimizer", ["rmsprop", "adam"])
@pytest.mark.parametrize("n_frozen,n_mixer,tau", [(0, 61000, 0.005), (30000, 61000, 0.3), (0, 0, 1.0)])
def test_clip_soft_with_denominator(optimizer, n_frozen, n_mixer, tau):
    """The *_soft clip entry against its namesake on identical inputs: parameters, gradient, optimiser state and scalars
    bit-identical (the namesake is checked against numpy by tests/test_data_parallel.py and tests/test_gpu_adam.py), and
    the targets equal to numpy's fp32 blend of the post-step parameters, the frozen prefix included."""
    n_agent = 40000
    P = n_agent + n_mixer
    rng, p, t = _buffers(P, n_agent, 7)
    state_n = nat.adam_state_floats(P) if optimizer == "adam" else P
    runs = []
    for soft in (False, True):
        agent, mixer = _dev(p[:n_agent]), (_dev(p[n_agent:]) if n_mixer else None)
        tagent, tmixer = _dev(t[:n_agent]), (_dev(t[n_agent:]) if n_mixer else None)
        state = th.zeros(state_n, device=DEV)
        scalars, scratch = th.zeros(64, device=DEV), th.zeros((P + 255) // 256, device=DEV)
        denom = th.tensor([37.0], device=DEV)
        g_rng = np.random.default_rng(3)
        st = nat.SoftTarget(tau, nat.ptr(tagent), nat.ptr(tmixer))
        for i in range(3):
            tgt0 = np.concatenate([tagent.cpu().numpy()] + ([tmixer.cpu().numpy()] if n_mixer else []))
            grad = _dev((g_rng.standard_normal(P) * 20).astype(np.float32))
            if optimizer == "adam":
                h = nat.AdamHyper(1e-3, 0.9, 0.999, 1e-8, 1e-4, 0.5)
                args = (nat.ptr(agent), n_agent, nat.ptr(mixer), n_mixer, nat.ptr(grad), nat.ptr(state), C.byref(h),
                        nat.ptr(scalars), nat.ptr(scratch), nat.ptr(denom), n_frozen)
                fn = "mal_clip_adam"
            else:
                args = (nat.ptr(agent), n_agent, nat.ptr(mixer), n_mixer, nat.ptr(grad), nat.ptr(state), 5e-4, 0.99,
                        1e-5, 0.5, nat.ptr(scalars), nat.ptr(scratch), nat.ptr(denom), n_frozen)
                fn = "mal_clip_rmsprop"
            if soft:
                nat.check(getattr(nat.lib(), fn + "_soft")(*args, C.byref(st), nat.current_stream()), fn + "_soft")
            else:
                nat.check(getattr(nat.lib(), fn)(*args, nat.current_stream()), fn)
            th.cuda.synchronize()
            after = np.concatenate([agent.cpu().numpy()] + ([mixer.cpu().numpy()] if n_mixer else []))
            tnow = np.concatenate([tagent.cpu().numpy()] + ([tmixer.cpu().numpy()] if n_mixer else []))
            if soft:
                _blend_check(tgt0, after, tau, tnow)
                if n_frozen:
                    assert np.array_equal(after[:n_frozen], p[:n_frozen]) and not np.array_equal(tnow[:n_frozen],
                                                                                                 t[:n_frozen])
            else:
                assert np.array_equal(tnow, t)
            runs.append([after, grad.cpu().numpy(), state.cpu().numpy(), scalars.cpu().numpy()])
    for a, b in zip(runs[:3], runs[3:]):
        for x, y in zip(a, b):
            assert np.array_equal(x, y)


@pytest.mark.parametrize("optimizer", ["rmsprop", "adam"])
@pytest.mark.parametrize("world", [2, 4, 8])
def test_peer_allreduce_soft_one_device_fake_peers(optimizer, world):
    """The two peer *_soft entries with W fake ranks on one device (raw peer pointers), against their namesakes and the
    numpy blend; W = 8 also has a frozen agent prefix."""
    n_agent, n_mixer = 3000, 5000
    P = n_agent + n_mixer
    n_frozen = n_agent if world == 8 else 0
    rng, p, t = _buffers(P, n_agent, world)
    bufs = []
    for r in range(world):
        tail = np.zeros(DP_TAIL, np.float32)
        tail[4] = 10.0 + r
        bufs.append(_dev(np.concatenate([(rng.standard_normal(P) * 5).astype(np.float32), tail])))
    ptrs = (C.c_void_p * world)(*[b.data_ptr() for b in bufs])
    tau = 0.25
    runs = []
    for soft in (False, True):
        agent, mixer, tagent, tmixer = _dev(p[:n_agent]), _dev(p[n_agent:]), _dev(t[:n_agent]), _dev(t[n_agent:])
        state = th.zeros(nat.adam_state_floats(P) if optimizer == "adam" else P, device=DEV)
        grad, tail_out = th.full((P,), 7.0, device=DEV), th.zeros(DP_TAIL, device=DEV)
        scalars, scratch = th.zeros(64, device=DEV), th.zeros((P + 255) // 256, device=DEV)
        st = nat.SoftTarget(tau, nat.ptr(tagent), nat.ptr(tmixer))
        h = nat.AdamHyper(1e-3, 0.9, 0.999, 1e-8, 0.0, 1.0)
        for i in range(2):
            tgt0 = np.concatenate([tagent.cpu().numpy(), tmixer.cpu().numpy()])
            head = (ptrs, world, nat.ptr(agent), n_agent, nat.ptr(mixer), n_mixer, nat.ptr(grad), nat.ptr(tail_out),
                    DP_TAIL, nat.ptr(state))
            if optimizer == "adam":
                args, fn = head + (C.byref(h), nat.ptr(scalars), nat.ptr(scratch), n_frozen), "mal_peer_allreduce_clip_adam"
            else:
                args = head + (5e-4, 0.99, 1e-5, 1.0, nat.ptr(scalars), nat.ptr(scratch), n_frozen)
                fn = "mal_peer_allreduce_clip_rmsprop"
            if soft:
                nat.check(getattr(nat.lib(), fn + "_soft")(*args, C.byref(st), nat.current_stream()), fn + "_soft")
            else:
                nat.check(getattr(nat.lib(), fn)(*args, nat.current_stream()), fn)
            th.cuda.synchronize()
            after = np.concatenate([agent.cpu().numpy(), mixer.cpu().numpy()])
            tnow = np.concatenate([tagent.cpu().numpy(), tmixer.cpu().numpy()])
            if soft:
                _blend_check(tgt0, after, tau, tnow)
            else:
                assert np.array_equal(tnow, t)
            runs.append([after, grad.cpu().numpy(), tail_out.cpu().numpy(), state.cpu().numpy(), scalars.cpu().numpy()])
    for a, b in zip(runs[:2], runs[2:]):
        for x, y in zip(a, b):
            assert np.array_equal(x, y)


# ---------------------------------------------------------------------------------------------- data-parallel
def _dp_worker(rank, world, port, out, nccl, fused, optimizer, tau):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dev = "cuda:%d" % (rank if nccl else 0)
    th.cuda.set_device(dev)
    if nccl:
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=th.device(dev))
    else:
        dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        from tests.gpu_helpers import seeded_system
        s = seeded_system(3, 8, 12, "qmix", True, seed=5, device=dev, data_parallel=True, learner_log_interval=0,
                          dp_fused=fused, optimizer=optimizer, target_update_interval_or_tau=tau)
        B = s.batch.batch_size
        lo, hi = rank * B // world, (rank + 1) * B // world
        for i in range(3):
            s.learner.train(s.batch[lo:hi], t_env=i, episode_num=i)
        th.cuda.synchronize()
        L = s.learner
        out.put((rank, np_params(s.mac.agent), np_params(L.mixer), np_params(L.target_mac.agent),
                 np_params(L.target_mixer), bool(getattr(L, "_dp_sym", None)), getattr(L, "_dp_sym_error", "")))
        dist.barrier()
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("nccl,fused,optimizer", [(False, False, "rmsprop"), (False, False, "adam"),
                                                  (True, False, "rmsprop"), (True, True, "adam")])
def test_dp_two_ranks_equals_full_batch(nccl, fused, optimizer):
    from tests.gpu_helpers import seeded_system
    if nccl and th.cuda.device_count() < 2:
        pytest.skip("needs two GPUs (gradient all-reduce over NCCL / NVLink)")
    tau = 0.2
    ctx = mp.get_context("spawn")
    out = ctx.SimpleQueue()
    port = _free_port()
    procs = [ctx.Process(target=_dp_worker, args=(r, 2, port, out, nccl, fused, optimizer, tau)) for r in range(2)]
    for p in procs:
        p.start()
    res = sorted([out.get(), out.get()], key=lambda r: r[0])
    for p in procs:
        p.join(300)
        assert p.exitcode == 0
    s = seeded_system(3, 8, 12, "qmix", True, seed=5, device="cuda:0", learner_log_interval=0, optimizer=optimizer,
                      target_update_interval_or_tau=tau)
    for i in range(3):
        s.learner.train(s.batch, t_env=i, episode_num=i)
    L = s.learner
    refs = [np_params(s.mac.agent), np_params(L.mixer), np_params(L.target_mac.agent), np_params(L.target_mixer)]
    for r in res:
        assert r[5] == fused, r[6]
        for got, ref, what in zip(r[1:5], refs, ("agent", "mixer", "target agent", "target mixer")):
            for k in ref:
                assert rel_err(got[k], ref[k]) <= TOL, "dp %s %s" % (what, k)
    for i in range(1, 5):                                 # replicas, targets included, are bit-identical
        assert all(np.array_equal(res[0][i][k], res[1][i][k]) for k in res[0][i])
