"""Prioritized episode replay on the B200: the sampler and the priority update against tests/per_ref.py, the
importance-weighted learner step against the fp64 per-episode oracle, `weights = ones` against the unweighted step, and
the `train_from_buffer` loop (no host sync, graph replay, two extra launches, equal to the loop done by hand)."""
import ctypes as C

import numpy as np
import pytest
import torch as th

import ma_league_b200 as M
from ma_league_b200 import _native as nat
from ma_league_b200.synthetic import synth_episode_data, fill_episode_batch
from tests import per_ref as R
from tests.gpu_helpers import build_system, np_params, np_batch
from tests.helpers import rel_err

pytestmark = pytest.mark.gpu
DEV = "cuda"


def _sample(p, n, B, beta, u=None):
    ids = th.empty(B, dtype=th.long, device=DEV)
    w = th.empty(B, dtype=th.float32, device=DEV)
    adv = C.c_uint64(0)
    nat.check(nat.lib().mal_per_sample(nat.ptr(p), n, B, beta, nat.ptr(u), 0, 0, nat.ptr(ids), nat.ptr(w), C.byref(adv),
                                       nat.current_stream()), "mal_per_sample")
    return ids, w


def _priorities(kind, n, gen):
    if kind == "equal":
        return th.full((n,), 0.75)
    if kind == "spread":                                   # several orders of magnitude, a few zeros
        p = 10.0 ** (th.rand(n, generator=gen) * 6 - 3)
        p[th.randperm(n, generator=gen)[: n // 50]] = 0.0
        if n > 0 and float(p.sum()) == 0.0:
            p[0] = 1.0
        return p
    return th.rand(n, generator=gen) + 0.01


@pytest.mark.parametrize("kind", ["equal", "spread", "uniform"])
@pytest.mark.parametrize("n,B", [(1, 32), (32, 32), (5000, 32), (5000, 1024), (10 ** 6, 128)])
def test_sampler_against_reference(n, B, kind):
    gen = th.Generator().manual_seed(n + B)
    p = _priorities(kind, n, gen).to(DEV)
    u = th.rand(B, generator=gen).to(DEV)
    beta = 0.4
    ids, w = _sample(p, n, B, beta, u)
    ids2, w2 = _sample(p, n, B, beta, u)
    assert th.equal(ids, ids2) and th.equal(w, w2)             # fixed reduction and scan order
    rid, rw, near = R.sample(p.cpu().numpy(), n, u.cpu().numpy(), beta)
    got = ids.cpu().numpy()
    bad = (got != rid) & ~near
    assert not bad.any(), (np.nonzero(bad)[0][:8], got[bad][:8], rid[bad][:8])
    assert (got >= 0).all() and (got < n).all()
    agree = got == rid
    assert np.all(np.abs(w.cpu().numpy()[agree] - rw[agree]) <= 1e-6 * np.maximum(1.0, rw[agree]))
    assert (p[ids] > 0).all()


def test_sampler_philox_matches_torch_rand_and_generator():
    gen = th.Generator().manual_seed(3)
    p = _priorities("spread", 5000, gen).to(DEV)
    scheme_sys = build_system(3, 9, 32, 48, 4, 5, "vdn", True)
    buf = M.PrioritizedReplayBuffer(scheme_sys.scheme, scheme_sys.groups, 5000, 5, preprocess=scheme_sys.pre, device=DEV)
    buf.priorities.copy_(p)
    buf.episodes_in_buffer = 5000
    g = th.cuda.default_generators[th.cuda.current_device()]
    for B in (32, 1024, 3000):
        th.manual_seed(123)
        u = th.rand(B, device=DEV)
        off_ref = g.get_offset()
        th.manual_seed(123)
        ids, w = buf.sample_ids(B, beta=0.6)
        assert g.get_offset() == off_ref, B
        ids_u, w_u = buf.sample_ids(B, beta=0.6, u=u)
        assert th.equal(ids, ids_u) and th.equal(w, w_u), B


def test_sampler_frequencies():
    """Fixed seed: over many draws each slot is drawn in proportion to p_i / total."""
    gen = th.Generator().manual_seed(11)
    p = (th.rand(17, generator=gen) * 4 + 0.05).to(DEV)
    B = 1 << 16
    counts = np.zeros(17)
    th.manual_seed(5)
    g = th.cuda.default_generators[th.cuda.current_device()]
    for _ in range(8):
        u = th.rand(B, device=DEV)
        ids, _ = _sample(p, 17, B, 0.5, u)
        counts += np.bincount(ids.cpu().numpy(), minlength=17)
    freq = counts / counts.sum()
    ref = (p / p.sum()).cpu().numpy()
    assert np.abs(freq - ref).max() < 2e-4, np.abs(freq - ref).max()      # stratified: error ~ 1 / (8 B) per slot
    assert g.get_offset() > 0


def _per_buffer(s, size, TT, alpha=0.6, beta=0.4, eps=1e-6, **kw):
    return M.PrioritizedReplayBuffer(s.scheme, s.groups, size, TT, preprocess=s.pre, device=DEV, alpha=alpha, beta=beta,
                                     eps=eps, **kw)


def _fill(s, buf, n_batches, bs, TT, seed, N, short=None):
    A, OBS, S = 6 + N, 8 + 8 * N, 16 * N
    gen = th.Generator().manual_seed(seed)
    for _ in range(n_batches):
        data, lens = synth_episode_data(bs, TT, N, A, OBS, S, gen, var_len=True, device=DEV)
        if short is not None:
            lens = th.clamp(lens, max=short)
        data["terminated"].zero_()
        data["terminated"][th.arange(bs), lens - 1] = 1
        buf.insert_episode_batch(fill_episode_batch(M.EpisodeBatch(s.scheme, s.groups, bs, TT, preprocess=s.pre, device=DEV),
                                                    data, lens))


def test_priority_update_and_insertion():
    s = build_system(3, 9, 32, 48, 4, 6, "qmix", True)
    buf = _per_buffer(s, 10, 6, alpha=0.7, eps=1e-3)
    _fill(s, buf, 1, 6, 6, 1, 3)
    assert th.equal(buf.priorities[:6], th.ones(6, device=DEV)) and float(buf.priorities[6:].abs().sum()) == 0
    gen = th.Generator().manual_seed(2)
    B, T = 9, 5
    for Q in (1, 3):
        ids = th.tensor([4, 1, 4, 0, 5, 1, 1, 2, 4], device=DEV)
        td = (th.randn(B, T, Q, generator=gen) * 3).to(DEV)
        mask = (th.rand(B, T, generator=gen) > 0.3).float().to(DEV)
        mask[3] = 0.0                                           # an episode without live transitions: eps^alpha
        p0, m0 = buf.priorities.cpu().numpy(), float(buf.max_priority)
        buf.update_priorities(ids, td, mask)
        rp, rm = R.update(p0, m0, ids.cpu().numpy(), td.cpu().numpy(), mask.cpu().numpy(), 0.7, 1e-3)
        assert np.allclose(buf.priorities.cpu().numpy(), rp, rtol=2e-6, atol=0)
        assert abs(float(buf.max_priority) - rm) <= 2e-6 * rm
    # wrap-around insert: 4 slots at the end and 2 at the start get the running maximum
    buf.max_priority.fill_(3.5)
    before = buf.priorities.clone()
    _fill(s, buf, 1, 6, 6, 3, 3)
    assert buf.buffer_index == 2
    assert th.equal(buf.priorities[6:], th.full((4,), 3.5, device=DEV))
    assert th.equal(buf.priorities[:2], th.full((2,), 3.5, device=DEV))
    assert th.equal(buf.priorities[2:6], before[2:6])


def _system(N, B, TT, mixer, layers=2, agent="rnn", last_action=True, seed=0, clip=1e9):
    A, OBS, S = 6 + N, 8 + 8 * N, 16 * N
    th.manual_seed(seed)
    s = build_system(N, A, OBS, S, B, TT, mixer, True, hypernet_layers=layers, clip=clip, agent=agent,
                     obs_last_action=last_action)
    gen = th.Generator().manual_seed(seed + 1)
    nets = list(s.learner.target_mac.parameters()) + (list(s.learner.target_mixer.parameters()) if mixer else [])
    with th.no_grad():
        for p in nets:
            p.add_(0.05 * th.randn(p.shape, generator=gen).to(DEV))
    data, lens = synth_episode_data(B, TT, N, A, OBS, S, gen, var_len=True, device=DEV)
    lens[0] = TT - 1
    s["batch"] = fill_episode_batch(M.EpisodeBatch(s.scheme, s.groups, B, TT, preprocess=s.pre, device=DEV), data, lens)
    s["w"] = (th.rand(B, generator=gen) * 0.9 + 0.1).to(DEV)
    return s


def _ref_grad(s, w, mixer, last_action):
    L = s.learner
    pm = np_params(L.mixer) if mixer else None
    ptm = np_params(L.target_mixer) if mixer else None
    loss, ag, mg = R.weighted_learner(np_params(s.mac.agent), np_params(L.target_mac.agent), pm, ptm, np_batch(s.batch),
                                      w.cpu().numpy().astype(np.float64), mixer=mixer, double_q=True, gamma=s.args.gamma,
                                      last_action=last_action)
    return loss, np.concatenate([v.ravel() for v in list(ag.values()) + list(mg.values())])


CASES = [(3, 4, 201, "qmix", 2, "rnn", True), (5, 4, 201, "qmix", 1, "rnn", True), (10, 2, 201, "vdn", 2, "rnn", True),
         (5, 4, 201, None, 2, "rnn", True), (5, 4, 201, "qmix", 2, "dqn", True), (3, 4, 201, "qmix", 2, "rnn", False),
         (20, 3, 21, "qmix", 2, "rnn", True), (20, 3, 21, None, 2, "dqn", True)]


@pytest.mark.parametrize("N,B,TT,mixer,layers,agent,last_action", CASES)
def test_weighted_step_against_oracle(N, B, TT, mixer, layers, agent, last_action):
    s = _system(N, B, TT, mixer, layers, agent, last_action, seed=N + B)
    L = s.learner
    loss, g_ref = _ref_grad(s, s.w, mixer, last_action)
    L.use_graphs = False
    L.train(s.batch, 0, 0, weights=s.w)
    th.cuda.synchronize()
    assert rel_err(L._grad.cpu().numpy(), g_ref) <= 1e-4, rel_err(L._grad.cpu().numpy(), g_ref)
    got_loss = float(L.scalars()[nat.SC_LOSS])
    assert abs(got_loss - loss) <= 1e-5 * abs(loss), (got_loss, loss)


def test_two_chained_weighted_steps_parameters_and_square_avg():
    from oracle import np_oracle as O
    s = _system(5, 4, 201, "qmix", seed=21)
    L, a = s.learner, s.args
    p = np.concatenate([v.ravel() for v in list(np_params(s.mac.agent).values()) + list(np_params(L.mixer).values())])
    p = p.astype(np.float64)
    sq = L.optimiser.flat_sq.cpu().numpy().astype(np.float64)
    ws = [s.w, s.w.flip(0) * 0.5]
    for w in ws:
        _, g = _ref_grad(s, w, "qmix", True)              # at the parameters the learner holds now
        L.train(s.batch, 0, 0, weights=w)
        th.cuda.synchronize()
        p, sq = O.rmsprop_update(p, g, sq, a.lr, a.optim_alpha, a.optim_eps)
    got = np.concatenate([v.ravel() for v in list(np_params(s.mac.agent).values()) + list(np_params(L.mixer).values())])
    assert rel_err(got, p) <= 1e-5
    assert rel_err(L.optimiser.flat_sq.cpu().numpy(), sq) <= 1e-4


@pytest.mark.parametrize("mixer", ["qmix", "vdn", None])
def test_weights_of_one_are_bit_identical_to_unweighted(mixer):
    outs = []
    for weighted in (False, True):
        s = _system(5, 8, 61, mixer, seed=4, clip=10.0)
        ones = th.ones(8, device=DEV)
        for i in range(4):                                # eager, capture, replay, replay
            s.learner.train(s.batch, i, 0, weights=ones if weighted else None)
        th.cuda.synchronize()
        assert s.learner.n_graph_replays >= 2
        nets = [s.mac.agent] + ([s.learner.mixer] if mixer else [])
        outs.append(([v.clone() for n in nets for v in n.state_dict().values()],
                     s.learner.optimiser.flat_sq.clone(), s.learner.scalars()[:8].clone()))
    for x, y in zip(outs[0][0], outs[1][0]):
        assert th.equal(x, y)
    assert th.equal(outs[0][1], outs[1][1]) and th.equal(outs[0][2], outs[1][2])


def _loop_system(seed, per=True, N=5, size=64, TT=31):
    s = _system(N, 8, TT, "qmix", seed=seed, clip=10.0)
    buf = _per_buffer(s, size, TT) if per else M.ReplayBuffer(s.scheme, s.groups, size, TT, preprocess=s.pre, device=DEV)
    _fill(s, buf, size // 8, 8, TT, seed + 7, N, short=20)
    return s, buf


@pytest.mark.parametrize("truncate", [False, True])
def test_train_from_buffer_equals_manual_loop(truncate):
    s1, b1 = _loop_system(9)
    s2, b2 = _loop_system(9)
    th.manual_seed(77)
    for i in range(4):
        s1.learner.train_from_buffer(b1, 8, t_env=i, episode_num=0, truncate=truncate)
    th.manual_seed(77)
    s2.learner.use_graphs = False
    for i in range(4):
        full = b2.sample(8)
        smp = full[:, :int(full.max_t_filled())] if truncate else full
        s2.learner.train(smp, i, 0, weights=full.weights)
        inter = s2.learner.intermediates(smp)
        b2.update_priorities(full.ids, inter["td"].contiguous(), inter["mask"].reshape(8, -1).contiguous())
    th.cuda.synchronize()
    assert s1.learner.n_graph_replays >= (0 if truncate else 2)
    for x, y in zip(s1.mac.agent.state_dict().values(), s2.mac.agent.state_dict().values()):
        assert th.equal(x, y)
    for x, y in zip(s1.learner.mixer.state_dict().values(), s2.learner.mixer.state_dict().values()):
        assert th.equal(x, y)
    assert th.equal(b1.priorities, b2.priorities) and th.equal(b1.max_priority, b2.max_priority)
    assert not th.equal(b1.priorities, th.ones_like(b1.priorities))


def test_train_from_buffer_no_sync_graph_replay_and_launches():
    counts = {}
    for per in (False, True):
        s, buf = _loop_system(13, per=per)
        L = s.learner
        np.random.seed(0)
        for i in range(3):                                  # eager, capture, replay; the first step logs
            L.train_from_buffer(buf, 8, t_env=i, episode_num=0)
        th.cuda.synchronize()
        r0, n0 = L.n_graph_replays, nat.lib().mal_launch_count()
        if per:
            th.cuda.set_sync_debug_mode("error")
        try:
            for i in range(5):
                L.train_from_buffer(buf, 8, t_env=3 + i, episode_num=0)
        finally:
            th.cuda.set_sync_debug_mode(0)
        th.cuda.synchronize()
        assert L.n_graph_replays - r0 == 5
        counts[per] = (nat.lib().mal_launch_count() - n0) / 5
    assert counts[True] <= counts[False] + 2, counts


def test_rejections():
    s, buf = _loop_system(3)
    s.args.data_parallel = True
    with pytest.raises(nat.MalError, match="data_parallel"):
        s.learner.train_from_buffer(buf, 8, 0, 0)
    with pytest.raises(nat.MalError, match="data_parallel"):
        s.learner.train(s.batch, 0, 0, weights=s.w)
    s.args.data_parallel = False
    with pytest.raises(nat.MalError, match="float32"):
        s.learner.train(s.batch, 0, 0, weights=th.ones(3, device=DEV))
    with pytest.raises(nat.MalError, match="device-resident"):
        M.PrioritizedReplayBuffer(s.scheme, s.groups, 16, 31, preprocess=s.pre, device="cpu")
    empty = _per_buffer(s, 16, 31)
    with pytest.raises(nat.MalError, match="no episode"):
        empty.sample(4)
