"""Prioritized episode replay on CPU: the per-episode weighted-gradient reference against autograd of the weighted loss
(fp64), the reference sampler / update rules, the host-only argument queries, the rejections and the exports."""
import ctypes as C

import numpy as np
import pytest
import torch as th

from oracle import np_oracle as O
from tests import per_ref as R
from tests.helpers import rel_err

TOL = 1e-9


@pytest.fixture(scope="module")
def nat():
    from ma_league_b200 import _native
    _native.build()
    return _native


def _problem(N, A, OBS, S, B, TT, kind, mixer, layers, seed):
    import ma_league_b200 as M
    from ma_league_b200.synthetic import make_scheme, synth_episode_data, fill_episode_batch
    rng = np.random.default_rng(seed)
    shapes = (O.agent_param_shapes if kind == "rnn" else O.dqn_agent_param_shapes)(OBS + A + N, A)
    ap, tp = O.init_params(shapes, rng), O.init_params(shapes, rng)
    mp = tmp = None
    if mixer == "qmix":
        ms = O.qmix_param_shapes(S, N, 8, 16, layers)
        mp, tmp = O.init_params(ms, rng), O.init_params(ms, rng)
    scheme, groups, pre = make_scheme(N, A, OBS, S)
    eb = M.EpisodeBatch(scheme, groups, B, TT, preprocess=pre, device="cpu")
    data, lens = synth_episode_data(B, TT, N, A, OBS, S, th.Generator().manual_seed(seed), var_len=True)
    fill_episode_batch(eb, data, lens)
    return ap, tp, mp, tmp, {k: v.numpy().copy() for k, v in eb.data.transition_data.items()}


@pytest.mark.parametrize("double_q", [True, False])
@pytest.mark.parametrize("kind", ["rnn", "dqn"])
@pytest.mark.parametrize("mixer,layers", [("qmix", 2), ("qmix", 1), ("vdn", 2), (None, 2)])
def test_per_episode_reference_equals_weighted_autograd(mixer, layers, kind, double_q):
    N, A, OBS, S, B, TT = 3, 5, 8, 12, 4, 9
    ap, tp, mp, tmp, batch = _problem(N, A, OBS, S, B, TT, kind, mixer, layers, seed=41 + layers + (kind == "dqn"))
    w = np.array([0.25, 1.0, 0.6, 0.9])
    kw = dict(mixer=mixer, double_q=double_q, gamma=0.99)
    loss, ag, mg = R.weighted_learner(ap, tp, mp, tmp, batch, w, **kw)
    tl, tag, tmg = R.torch_weighted(ap, tp, mp, tmp, batch, w, **kw)
    assert abs(loss - tl) <= TOL * abs(tl)
    for k in tag:
        assert rel_err(ag[k], tag[k]) <= TOL, (k, rel_err(ag[k], tag[k]))
    assert sorted(mg) == sorted(tmg)
    for k in tmg:
        assert rel_err(mg[k], tmg[k]) <= TOL, (k, rel_err(mg[k], tmg[k]))
    # weights of one: the unweighted oracle of the whole batch
    if mixer is not None:
        full = O.learner_forward_backward(ap, tp, mp, tmp, batch, dtype=np.float64, **kw)
        l1, g1, _ = R.weighted_learner(ap, tp, mp, tmp, batch, np.ones(B), **kw)
        assert abs(l1 - full["loss"]) <= TOL * abs(full["loss"])
        for k in g1:
            assert rel_err(g1[k], full["agent_grads"][k]) <= TOL, k


def test_input_layout_switch_weighted():
    N, A, OBS, S, B, TT = 3, 5, 8, 12, 3, 7
    ap, tp, mp, tmp, batch = _problem(N, A, OBS, S, B, TT, "rnn", "qmix", 2, seed=7)
    from tests import input_layout_ref as IL
    cols = IL.input_columns(OBS, A, N, False, True)
    ap = dict(ap, **{"fc1.weight": ap["fc1.weight"][:, cols]})
    tp = dict(tp, **{"fc1.weight": tp["fc1.weight"][:, cols]})
    w = np.array([0.5, 0.125, 1.0])
    kw = dict(mixer="qmix", double_q=True, gamma=0.99, last_action=False, agent_id=True)
    loss, ag, _ = R.weighted_learner(ap, tp, mp, tmp, batch, w, **kw)
    tl, tag, _ = R.torch_weighted(ap, tp, mp, tmp, batch, w, **kw)
    assert abs(loss - tl) <= TOL * abs(tl)
    for k in tag:
        assert rel_err(ag[k], tag[k]) <= TOL, k


def test_reference_sampler_and_update():
    p = np.array([1.0, 0.0, 3.0, 2.0, 2.0], dtype=np.float32)
    ids, w, near = R.sample(p, 5, np.array([0.25, 0.25, 0.25, 0.25], dtype=np.float32), beta=1.0)
    # total 8, points 0.5, 2.5, 4.5, 6.5 -> prefix sums 1, 1, 4, 6, 8: first prefix > point
    assert ids.tolist() == [0, 2, 3, 4] and not near.any()
    assert np.allclose(w, [0.0, 0.0, 0.0, 0.0])          # p_min = 0: every weight (0 / p)^beta
    ids, w, near = R.sample(p, 5, np.array([0.0, 0.0], dtype=np.float32), beta=0.5)
    assert ids.tolist() == [0, 3] and near.tolist() == [False, True]     # x = 4 sits on a boundary
    td = np.array([[[1.0], [-3.0]], [[2.0], [0.0]], [[5.0], [5.0]]])
    mask = np.array([[1.0, 1.0], [1.0, 0.0], [1.0, 1.0]])
    newp, mx = R.update(np.ones(6), 1.0, np.array([4, 1, 4]), td, mask, alpha=0.5, eps=0.0)
    assert newp[1] == 2.0 ** 0.5 and newp[4] == 5.0 ** 0.5 and mx == 5.0 ** 0.5   # batch index 2 wins slot 4
    assert newp[0] == 1.0


def test_argument_queries_without_device(nat):
    L = nat.lib()
    assert L.mal_per_sample_check(5000, 32, 0.4) == 0
    assert L.mal_per_sample_check(0, 32, 0.4) != 0 and b"no episode" in L.mal_last_error()
    assert L.mal_per_sample_check(10, 0, 0.4) != 0
    for bad in (-0.1, float("nan"), float("inf")):
        assert L.mal_per_sample_check(10, 4, bad) != 0 and b"beta" in L.mal_last_error()
        assert L.mal_per_update_check(4, 200, 1, bad, 1e-6) != 0 and b"alpha" in L.mal_last_error()
        assert L.mal_per_update_check(4, 200, 1, 0.6, bad) != 0 and b"eps" in L.mal_last_error()
    assert L.mal_per_update_check(4, 200, 5, 0.6, 1e-6) == 0
    assert L.mal_per_update_check(0, 200, 1, 0.6, 1e-6) != 0
    # the entries reject the same arguments before touching any pointer
    x = C.c_void_p(256)
    assert L.mal_per_sample(x, 0, 4, 0.4, None, 0, 0, x, x, None, None) != 0
    assert L.mal_per_update(x, x, 4, 10, 1, x, -1.0, 0.0, x, 10, x, None) != 0


def test_weighted_batch_rejected_in_unnormalized_mode(nat):
    L = nat.lib()
    b = nat.Batch(32, 201, 5, 11, 48, 80)
    b.weight = nat.Field(256, 1, 0)
    cfg = nat.LearnerCfg(nat.MIXER_QMIX2, 1, 32, 64, 0.99, 5e-4, 0.99, 1e-5, 10.0, 0, 1)
    plan = nat.Plan()
    assert L.mal_learner_plan(C.byref(b), C.byref(cfg), C.byref(plan)) != 0
    assert b"data-parallel" in L.mal_last_error()
    cfg.unnormalized = 0
    assert L.mal_learner_plan(C.byref(b), C.byref(cfg), C.byref(plan)) == 0


def test_exports_and_host_buffer_rejections(nat):
    import ma_league_b200 as M
    from ma_league_b200.components.replay_buffers import PrioritizedReplayBuffer, ReplayBuffer
    from ma_league_b200.synthetic import make_scheme
    assert M.PrioritizedReplayBuffer is PrioritizedReplayBuffer and issubclass(PrioritizedReplayBuffer, ReplayBuffer)
    for name in ("mal_per_sample", "mal_per_sample_check", "mal_per_update", "mal_per_update_check"):
        assert name in nat.EXPORTS and hasattr(nat.lib(), name)
    scheme, groups, pre = make_scheme(3, 9, 32, 48)
    with pytest.raises(nat.MalError, match="device-resident"):
        PrioritizedReplayBuffer(scheme, groups, 16, 5, preprocess=pre, device="cpu")
    for kw in (dict(alpha=-1.0), dict(beta=float("nan")), dict(eps=float("inf"))):
        with pytest.raises(nat.MalError, match="finite"):
            PrioritizedReplayBuffer(scheme, groups, 16, 5, preprocess=pre, device="cpu", **kw)


def test_beta_schedule():
    from ma_league_b200.components.replay_buffers.prioritized_replay_buffer import PrioritizedReplayBuffer
    buf = PrioritizedReplayBuffer.__new__(PrioritizedReplayBuffer)
    buf.beta, buf.beta_anneal_t = 0.4, 1000
    assert buf.beta_at(0) == 0.4 and abs(buf.beta_at(500) - 0.7) < 1e-12 and buf.beta_at(5000) == 1.0
    buf.beta_anneal_t = None
    assert buf.beta_at(5000) == 0.4
