"""TD(lambda) targets (`args.td_lambda`) on CPU: the fp64 reference of tests/td_lambda_ref.py against fp64 autograd of the
reference learner with build_td_lambda_targets, lambda = 0 against the 1-step oracle, the recursion's boundary cases, and
the host-side rejections and defaults of mal_learner_plan and QLearner."""
import ctypes as C
import math

import numpy as np
import pytest
import torch as th

from oracle import np_oracle as O
from tests import input_layout_ref as IL
from tests import td_lambda_ref as R
from tests.helpers import rel_err

TOL = 1e-9


@pytest.fixture(scope="module")
def nat():
    from ma_league_b200 import _native
    _native.build()
    return _native


def _problem(N, A, OBS, S, B, TT, kind, mixer, layers, seed, d_in=None):
    import ma_league_b200 as M
    from ma_league_b200.synthetic import make_scheme, synth_episode_data, fill_episode_batch
    rng = np.random.default_rng(seed)
    shapes = (O.agent_param_shapes if kind == "rnn" else O.dqn_agent_param_shapes)(d_in or OBS + A + N, A)
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


def _compare(ap, tp, mp, tmp, batch, **kw):
    ref = R.learner_forward_backward(ap, tp, mp, tmp, batch, **kw)
    tl, tag, tmg, tt = R.torch_loss_grads(ap, tp, mp, tmp, batch, **kw)
    assert abs(ref["loss"] - tl) <= TOL * abs(tl)
    assert rel_err(ref["targets"], tt) <= TOL
    for k in tag:
        assert rel_err(ref["agent_grads"][k], tag[k]) <= TOL, (k, rel_err(ref["agent_grads"][k], tag[k]))
    assert sorted(ref["mixer_grads"]) == sorted(tmg)
    for k in tmg:
        assert rel_err(ref["mixer_grads"][k], tmg[k]) <= TOL, (k, rel_err(ref["mixer_grads"][k], tmg[k]))
    return ref


@pytest.mark.parametrize("weighted", [False, True])
@pytest.mark.parametrize("lam", [0.0, 0.6, 1.0])
@pytest.mark.parametrize("mixer,layers,kind", [("qmix", 2, "rnn"), ("qmix", 1, "dqn"), ("vdn", 2, "rnn"), (None, 2, "rnn")])
def test_reference_equals_autograd_with_build_td_lambda_targets(mixer, layers, kind, lam, weighted):
    N, A, OBS, S, B, TT = 3, 5, 8, 12, 4, 9
    ap, tp, mp, tmp, batch = _problem(N, A, OBS, S, B, TT, kind, mixer, layers, seed=11 + layers + (kind == "dqn"))
    w = np.array([0.25, 1.0, 0.6, 0.9]) if weighted else None
    _compare(ap, tp, mp, tmp, batch, mixer=mixer, double_q=True, gamma=0.99, td_lambda=lam, weights=w)


def test_reference_switched_input_layout_and_single_q():
    N, A, OBS, S, B, TT = 3, 5, 8, 12, 3, 7
    cols = IL.input_columns(OBS, A, N, False, True)
    ap, tp, mp, tmp, batch = _problem(N, A, OBS, S, B, TT, "rnn", "qmix", 2, seed=7, d_in=len(cols))
    _compare(ap, tp, mp, tmp, batch, mixer="qmix", double_q=False, gamma=0.95, td_lambda=0.6, last_action=False)


@pytest.mark.parametrize("mixer", ["qmix", "vdn"])
def test_lambda_zero_equals_one_step_oracle(mixer):
    N, A, OBS, S, B, TT = 3, 5, 8, 12, 4, 9
    ap, tp, mp, tmp, batch = _problem(N, A, OBS, S, B, TT, "rnn", mixer, 2, seed=3)
    kw = dict(mixer=mixer, double_q=True, gamma=0.99)
    one = O.learner_forward_backward(ap, tp, mp, tmp, batch, dtype=np.float64, **kw)
    lam = R.learner_forward_backward(ap, tp, mp, tmp, batch, td_lambda=0.0, **kw)
    assert abs(lam["loss"] - one["loss"]) <= TOL * abs(one["loss"])
    for k in ("td_error_abs", "q_taken_mean", "target_mean", "mask_sum", "trained_steps"):
        assert abs(lam["stats"][k] - one["stats"][k]) <= TOL * max(1.0, abs(one["stats"][k])), k
    m = one["mask"] > 0
    assert np.allclose(lam["targets"][m], one["targets"][m], rtol=TOL, atol=0)
    assert np.all(lam["targets"][~m] == 0.0)                   # lambda = 0: m * (1-step target)
    for k in one["agent_grads"]:
        assert rel_err(lam["agent_grads"][k], one["agent_grads"][k]) <= TOL, k
    for k in one["mixer_grads"]:
        assert rel_err(lam["mixer_grads"][k], one["mixer_grads"][k]) <= TOL, k


def test_recursion_boundaries():
    """Terminated inside the window: the padding contributes nothing and the returns equal those of the truncated episode.
    Not terminated and shorter than the window: the return bootstraps from the window's last row, as the formula says."""
    rng = np.random.default_rng(0)
    T, gamma, lam = 12, 0.9, 0.7
    tq = rng.normal(size=(2, T, 1))
    r = rng.normal(size=(2, T, 1))
    term = np.zeros((2, T, 1))
    mask = np.zeros((2, T, 1))
    term[0, 6] = 1.0
    mask[0, :7] = 1.0                                          # episode 0: 7 steps, terminated on its last
    mask[1, :5] = 1.0                                          # episode 1: 5 steps, never terminated
    R_ = R.lambda_returns(tq, r, term, mask, gamma, lam)
    tr = R.lambda_returns(tq[:1, :7], r[:1, :7], term[:1, :7], mask[:1, :7], gamma, lam)
    assert np.allclose(R_[0, :7], tr[0], rtol=1e-12, atol=1e-12)
    assert np.all(R_[0, 7:] == 0.0)
    want = np.zeros(T + 1)
    want[T] = tq[1, T - 1, 0]
    for t in range(T - 1, -1, -1):
        want[t] = lam * gamma * want[t + 1] + mask[1, t, 0] * (r[1, t, 0] + (1 - lam) * gamma * tq[1, t, 0])
    assert np.allclose(R_[1, :, 0], want[:T], rtol=1e-12, atol=0)
    assert abs(R_[1, 4, 0] - (r[1, 4, 0] + (1 - lam) * gamma * tq[1, 4, 0] + (lam * gamma) ** (T - 4) * tq[1, T - 1, 0])) < 1e-12


def _cfg(nat, returns=None, lam=None):
    cfg = nat.LearnerCfg(nat.MIXER_QMIX2, 1, 32, 64, 0.99, 5e-4, 0.99, 1e-5, 10.0, 0)
    if returns is not None:
        cfg.returns = returns
    if lam is not None:
        cfg.td_lambda = lam
    return cfg


def test_plan_zero_tail_default_and_rejections(nat):
    lib = nat.lib()
    b = nat.Batch(32, 201, 5, 11, 48, 80)
    plan, ref = nat.Plan(), nat.Plan()
    cfg = _cfg(nat)
    assert cfg.returns == nat.RETURNS_ONE_STEP and cfg.td_lambda == 0.0    # ten positional values: a zeroed tail
    assert lib.mal_learner_plan(C.byref(b), C.byref(cfg), C.byref(ref)) == 0
    for lam in (0.0, 0.6, 1.0):                                # no new workspace: the plan is the 1-step plan
        assert lib.mal_learner_plan(C.byref(b), C.byref(_cfg(nat, nat.RETURNS_TD_LAMBDA, lam)), C.byref(plan)) == 0
        assert all(getattr(plan, n) == getattr(ref, n) for n in nat._PLAN_FIELDS)
    assert lib.mal_learner_plan(C.byref(b), C.byref(_cfg(nat, 2, 0.5)), C.byref(plan)) != 0
    assert b"returns 2 not recognised" in lib.mal_last_error()
    for lam in (-0.01, 1.01, math.nan, math.inf, -math.inf):
        assert lib.mal_learner_plan(C.byref(b), C.byref(_cfg(nat, nat.RETURNS_TD_LAMBDA, lam)), C.byref(plan)) != 0
        assert b"td_lambda" in lib.mal_last_error()


def _cpu_learner(**over):
    from tests.gpu_helpers import build_system
    return build_system(3, 9, 32, 48, 4, 6, "qmix", True, device="cpu", **over).learner


def test_qlearner_fills_and_validates_td_lambda(nat):
    L = _cpu_learner()
    cfg = L._cfg()
    assert cfg.returns == nat.RETURNS_ONE_STEP and cfg.td_lambda == 0.0   # key absent
    L.args.td_lambda = None
    assert L._cfg().returns == nat.RETURNS_ONE_STEP
    for v in (0, 0.6, 1, np.float32(0.25)):
        L.args.td_lambda = v
        cfg = L._cfg()
        assert cfg.returns == nat.RETURNS_TD_LAMBDA and cfg.td_lambda == np.float32(v)
    for v in (-0.1, 1.5, float("nan"), float("inf"), "0.6", True, [0.6]):
        L.args.td_lambda = v
        with pytest.raises(nat.MalError, match="td_lambda"):
            L._cfg()
