"""Independent Q-learners (`mixer: None`) on CPU: the hand-derived IQL reference against autograd, planning without a
device and the QLearner surface (q_learner.py:34-125 with self.mixer = None)."""
import ctypes as C

import numpy as np
import pytest
import torch as th

from oracle import np_oracle as O
from tests import iql_ref as R
from tests.helpers import rel_err

TOL = 1e-5


@pytest.fixture(scope="module")
def nat():
    from ma_league_b200 import _native
    _native.build()
    return _native


def _problem(N, A, OBS, S, B, TT, kind, seed):
    import ma_league_b200 as M
    from ma_league_b200.synthetic import make_scheme, synth_episode_data, fill_episode_batch
    rng = np.random.default_rng(seed)
    shapes = (O.agent_param_shapes if kind == "rnn" else O.dqn_agent_param_shapes)(OBS + A + N, A)
    ap, tp = O.init_params(shapes, rng), O.init_params(shapes, rng)
    scheme, groups, pre = make_scheme(N, A, OBS, S)
    eb = M.EpisodeBatch(scheme, groups, B, TT, preprocess=pre, device="cpu")
    data, lens = synth_episode_data(B, TT, N, A, OBS, S, th.Generator().manual_seed(seed))
    fill_episode_batch(eb, data, lens)
    return ap, tp, {k: v.numpy().copy() for k, v in eb.data.transition_data.items()}


def _norm_close(a, ref, what):
    assert np.shape(a) == np.shape(ref), (what, np.shape(a), np.shape(ref))
    assert rel_err(a, ref) <= TOL, (what, rel_err(a, ref))


def _close(a, ref, what):
    assert abs(float(a) - float(ref)) <= TOL * max(1.0, abs(float(ref))), (what, float(a), float(ref))


@pytest.mark.parametrize("double_q", [True, False])
@pytest.mark.parametrize("kind", ["rnn", "dqn"])
def test_oracle_equals_torch_port_autograd(kind, double_q):
    """Loss, every agent gradient, one RMSprop step and the logged statistics of the fp64 IQL reference against the torch
    port's op sequence (fp32, autograd backward, stock RMSprop), norm-wise per tensor."""
    N, A, OBS, S, B, TT = 3, 5, 8, 12, 4, 9
    lr, alpha, eps, gamma = 5e-4, 0.99, 1e-5, 0.99
    ap, tp, batch = _problem(N, A, OBS, S, B, TT, kind, seed=29 + (kind == "dqn"))
    ref = R.learner_forward_backward(ap, tp, batch, double_q=double_q, gamma=gamma, dtype=np.float64)
    T = TT - 1
    assert ref["q_tot"].shape == ref["targets"].shape == ref["td"].shape == (B, T, N)
    assert ref["mask"].shape == (B, T, 1) and ref["mixer_grads"] == {}
    # clip far above the gradient norm: p.grad after clip_grad_norm_ is the raw gradient
    port = R.torch_port_train(ap, tp, {k: th.from_numpy(v) for k, v in batch.items()}, double_q=double_q, gamma=gamma,
                              lr=lr, alpha=alpha, eps=eps, clip=1e9)
    _close(port["loss"], ref["loss"], "loss")
    for k, p in port["params"].items():
        _norm_close(port["grads"][k].numpy(), ref["agent_grads"][k], "grad " + k)
        new, sq = O.rmsprop_update(ap[k].astype(np.float64), ref["agent_grads"][k], np.zeros(ap[k].shape), lr, alpha, eps)
        _norm_close(p.detach().numpy() - ap[k], new - ap[k], "RMSprop step " + k)
        _norm_close(port["opt"].state[p]["square_avg"].numpy(), sq, "square_avg " + k)
    for k in ("td_error_abs", "q_taken_mean", "target_mean", "mask_sum"):
        _close(port["stats"][k], ref["stats"][k], k)
    assert port["stats"]["trained_steps"] == ref["stats"]["trained_steps"] == N * int(np.count_nonzero(ref["mask"]))
    assert float(ref["stats"]["mask_sum"]) == N * float(ref["mask"].sum())


def test_single_agent_iql_is_vdn():
    """With one agent the sum over agents is the identity: the IQL reference equals the shared oracle's VDN learner."""
    ap, tp, batch = _problem(1, 4, 8, 12, 3, 7, "rnn", seed=5)
    a = R.learner_forward_backward(ap, tp, batch, double_q=True, gamma=0.99, dtype=np.float64)
    b = O.learner_forward_backward(ap, tp, None, None, batch, mixer="vdn", double_q=True, gamma=0.99, dtype=np.float64)
    assert a["loss"] == b["loss"]
    for k in a["agent_grads"]:
        assert np.array_equal(a["agent_grads"][k], b["agent_grads"][k]), k
    for k in ("td_error_abs", "q_taken_mean", "target_mean", "mask_sum", "trained_steps"):
        assert a["stats"][k] == b["stats"][k], k


@pytest.mark.parametrize("kind", ["rnn", "dqn"])
@pytest.mark.parametrize("N", [3, 5, 20])
def test_plan_without_mixer(nat, N, kind):
    lib = nat.lib()
    A, OBS, S, B, TT = 6 + N, 8 + 8 * N, 16 * N, 32, 201
    k = nat.AGENT_RNN if kind == "rnn" else nat.AGENT_DQN
    b = nat.Batch(B, TT, N, A, OBS, S)
    plans = {}
    for mixer in (nat.MIXER_VDN, nat.MIXER_NONE):
        cfg = nat.LearnerCfg(mixer, 1, 0, 0, 0.99, 5e-4, 0.99, 1e-5, 10.0, 0, 0, 0, k)
        plan = nat.Plan()
        assert lib.mal_learner_plan(C.byref(b), C.byref(cfg), C.byref(plan)) == 0, lib.mal_last_error()
        plans[mixer] = plan
    iql, vdn = plans[nat.MIXER_NONE], plans[nat.MIXER_VDN]
    assert iql.n_agent_params == vdn.n_agent_params == lib.mal_agent_param_count_kind(k, OBS + A + N, A)
    assert iql.n_mixer_params == 0
    offs = [getattr(iql, n) for n in nat._PLAN_FIELDS if n not in ("total_bytes", "n_agent_params", "n_mixer_params",
                                                                    "partials_bytes")]
    assert all(0 <= o < iql.total_bytes and o % 256 == 0 for o in offs)
    # q_tot / target_q_tot / targets / td hold one value per agent; the mask one per transition
    per_agent = B * (TT - 1) * N * 4
    for lo, hi in (("q_tot", "target_q_tot"), ("target_q_tot", "targets"), ("targets", "td"), ("td", "d_a2")):
        assert getattr(iql, hi) - getattr(iql, lo) >= per_agent, lo
    assert iql.y1_tg == iql.y1_on and iql.a2_tg == iql.a2_on                       # no hypernet intermediates
    assert lib.mal_mixer_param_count(nat.MIXER_NONE, S, N, 32, 64) == 0


def test_mixer_forward_rejects_no_mixer(nat):
    lib = nat.lib()
    x = C.c_void_p(256)
    assert lib.mal_mixer_forward(nat.MIXER_NONE, 2, 3, 4, 8, 32, 64, None, x, None, 0, 0, None, x, None) != 0
    assert b"not recognised" in lib.mal_last_error()


def _cpu_learner(**over):
    import ma_league_b200 as M
    from ma_league_b200.synthetic import make_args, make_scheme
    N, A, OBS, S = 3, 9, 32, 48
    args = make_args(N, A, S, mixer=None, device="cpu", **over)
    scheme, groups, pre = make_scheme(N, A, OBS, S)
    eb = M.EpisodeBatch(scheme, groups, 2, 5, preprocess=pre, device="cpu")
    mac = M.mac_REGISTRY["basic"](eb.scheme, groups, args)

    class Log:
        def log_stat(self, *a): pass
        def info(self, *a): pass
    return M.learner_REGISTRY["q"](mac, eb.scheme, Log(), args, name="home"), mac


@pytest.mark.parametrize("agent", ["rnn", "dqn"])
def test_qlearner_without_mixer_builds_on_cpu(agent, tmp_path):
    from ma_league_b200 import _native as nat
    L, mac = _cpu_learner(agent=agent)
    assert L.mixer is None and L.target_mixer is None
    params = L.parameters()
    assert len(params) == len(list(mac.parameters())) > 0
    assert all(a is b for a, b in zip(params, mac.parameters()))
    L.build_optimizer()
    assert L.optimiser.flat_sq.numel() == sum(p.numel() for p in mac.parameters())
    cfg = L._cfg()
    assert cfg.mixer == nat.MIXER_NONE and cfg.embed == 0 and cfg.hyper_embed == 0 and cfg.freeze_agent == 0
    L.save_models(str(tmp_path))
    assert sorted(f.name for f in tmp_path.iterdir()) == ["home_qlearner_agent.th", "home_qlearner_opt.th"]
    L.load_models(str(tmp_path))


def test_frozen_agent_without_mixer_is_rejected():
    from ma_league_b200 import _native as nat
    L, mac = _cpu_learner(freeze_native=True)
    mac.freeze_agent_weights()
    with pytest.raises(nat.MalError, match="nothing|no parameter"):
        L.build_optimizer()
    L2, mac2 = _cpu_learner()
    L2.build_optimizer()
    mac2.freeze_agent_weights()                          # frozen after the optimiser was built: train() refuses
    with pytest.raises(nat.MalError, match="no parameter"):
        L2._cfg()
