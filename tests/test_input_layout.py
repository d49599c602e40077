"""Agent inputs with obs_last_action / obs_agent_id switched off: planning, input assembly and the reference, on CPU."""
import ctypes as C

import numpy as np
import pytest
import torch as th

from oracle import np_oracle as O
from tests.helpers import assert_close
from tests.input_layout_ref import LAYOUTS, build_inputs, d_in, learner_forward_backward, torch_loss_grads


@pytest.fixture(scope="module")
def nat():
    from ma_league_b200 import _native
    _native.build()
    return _native


@pytest.mark.parametrize("kind", ["rnn", "dqn"])
@pytest.mark.parametrize("N", [3, 5, 20])
def test_plan_parameter_count_follows_the_input_switches(nat, N, kind):
    lib = nat.lib()
    A, OBS, S = 6 + N, 8 + 8 * N, 16 * N
    k = nat.AGENT_RNN if kind == "rnn" else nat.AGENT_DQN
    b = nat.Batch(32, 201, N, A, OBS, S)
    plan = nat.Plan()
    counts = {}
    for last, aid in LAYOUTS:
        cfg = nat.LearnerCfg(nat.MIXER_QMIX2, 1, 32, 64, 0.99, 5e-4, 0.99, 1e-5, 10.0, 0, 0, 0, k,
                             nat.agent_input_flags(last, aid))
        assert lib.mal_learner_plan(C.byref(b), C.byref(cfg), C.byref(plan)) == 0
        assert plan.n_agent_params == lib.mal_agent_param_count_kind(k, d_in(OBS, A, N, last, aid), A)
        counts[(last, aid)] = plan.n_agent_params
    # a zero-filled agent_input (callers that predate the field) is the default layout
    cfg = nat.LearnerCfg(nat.MIXER_QMIX2, 1, 32, 64, 0.99, 5e-4, 0.99, 1e-5, 10.0, 0, 0, 0, k)
    assert lib.mal_learner_plan(C.byref(b), C.byref(cfg), C.byref(plan)) == 0
    assert plan.n_agent_params == counts[(True, True)]
    if N == 5 and kind == "rnn":
        assert plan.n_agent_params == 29835
    cfg.agent_input = 4
    assert lib.mal_learner_plan(C.byref(b), C.byref(cfg), C.byref(plan)) != 0
    assert b"agent_input" in lib.mal_last_error()


def test_step_argument_bits_are_checked(nat):
    lib = nat.lib()
    x = th.zeros(64)
    # dense together with agent-input bits, and unknown bits, are refused before anything is launched
    for bits in (3, 8):
        assert lib.mal_agent_step(x.data_ptr(), 1, 1, 4, 2, bits, x.data_ptr(), 4, None, 0, None, x.data_ptr(),
                                  x.data_ptr(), None, None) != 0
        assert b"dense_input" in lib.mal_last_error()
        assert lib.mal_dqn_step(x.data_ptr(), 1, 1, 4, 2, bits, x.data_ptr(), 4, None, 0, x.data_ptr(), None, None) != 0


def _mac(N, A, OBS, S, last, aid, B=3, TT=4):
    import ma_league_b200 as M
    from ma_league_b200.synthetic import make_args, make_scheme, synth_episode_data, fill_episode_batch
    args = make_args(N, A, S, device="cpu", obs_last_action=last, obs_agent_id=aid)
    scheme, groups, pre = make_scheme(N, A, OBS, S)
    eb = M.EpisodeBatch(scheme, groups, B, TT, preprocess=pre, device="cpu")
    data, lens = synth_episode_data(B, TT, N, A, OBS, S, th.Generator().manual_seed(N), var_len=False)
    fill_episode_batch(eb, data, lens)
    mac = M.mac_REGISTRY["basic"](eb.scheme, groups, args)
    return mac, eb


@pytest.mark.parametrize("last,aid", LAYOUTS)
def test_oracle_inputs_equal_the_controller_inputs(last, aid):
    N, A, OBS, S = 4, 7, 12, 20
    mac, eb = _mac(N, A, OBS, S, last, aid)
    assert mac.input_shape == d_in(OBS, A, N, last, aid) == mac.agent.fc1.weight.shape[1]
    obs, oh = eb["obs"].numpy(), eb["actions_onehot"].numpy()
    for t in range(eb.max_seq_length):
        got = mac._build_inputs(eb, t).numpy()
        ref = build_inputs(obs, oh, t, last, aid)
        assert got.shape == ref.shape and np.array_equal(got, ref), t
    if last and aid:
        assert np.array_equal(build_inputs(obs, oh, 2), O.build_inputs(obs, oh, 2))


def _random_problem(N, A, OBS, S, B, TT, mixer, kind, last, aid, seed):
    from ma_league_b200.synthetic import synth_episode_data, fill_episode_batch
    import ma_league_b200 as M
    from ma_league_b200.synthetic import make_scheme
    rng = np.random.default_rng(seed)
    shapes = (O.agent_param_shapes if kind == "rnn" else O.dqn_agent_param_shapes)(d_in(OBS, A, N, last, aid), A)
    ap, tp = O.init_params(shapes, rng), O.init_params(shapes, rng)
    mp = tmp = None
    if mixer == "qmix":
        ms = O.qmix_param_shapes(S, N, 32, 64)
        mp, tmp = O.init_params(ms, rng), O.init_params(ms, rng)
    scheme, groups, pre = make_scheme(N, A, OBS, S)
    eb = M.EpisodeBatch(scheme, groups, B, TT, preprocess=pre, device="cpu")
    data, lens = synth_episode_data(B, TT, N, A, OBS, S, th.Generator().manual_seed(seed))
    fill_episode_batch(eb, data, lens)
    batch = {k: v.numpy().copy() for k, v in eb.data.transition_data.items()}
    return ap, tp, mp, tmp, batch


@pytest.mark.parametrize("last,aid", LAYOUTS)
@pytest.mark.parametrize("mixer,kind", [("qmix", "rnn"), ("vdn", "rnn"), ("qmix", "dqn")])
def test_numpy_reference_gradient_equals_autograd(last, aid, mixer, kind):
    """The embedded-layout numpy reference (hand-derived backward) against autograd through the reduced th.cat input."""
    N, A, OBS, S, B, TT = 3, 5, 8, 12, 3, 6
    ap, tp, mp, tmp, batch = _random_problem(N, A, OBS, S, B, TT, mixer, kind, last, aid, seed=17)
    ref = learner_forward_backward(ap, tp, mp, tmp, batch, mixer=mixer, double_q=True, gamma=0.99, dtype=np.float64,
                                   last_action=last, agent_id=aid)
    loss, ag, mg = torch_loss_grads(ap, tp, mp, tmp, batch, mixer=mixer, double_q=True, gamma=0.99,
                                    last_action=last, agent_id=aid)
    assert abs(loss - float(ref["loss"])) <= 1e-5 * abs(loss)
    for k, v in ag.items():
        assert ref["agent_grads"][k].shape == v.shape, k
        assert_close(ref["agent_grads"][k], v, 1e-5, "agent " + k)
    for k, v in mg.items():
        assert_close(ref["mixer_grads"][k], v, 1e-5, "mixer " + k)
