"""CPU side of autograd through the modules (`args.autograd_forward`): the restated reference learner of
tests/autograd_ref.py against the fp64 oracle, the backward entry points' host-side checks and the ABI surface."""
from collections import OrderedDict

import numpy as np
import pytest
import torch as th

import ma_league_b200._native as nat
from oracle import np_oracle as O
from oracle import torch_port as TP
from tests import iql_ref as R
from tests.autograd_ref import reference_loss
from tests.helpers import assert_close


def _system(N, B, TT, mixer, agent="rnn", seed=0):
    A, OBS, S = 6 + N, 8 + 8 * N, 16 * N
    rng = np.random.default_rng(seed)
    shapes = (O.dqn_agent_param_shapes if agent == "dqn" else O.agent_param_shapes)(OBS + A + N, A)
    ap = O.init_params(shapes, rng, np.float64)
    tp = OrderedDict((k, v + 0.05 * rng.standard_normal(v.shape)) for k, v in ap.items())
    mp = tmp = None
    if mixer == "qmix":
        mp = O.init_params(O.qmix_param_shapes(S, N), rng, np.float64)
        tmp = OrderedDict((k, v + 0.05 * rng.standard_normal(v.shape)) for k, v in mp.items())
    avail = (rng.random((B, TT, N, A)) < 0.7).astype(np.int32)
    avail[..., 0] = 1
    actions = np.argmax(avail / rng.exponential(size=avail.shape), axis=-1)[..., None].astype(np.int64)
    lens = rng.integers(TT // 2, TT, size=B)
    lens[0] = TT - 1
    filled = (np.arange(TT)[None, :] < lens[:, None]).astype(np.int64)[..., None]
    term = np.zeros((B, TT, 1), np.uint8)
    term[np.arange(B), lens - 1] = 1
    batch = dict(obs=rng.standard_normal((B, TT, N, OBS)), state=rng.standard_normal((B, TT, S)),
                 reward=rng.standard_normal((B, TT, 1)), actions=actions, avail_actions=avail, terminated=term,
                 filled=filled, actions_onehot=np.eye(A)[actions[..., 0]] * filled[..., None])
    return ap, tp, mp, tmp, batch


def _torch_port_loss(ap, tp, mp, tmp, batch, mixer, double_q, gamma):
    P = lambda d, g: OrderedDict((k, th.tensor(v, dtype=th.float64, requires_grad=g)) for k, v in d.items())
    pa, pt = P(ap, True), P(tp, False)
    pm, ptm = (P(mp, True), P(tmp, False)) if mixer == "qmix" else (None, None)
    tb = {k: th.from_numpy(np.ascontiguousarray(v)) for k, v in batch.items()}
    tb["reward"] = tb["reward"].double()
    B, _, N, _ = tb["obs"].shape
    state = {"on": th.zeros(B * N, 64, dtype=th.float64), "tg": th.zeros(B * N, 64, dtype=th.float64)}

    def step(p, key):
        def f(t):
            q, state[key] = TP.agent_step(p, tb, t, state[key])
            return q
        return f
    mix = tmix = None
    if mixer == "qmix":
        mix, tmix = (lambda q, s: TP.qmix(pm, q, s)), (lambda q, s: TP.qmix(ptm, q, s))
    elif mixer == "vdn":
        mix = tmix = lambda q, s: q.sum(dim=2, keepdim=True)
    loss, _ = reference_loss(tb, step(pa, "on"), step(pt, "tg"), mix, tmix, double_q=double_q, gamma=gamma)
    loss.backward()
    grads = {k: v.grad.numpy() for k, v in pa.items()}
    mgrads = {k: v.grad.numpy() for k, v in pm.items()} if pm is not None else {}
    return float(loss.detach()), grads, mgrads


@pytest.mark.parametrize("mixer", ["qmix", "vdn", None])
@pytest.mark.parametrize("double_q", [True, False])
@pytest.mark.parametrize("agent", ["rnn", "dqn"])
def test_restated_reference_learner_equals_oracle(mixer, double_q, agent):
    ap, tp, mp, tmp, batch = _system(3, 4, 9, mixer, agent)
    loss, grads, mgrads = _torch_port_loss(ap, tp, mp, tmp, batch, mixer, double_q, 0.99)
    if mixer is None:
        ref = R.learner_forward_backward(ap, tp, batch, double_q=double_q, gamma=0.99)
    else:
        ref = O.learner_forward_backward(ap, tp, mp, tmp, batch, mixer=mixer, double_q=double_q, gamma=0.99,
                                         dtype=np.float64)
    assert abs(loss - ref["loss"]) <= 1e-12 * max(1.0, abs(ref["loss"]))
    for k, v in ref["agent_grads"].items():
        assert_close(grads[k], v, 1e-10, "agent " + k)
    for k, v in ref["mixer_grads"].items():
        assert_close(mgrads[k], v, 1e-10, "mixer " + k)


def test_backward_workspace_queries_and_rejection_without_a_device():
    L = nat.lib()
    for kind in (nat.AGENT_RNN, nat.AGENT_DQN):
        for dense in (0, nat.STEP_DENSE, nat.IN_NO_LAST_ACTION << 1, (nat.IN_NO_LAST_ACTION | nat.IN_NO_AGENT_ID) << 1):
            small = L.mal_agent_step_backward_workspace(kind, 160, 5, 48, 11, dense)
            big = L.mal_agent_step_backward_workspace(kind, 20480, 20, 168, 26, dense)
            assert 0 < small < big and small % 256 == 0
    assert L.mal_agent_step_backward_workspace(2, 160, 5, 48, 11, 0) == -1
    assert L.mal_agent_step_backward_workspace(nat.AGENT_RNN, 160, 5, 48, 33, 0) == -1
    assert L.mal_agent_step_backward_workspace(nat.AGENT_RNN, 160, 5, 48, 11, 8) == -1
    assert L.mal_agent_step_backward_workspace(nat.AGENT_RNN, 160, 5, 48, 11, 3) == -1
    assert L.mal_agent_step_backward_workspace(nat.AGENT_RNN, 0, 5, 48, 11, 0) == -1
    for mixer in (nat.MIXER_QMIX2, nat.MIXER_QMIX1):
        assert L.mal_mixer_backward_workspace(mixer, 32, 200, 5, 80, 32, 64) > 0
    assert L.mal_mixer_backward_workspace(nat.MIXER_VDN, 32, 200, 5, 80, 32, 64) == -1
    assert L.mal_mixer_backward_workspace(nat.MIXER_NONE, 32, 200, 5, 80, 32, 64) == -1
    assert L.mal_mixer_backward_workspace(nat.MIXER_QMIX2, 32, 200, 5, 80, 33, 64) == -1
    assert b"has no kernel backward" in L.mal_last_error() or b"mixing_embed_dim" in L.mal_last_error()
    rc = L.mal_mixer_backward(nat.MIXER_QMIX2, 2, 3, 2, 4, 8, 8, None, None, None, 0, 0, None, None, None, None, None, None)
    assert rc != 0 and b"null argument" in L.mal_last_error()
    rc = L.mal_agent_step_backward(nat.AGENT_DQN, None, 4, 2, 3, 2, 0, None, 0, None, 0, None, None, None, None, None, None,
                                   None)
    assert rc != 0 and b"required" in L.mal_last_error()


def test_backward_symbols_exported_and_abi_version():
    L = nat.lib()
    assert L.mal_version() == nat.ABI_VERSION == 6
    for name in ("mal_agent_step_backward", "mal_agent_step_backward_workspace", "mal_mixer_backward",
                 "mal_mixer_backward_workspace"):
        assert name in nat.EXPORTS and hasattr(L, name)
