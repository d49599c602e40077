"""Autograd through BasicMAC.forward, the agent networks and the mixers (`args.autograd_forward`), against the fp64
oracle's hand-derived backwards (np_oracle.agent_backward / qmix_backward) and the fused learner's gradient."""
import copy

import numpy as np
import pytest
import torch as th

import ma_league_b200._native as nat
from ma_league_b200.modules.agents import REGISTRY as AGENTS
from ma_league_b200.modules.mixers import QMixer, VDNMixer
from ma_league_b200.synthetic import make_args
from oracle import np_oracle as O
from tests import iql_ref as R
from tests import input_layout_ref as IL
from tests.autograd_ref import reference_loss
from tests.gpu_helpers import np_batch, np_params, seeded_system
from tests.helpers import RTOL, assert_close
from tests.test_gpu_iql import iql_system

pytestmark = pytest.mark.gpu


def _grads(module):
    return {k: (p.grad.detach().cpu().numpy().copy() if p.grad is not None else None) for k, p in module.named_parameters()}


def _agent(kind, d_in, A, seed=0):
    th.manual_seed(seed)
    args = make_args(4, A, 16, agent=kind, autograd_forward=True)
    cls = AGENTS[kind]
    return cls(d_in, args)


# ---------------------------------------------------------------------------------------------- 1. one step
@pytest.mark.parametrize("kind", ["rnn", "dqn"])
@pytest.mark.parametrize("rows,d_in", [(1, 37), (160, 53), (1280, 100), (20480, 214)])
def test_agent_step_backward_against_oracle(kind, rows, d_in):
    A = 11
    agent = _agent(kind, d_in, A)
    g = th.Generator().manual_seed(rows + d_in)
    x = th.randn(rows, d_in, generator=g).cuda()
    h = (0.5 * th.randn(rows, 64, generator=g)).cuda().requires_grad_(kind == "rnn")
    dq = th.randn(rows, A, generator=g).cuda()
    dh = th.randn(rows, 64, generator=g).cuda()
    q, h_out = agent(x, h)
    assert q.grad_fn is not None
    with th.no_grad():
        q0, h0 = agent(x, h)
    assert th.equal(q, q0) and (kind == "dqn" or th.equal(h_out, h0))       # same kernel launch as without recording
    if kind == "rnn":
        th.autograd.backward([q, h_out], [dq, dh])
    else:
        q.backward(dq)
    p = {k: v.astype(np.float64) for k, v in np_params(agent).items()}
    xn, hn = x.cpu().double().numpy(), h.detach().cpu().double().numpy()
    if kind == "rnn":
        _, _, c = O.drqn_step(p, xn, hn)
    else:
        _, _, c = O.dqn_step(p, xn)
    if kind == "rnn":
        ref, dh_prev = _rnn_step_backward(p, c, dq.cpu().double().numpy(), dh.cpu().double().numpy())
        assert_close(h.grad.cpu().numpy(), dh_prev, RTOL, "d h_in")
    else:
        ref = O.agent_backward(p, [c], dq.cpu().double().numpy().reshape(rows, 1, 1, A))
    got = _grads(agent)
    for k, v in ref.items():
        assert_close(got[k], v, RTOL, k)


def _rnn_step_backward(p, c, dq, dh_out):
    """np_oracle.agent_backward's step body with an upstream d h_out; returns (grads, d h_prev)."""
    from collections import OrderedDict
    g = OrderedDict((k, np.zeros_like(v)) for k, v in p.items())
    g["fc2.weight"] += dq.T @ c["h"]
    g["fc2.bias"] += dq.sum(axis=0)
    dh = dh_out + dq @ p["fc2.weight"]
    dn = dh * (1 - c["z"]); dz = dh * (c["h_prev"] - c["n"])
    dn_pre = dn * (1 - c["n"] ** 2); dr = dn_pre * c["ghn"]
    dz_pre = dz * c["z"] * (1 - c["z"]); dr_pre = dr * c["r"] * (1 - c["r"])
    dgi = np.concatenate([dr_pre, dz_pre, dn_pre], axis=1)
    dgh = np.concatenate([dr_pre, dz_pre, dn_pre * c["r"]], axis=1)
    g["gru.weight_ih"] += dgi.T @ c["x"]; g["gru.bias_ih"] += dgi.sum(axis=0)
    g["gru.weight_hh"] += dgh.T @ c["h_prev"]; g["gru.bias_hh"] += dgh.sum(axis=0)
    dh_prev = dh * c["z"] + dgh @ p["gru.weight_hh"]
    dx = (dgi @ p["gru.weight_ih"]) * (c["x"] > 0)
    g["fc1.weight"] += dx.T @ c["inp"]; g["fc1.bias"] += dx.sum(axis=0)
    return g, dh_prev


# ---------------------------------------------------------------------------------------------- 2. mac unroll
def _mac_system(N, B, TT, agent="rnn", last=True, aid=True, seed=0):
    s = seeded_system(N, B, TT, "vdn", seed=seed, agent=agent, obs_last_action=last, obs_agent_id=aid,
                      autograd_forward=True)
    return s


@pytest.mark.parametrize("N,B,TT,agent,last,aid", [
    (3, 32, 201, "rnn", True, True), (5, 32, 201, "rnn", True, True), (10, 128, 201, "rnn", True, True),
    (20, 64, 9, "rnn", True, True), (5, 32, 201, "rnn", False, True), (5, 32, 201, "rnn", True, False),
    (5, 32, 201, "rnn", False, False), (5, 32, 201, "dqn", True, True)])
def test_mac_unroll_backward_against_oracle(N, B, TT, agent, last, aid):
    s = _mac_system(N, B, TT, agent, last, aid)
    mac, eb = s.mac, s.batch
    A = s.args.n_actions
    mac.init_hidden(B)
    out = th.stack([mac.forward(eb, t) for t in range(TT)], dim=1)
    g = th.Generator().manual_seed(7)
    dQ = th.randn(out.shape, generator=g).cuda()
    out.backward(dQ)
    nb = np_batch(eb)
    OBS = nb["obs"].shape[-1]
    cols = IL.input_columns(OBS, A, N, last, aid)
    p = {k: v.astype(np.float64) for k, v in IL.embed_agent(np_params(mac.agent), cols, OBS + A + N).items()}
    mac_out, caches = O.unroll(p, nb["obs"].astype(np.float64), nb["actions_onehot"].astype(np.float64))
    assert_close(out.detach().cpu().numpy(), mac_out, RTOL, "mac_out")
    x_mask = np.stack([c["x_pre"] > 0 for c in caches])
    ref = O.agent_backward(p, caches, dQ.cpu().double().numpy(), x_mask)
    got = _grads(mac.agent)
    ref_fc1 = ref["fc1.weight"][:, cols]
    assert_close(got["fc1.weight"], ref_fc1, RTOL, "fc1.weight")
    for k, v in ref.items():
        if k != "fc1.weight":
            assert_close(got[k], v, RTOL, k)


# ---------------------------------------------------------------------------------------------- 3. mixers
@pytest.mark.parametrize("layers", [1, 2])
@pytest.mark.parametrize("N,B,T", [(5, 32, 200), (10, 128, 50)])
def test_qmixer_backward_against_oracle(layers, N, B, T):
    S = 16 * N
    th.manual_seed(3)
    args = make_args(N, 6 + N, S, hypernet_layers=layers, autograd_forward=True)
    mixer = QMixer(args)
    g = th.Generator().manual_seed(4)
    qs = th.randn(B, T, N, generator=g).cuda().requires_grad_(True)
    st = th.randn(B, T + 1, S, generator=g).cuda()[:, :-1]            # strided view like batch["state"][:, :-1]
    dqt = th.randn(B, T, 1, generator=g).cuda()
    y = mixer(qs, st)
    with th.no_grad():
        y0 = mixer(qs, st)
    assert th.equal(y, y0)
    y.backward(dqt)
    mp = {k: v.astype(np.float64) for k, v in np_params(mixer).items()}
    yr, cache = O.qmix_forward(mp, qs.detach().cpu().double().numpy(), st.cpu().double().numpy())
    assert_close(y.detach().cpu().numpy(), yr, RTOL, "q_tot")
    grads, dq = O.qmix_backward(mp, cache, dqt.cpu().double().numpy())
    assert_close(qs.grad.cpu().numpy(), dq.reshape(B, T, N), RTOL, "d agent_qs")
    got = _grads(mixer)
    for k, v in grads.items():
        assert_close(got[k], v, RTOL, k)
    with pytest.raises(nat.MalError):
        mixer(qs, st.clone().requires_grad_(True))


def test_vdn_mixer_backward():
    args = make_args(5, 11, 80, mixer="vdn", autograd_forward=True)
    mixer = VDNMixer(args)
    qs = th.randn(4, 7, 5, device="cuda", requires_grad=True)
    y = mixer(qs, None)
    with th.no_grad():
        y0 = mixer(qs, None)
    assert y.grad_fn is not None and th.equal(y, y0)
    d = th.randn(4, 7, 1, device="cuda")
    y.backward(d)
    assert th.equal(qs.grad, d.expand(4, 7, 5))


# ---------------------------------------------------------------------------------------------- 4. end to end
def _reference_through_modules(s, double_q):
    L, eb = s.learner, s.batch
    B = eb.batch_size
    mac, tmac = L.mac, L.target_mac
    mac.init_hidden(B)
    tmac.init_hidden(B)
    tb = {k: eb[k] for k in ("reward", "actions", "terminated", "filled", "avail_actions", "state", "obs")}
    mix = L.mixer
    tmix = L.target_mixer if mix is not None else None
    mix_f = (lambda q, st: mix(q, st if isinstance(mix, QMixer) else eb)) if mix is not None else None
    tmix_f = (lambda q, st: tmix(q, st if isinstance(tmix, QMixer) else eb)) if tmix is not None else None
    loss, _ = reference_loss(tb, lambda t: mac.forward(eb, t), lambda t: tmac.forward(eb, t), mix_f, tmix_f,
                             double_q=double_q, gamma=s.args.gamma)
    return loss


@pytest.mark.parametrize("mixer", ["qmix", "vdn", None])
@pytest.mark.parametrize("double_q", [True, False])
def test_reference_learner_on_modules_end_to_end(mixer, double_q):
    if mixer is None:
        s = iql_system(5, 32, 201, double_q=double_q, clip=1e9, autograd_forward=True)
    else:
        s = seeded_system(5, 32, 201, mixer, double_q=double_q, clip=1e9, autograd_forward=True)
    L = s.learner
    params = list(L.mac.parameters()) + (list(L.mixer.parameters()) if L.mixer is not None else [])
    flat = L.forward_backward(s.batch).clone()
    th.cuda.synchronize()
    loss = _reference_through_modules(s, double_q)
    loss.backward()
    got = th.cat([p.grad.reshape(-1) for p in params])
    assert_close(got.cpu().numpy(), flat.cpu().numpy(), RTOL, "gradient against the fused learner")
    nb = np_batch(s.batch)
    if mixer is None:
        ref = R.learner_forward_backward(np_params(L.mac.agent), np_params(L.target_mac.agent), nb, double_q=double_q,
                                         gamma=s.args.gamma)
    else:
        ref = O.learner_forward_backward(np_params(L.mac.agent), np_params(L.target_mac.agent),
                                         np_params(L.mixer) if mixer == "qmix" else None,
                                         np_params(L.target_mixer) if mixer == "qmix" else None, nb, mixer=mixer,
                                         double_q=double_q, gamma=s.args.gamma, dtype=np.float64)
    assert abs(float(loss.detach()) - ref["loss"]) <= RTOL * abs(ref["loss"])
    got_a = _grads(L.mac.agent)
    for k, v in ref["agent_grads"].items():
        assert_close(got_a[k], v, RTOL, "agent " + k)
    if mixer == "qmix":
        got_m = _grads(L.mixer)
        for k, v in ref["mixer_grads"].items():
            assert_close(got_m[k], v, RTOL, "mixer " + k)
    # one stock RMSprop step against the oracle's update (flat over all parameters, like test_gpu_iql)
    opt = th.optim.RMSprop(params, lr=s.args.lr, alpha=s.args.optim_alpha, eps=s.args.optim_eps)
    p0 = np.concatenate([p.detach().cpu().double().numpy().ravel() for p in params])
    ref_g = list(ref["agent_grads"].values()) + (list(ref["mixer_grads"].values()) if mixer == "qmix" else [])
    p1, _ = O.rmsprop_update(p0, np.concatenate([g.ravel() for g in ref_g]), np.zeros_like(p0), s.args.lr,
                             s.args.optim_alpha, s.args.optim_eps)
    own = np.concatenate([p.grad.detach().cpu().double().numpy().ravel() for p in params])
    p1_own, _ = O.rmsprop_update(p0, own, np.zeros_like(p0), s.args.lr, s.args.optim_alpha, s.args.optim_eps)
    opt.step()
    got = np.concatenate([p.detach().cpu().numpy().ravel() for p in params])
    assert_close(got, p1_own, RTOL, "RMSprop step on the recorded gradient")
    # the first RMSprop step divides by |g| (plus eps): the update of a near-zero gradient element amplifies its 1e-5
    # relative error, so the oracle's update is compared as in test_gpu_iql (1e-3 on the update)
    assert_close(got - p0, p1 - p0, 1e-3, "update of the RMSprop step")


# ---------------------------------------------------------------------------------------------- 5. behaviour kept
def test_switch_off_keeps_inference_only_and_outputs_bit_identical():
    s_off = seeded_system(5, 8, 12, "qmix")
    s_on = seeded_system(5, 8, 12, "qmix", autograd_forward=True)
    assert copy.deepcopy(s_on.mac).args.autograd_forward and s_on.learner.target_mac.args.autograd_forward
    outs = []
    for s in (s_off, s_on):
        s.mac.init_hidden(8)
        outs.append(th.stack([s.mac.forward(s.batch, t) for t in range(12)], dim=1))
    assert outs[0].grad_fn is None and outs[1].grad_fn is not None
    assert th.equal(outs[0], outs[1].detach())
    mac = s_on.mac
    mac.init_hidden(8)
    mac.select_actions(s_on.batch, 0, 0, test_mode=True)
    assert mac.hidden_states.grad_fn is None
    with th.no_grad():
        mac.init_hidden(8)
        assert mac.forward(s_on.batch, 0).grad_fn is None


def test_backward_reproducible_accumulating_and_version_checked():
    s = seeded_system(5, 16, 30, "qmix", autograd_forward=True)
    mac, mixer = s.mac, s.learner.mixer
    params = list(mac.parameters()) + list(mixer.parameters())

    def run():
        mac.init_hidden(16)
        out = th.stack([mac.forward(s.batch, t) for t in range(30)], dim=1)
        chosen = th.gather(out[:, :-1], 3, s.batch["actions"][:, :-1]).squeeze(3)
        return (mixer(chosen, s.batch["state"][:, :-1]) ** 2).sum()
    for p in params:
        p.grad = None
    run().backward()
    g1 = [p.grad.clone() for p in params]
    for p in params:
        p.grad = None
    run().backward()
    assert all(th.equal(a, p.grad) for a, p in zip(g1, params))
    run().backward()
    assert all(th.allclose(2 * a, p.grad, rtol=1e-6, atol=0) for a, p in zip(g1, params))
    loss = run()
    opt = th.optim.RMSprop(params, lr=1e-3)
    opt.step()
    with pytest.raises(RuntimeError, match="modified by an inplace operation"):
        loss.backward()


def test_frozen_agent_gets_no_gradient_mixer_trains():
    s = seeded_system(5, 8, 12, "qmix", freeze_native=True, autograd_forward=True)
    mac, mixer = s.mac, s.learner.mixer
    mac.init_hidden(8)
    out = th.stack([mac.forward(s.batch, t) for t in range(12)], dim=1)
    chosen = th.gather(out[:, :-1], 3, s.batch["actions"][:, :-1]).squeeze(3)
    mixer(chosen, s.batch["state"][:, :-1]).sum().backward()
    assert all(p.grad is None for p in mac.parameters())
    assert all(p.grad is not None and th.isfinite(p.grad).all() for p in mixer.parameters())


def test_dense_input_requiring_grad_raises():
    agent = _agent("rnn", 20, 5)
    x = th.randn(4, 20, device="cuda", requires_grad=True)
    with pytest.raises(nat.MalError):
        agent(x, th.zeros(4, 64, device="cuda"))
