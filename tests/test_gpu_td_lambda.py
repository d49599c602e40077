"""TD(lambda) targets (`args.td_lambda`) through the CUDA learner step, against the fp64 reference of
tests/td_lambda_ref.py: targets / td, loss, statistics and every gradient for QMIX (2 and 1 layers), VDN and IQL, both
agents, both double_q settings, a switched input layout and a frozen agent; chained steps; eager against graph replay and
re-capture when lambda changes; prioritized replay; `train_from_buffer` masked against truncated and against the loop by
hand; two un-normalised halves through the peer exchange against the full batch; the launch count of a lambda step."""
import ctypes as C

import numpy as np
import pytest
import torch as th

import ma_league_b200 as M
from ma_league_b200 import _native as nat
from ma_league_b200.learners.q_learner import DP_RAW, DP_TAIL
from ma_league_b200.synthetic import synth_episode_data, fill_episode_batch
from oracle import np_oracle as O
from tests import td_lambda_ref as R
from tests.gpu_helpers import build_system, np_params, np_batch
from tests.helpers import assert_close, rel_err
from tests.test_gpu_learner import _discrete_choices

pytestmark = pytest.mark.gpu
DEV = "cuda"
TOL = 1e-5
STATS = ("loss", "grad_norm", "td_error_abs", "q_taken_mean", "target_mean")


def _system(N, B, TT, mixer, lam, layers=2, agent="rnn", double_q=True, layout=(True, True), seed=0, clip=10.0,
            open_ended=True, **kw):
    """A = 6 + N, OBS = 8 + 8N, S = 16N, perturbed targets, episode lengths in [T/2, T]; episode 0 fills the window and,
    with `open_ended`, episode 1 is a short episode that ends without `terminated`."""
    A, OBS, S = 6 + N, 8 + 8 * N, 16 * N
    th.manual_seed(seed)
    s = build_system(N, A, OBS, S, B, TT, mixer, double_q, hypernet_layers=layers, clip=clip, agent=agent,
                     obs_last_action=layout[0], obs_agent_id=layout[1], td_lambda=lam, learner_log_interval=0, **kw)
    gen = th.Generator().manual_seed(seed + 1)
    nets = list(s.learner.target_mac.parameters()) + (list(s.learner.target_mixer.parameters()) if mixer else [])
    with th.no_grad():
        for p in nets:
            p.add_(0.05 * th.randn(p.shape, generator=gen).to(DEV))
    data, lens = synth_episode_data(B, TT, N, A, OBS, S, gen, var_len=True, device=DEV)
    lens[0] = TT - 1
    if open_ended and B > 1:
        lens[1] = max(2, (TT - 1) // 3)
    eb = fill_episode_batch(M.EpisodeBatch(s.scheme, s.groups, B, TT, preprocess=s.pre, device=DEV), data, lens)
    if open_ended and B > 1:
        eb.data.transition_data["terminated"][1].zero_()
    s["batch"] = eb
    s["mixer"], s["layout"] = mixer, layout
    return s


def _nets(s):
    L = s.learner
    return [s.mac.agent] + ([L.mixer] if s.mixer else [])


def _flat_params(s):
    return np.concatenate([v.ravel() for n in _nets(s) for v in np_params(n).values()]).astype(np.float64)


def _oracle(s, lam, params=None, weights=None, batch=None, **kw):
    L = s.learner
    ap, mp = params if params is not None else (np_params(s.mac.agent), np_params(L.mixer) if s.mixer else None)
    return R.learner_forward_backward(ap, np_params(L.target_mac.agent), mp,
                                      np_params(L.target_mixer) if s.mixer else None,
                                      np_batch(s.batch) if batch is None else batch, mixer=s.mixer,
                                      double_q=bool(s.args.double_q), gamma=s.args.gamma, td_lambda=lam, weights=weights,
                                      last_action=s.layout[0], agent_id=s.layout[1], **kw)


def _ref_flat(ref):
    return np.concatenate([v.ravel() for v in list(ref["agent_grads"].values()) + list(ref["mixer_grads"].values())])


def against_oracle(s, lam, params=None, weights=None):
    """One forward + backward on the device against the reference (near-ties of the double-Q arg-max and of the ReLU /
    abs derivatives handled as in tests/test_gpu_learner.py).  Returns the reference."""
    L = s.learner
    if weights is not None:
        bs, cfg, f = L._prepare(s.batch)
        bs.weight = nat.Field(weights.data_ptr(), weights.stride(0), 0)
        with nat.on_device(DEV):
            nat.check(nat.lib().mal_learner_forward(C.byref(bs), C.byref(cfg), C.byref(L._plan), nat.ptr(f["agent"]),
                                                    nat.ptr(f["tagent"]), nat.ptr(f["mixer"]), nat.ptr(f["tmixer"]),
                                                    nat.ptr(L._ws), nat.current_stream()), "mal_learner_forward")
            nat.check(nat.lib().mal_learner_backward(C.byref(bs), C.byref(cfg), C.byref(L._plan), nat.ptr(f["agent"]),
                                                     nat.ptr(f["mixer"]), nat.ptr(L._ws), nat.ptr(L._grad),
                                                     nat.current_stream()), "mal_learner_backward")
        flat = L._grad
    else:
        flat = L.forward_backward(s.batch)
    th.cuda.synchronize()
    got = flat.cpu().numpy().astype(np.float64)
    it = {k: v.cpu().numpy() for k, v in L.intermediates(s.batch).items()}
    w = None if weights is None else weights.cpu().numpy().astype(np.float64)
    ref = _oracle(s, lam, params, w)
    flips = np.argwhere(it["argmax"].astype(np.int64) != ref["argmax"])
    if len(flips):
        oq = ref["mac_out"][:, 1:].copy()
        oq[np_batch(s.batch)["avail_actions"][:, 1:] == 0] = O.NEG_MASK
        for b, t, n in flips:
            row = oq[b, t, n]
            gap = abs(row[ref["argmax"][b, t, n]] - row[it["argmax"][b, t, n]])
            assert gap <= 1e-5 * max(1.0, np.abs(row[row > O.NEG_MASK]).max()), ("argmax flip without a near-tie", b, t, n)
        assert len(flips) <= 1 + it["argmax"].size // 100000, "%d argmax flips" % len(flips)
    discrete, n_diff = _discrete_choices(it, ref, s.mixer)
    if len(flips) or n_diff:
        ref = _oracle(s, lam, params, w, argmax_override=it["argmax"].astype(np.int64), discrete=discrete)
    assert_close(it["mask"], ref["mask"], 0, "mask")
    assert_close(it["target_q_tot"], ref["target_q_tot"], TOL, "target_q_tot")
    assert_close(it["q_tot"], ref["q_tot"], TOL, "q_tot")
    assert_close(it["targets"], ref["targets"], TOL, "targets")
    assert_close(it["td"], ref["td"], TOL, "td")
    sc, st = it["scalars"], ref["stats"]
    assert abs(sc[nat.SC_LOSS] - ref["loss"]) <= TOL * abs(ref["loss"]), (sc[nat.SC_LOSS], ref["loss"])
    assert sc[nat.SC_MASK_SUM] == st["mask_sum"]
    for i, k in ((nat.SC_TD_ABS, "td_error_abs"), (nat.SC_Q_TAKEN, "q_taken_mean"), (nat.SC_TARGET, "target_mean")):
        assert abs(sc[i] - st[k]) <= TOL * max(1.0, abs(st[k])), (k, sc[i], st[k])
    assert int(sc[nat.SC_MASK_COUNT:nat.SC_MASK_COUNT + 1].view(np.int32)[0]) == st["trained_steps"]
    off = 0
    for k, v in list(ref["agent_grads"].items()) + list(ref["mixer_grads"].items()):
        assert_close(got[off:off + v.size].reshape(v.shape), v, TOL, "grad " + k)
        off += v.size
    assert off == got.size
    return ref


def two_steps(s, lam):
    """against_oracle, then train() (graphs on) twice, chained through the reference from the same start: the logged
    statistics, the parameters and square_avg after each step."""
    L, a = s.learner, s.args
    nets = _nets(s)
    params = [{k: v.astype(np.float64) for k, v in np_params(n).items()} for n in nets]
    p = np.concatenate([v.ravel() for d in params for v in d.values()])
    sq = np.zeros(p.size)
    for i in range(2):
        ref = against_oracle(s, lam, (params[0], params[1] if s.mixer else None))
        norm, (g_clip,) = O.clip_grad_norm([_ref_flat(ref)], a.grad_norm_clip)
        p1, sq = O.rmsprop_update(p, g_clip, sq, a.lr, a.optim_alpha, a.optim_eps)
        L.train(s.batch, t_env=i, episode_num=0)
        th.cuda.synchronize()
        logged = {k[len("home_qlearner_"):]: v[0] for k, v in s.logger.stats.items()}
        want = dict(loss=ref["loss"], grad_norm=norm, **{k: ref["stats"][k] for k in STATS[2:]})
        for k in STATS:
            assert abs(logged[k] - want[k]) <= TOL * max(1.0, abs(want[k])), (i, k, logged[k], want[k])
        got = _flat_params(s)
        assert_close(got, p1, TOL, "parameters after step %d" % (i + 1))
        assert rel_err(L.optimiser.flat_sq.cpu().numpy(), sq) < 1e-4, "square_avg after step %d" % (i + 1)
        p, off = p1, 0
        for d in params:
            for k, v in d.items():
                d[k] = p[off:off + v.size].reshape(v.shape)
                off += v.size


# ---------------------------------------------------------------------------------------------- shapes and variations
CASES = [  # N, B, TT, mixer, layers, agent, double_q, layout, lambda
    (3, 32, 201, "qmix", 2, "rnn", True, (True, True), 0.6),
    (5, 32, 201, "qmix", 2, "rnn", True, (True, True), 1.0),
    (5, 32, 201, "qmix", 2, "rnn", True, (True, True), 0.0),
    (10, 128, 201, "qmix", 2, "rnn", True, (True, True), 0.6),
    (20, 16, 24, "qmix", 2, "rnn", True, (True, True), 0.6),
    (5, 32, 201, "qmix", 1, "rnn", False, (True, True), 0.6),
    (5, 32, 201, "vdn", 2, "rnn", True, (True, True), 0.6),
    (10, 32, 201, "vdn", 2, "rnn", True, (True, True), 1.0),
    (5, 32, 201, None, 2, "rnn", True, (True, True), 0.6),
    (20, 16, 24, None, 2, "dqn", True, (True, True), 1.0),
    (5, 32, 201, "qmix", 2, "dqn", True, (True, True), 0.6),
    (3, 16, 40, "qmix", 2, "rnn", True, (False, True), 0.6),
]


@pytest.mark.parametrize("N,B,TT,mixer,layers,agent,double_q,layout,lam", CASES)
def test_lambda_step_against_reference(N, B, TT, mixer, layers, agent, double_q, layout, lam):
    s = _system(N, B, TT, mixer, lam, layers, agent, double_q, layout, seed=200 + N + TT)
    two_steps(s, lam)


def test_frozen_agent():
    s = _system(5, 16, 61, "qmix", 0.6, seed=9)
    s.mac.freeze_agent_weights()
    L = s.learner
    agent0 = np_params(s.mac.agent)
    ref = _oracle(s, 0.6)
    L.train(s.batch, 0, 0)
    th.cuda.synchronize()
    n_agent = sum(v.size for v in agent0.values())
    g = L._grad.cpu().numpy()
    assert not g[:n_agent].any()
    norm, (g_clip,) = O.clip_grad_norm([np.concatenate([v.ravel() for v in ref["mixer_grads"].values()])], s.args.grad_norm_clip)
    assert_close(g[n_agent:], g_clip, TOL, "mixer gradient with a frozen agent")
    for k, v in np_params(s.mac.agent).items():
        assert np.array_equal(v, agent0[k]), k


# ---------------------------------------------------------------------------------------------- graphs
def _state(s):
    """Parameters, square_avg and the scalars the step writes (slot SC_STATUS is not written by the learner step)."""
    return [v.clone() for n in _nets(s) for v in n.state_dict().values()] + \
        [s.learner.optimiser.flat_sq.clone(), s.learner.scalars()[:nat.SC_STATUS].clone()]


@pytest.mark.parametrize("mixer", ["qmix", None])
def test_graph_replay_bit_identical_to_eager_and_recapture_on_lambda_change(mixer):
    outs = []
    for graphs in (False, True):
        s = _system(5, 8, 61, mixer, 0.6, seed=4)
        s.learner.use_graphs = graphs
        for i in range(4):                                     # eager, capture (which performs the step), replay, replay
            s.learner.train(s.batch, i, 0)
        th.cuda.synchronize()
        assert s.learner.n_graph_captures == (1 if graphs else 0)
        assert s.learner.n_graph_replays == (2 if graphs else 0)
        outs.append(_state(s))
    for x, y in zip(*outs):
        assert th.equal(x, y)
    # lambda changes between steps: its own key (eager, capture, replay), never a replay of the 0.6 graph
    L = s.learner
    replays, captures = L.n_graph_replays, L.n_graph_captures
    for lam in (0.25, 0.25, None, 0.25, 0.25):
        s.args.td_lambda = lam
        ref = _oracle(s, 0.0 if lam is None else lam)
        L.train(s.batch, 9, 0)
        th.cuda.synchronize()
        norm, _ = O.clip_grad_norm([_ref_flat(ref)], s.args.grad_norm_clip)
        if lam is not None:
            assert abs(s.logger.stats["home_qlearner_loss"][0] - ref["loss"]) <= TOL * abs(ref["loss"])
            assert abs(s.logger.stats["home_qlearner_target_mean"][0] - ref["stats"]["target_mean"]) <= \
                TOL * max(1.0, abs(ref["stats"]["target_mean"]))
            assert abs(s.logger.stats["home_qlearner_grad_norm"][0] - norm) <= TOL * norm
    assert L.n_graph_captures == captures + 1 and L.n_graph_replays == replays + 2


def test_launch_count_is_one_step_plus_two():
    counts = {}
    for lam in (None, 0.6):
        s = _system(5, 8, 61, "qmix", lam, seed=5)
        s.learner.use_graphs = False
        s.learner.train(s.batch, 0, 0)
        th.cuda.synchronize()
        n0 = nat.lib().mal_launch_count()
        s.learner.train(s.batch, 1, 0)
        th.cuda.synchronize()
        counts[lam] = nat.lib().mal_launch_count() - n0
    assert counts[0.6] == counts[None] + 2, counts


# ---------------------------------------------------------------------------------------------- prioritized replay
@pytest.mark.parametrize("N,B,TT,mixer", [(5, 32, 201, "qmix"), (5, 16, 61, None), (10, 8, 201, "vdn")])
def test_weighted_lambda_step(N, B, TT, mixer):
    s = _system(N, B, TT, mixer, 0.6, seed=31 + N)
    w = (th.rand(B, generator=th.Generator().manual_seed(3)) * 0.9 + 0.1).to(DEV)
    against_oracle(s, 0.6, weights=w)


def _per_buffer(s, size, TT, **kw):
    return M.PrioritizedReplayBuffer(s.scheme, s.groups, size, TT, preprocess=s.pre, device=DEV, alpha=0.6, beta=0.4,
                                     eps=1e-6, **kw)


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


def _loop_system(seed, per, N=5, size=64, TT=31, lam=0.6):
    s = _system(N, 8, TT, "qmix", lam, seed=seed, open_ended=False)
    buf = _per_buffer(s, size, TT) if per else M.ReplayBuffer(s.scheme, s.groups, size, TT, preprocess=s.pre, device=DEV)
    _fill(s, buf, size // 8, 8, TT, seed + 7, N, short=20)
    return s, buf


@pytest.mark.parametrize("per", [False, True])
def test_train_from_buffer_equals_manual_loop(per):
    s1, b1 = _loop_system(9, per)
    s2, b2 = _loop_system(9, per)
    th.manual_seed(77)
    np.random.seed(77)                                        # the uniform buffer samples with numpy, PER with torch
    for i in range(4):
        s1.learner.train_from_buffer(b1, 8, t_env=i, episode_num=0)
    th.manual_seed(77)
    np.random.seed(77)
    s2.learner.use_graphs = False
    for i in range(4):
        full = b2.sample(8)
        s2.learner.train(full, i, 0, weights=full.weights if per else None)
        if per:
            inter = s2.learner.intermediates(full)
            b2.update_priorities(full.ids, inter["td"].contiguous(), inter["mask"].reshape(8, -1).contiguous())
    th.cuda.synchronize()
    assert s1.learner.n_graph_replays >= 2
    for x, y in zip(_state(s1), _state(s2)):
        assert th.equal(x, y)
    if per:
        assert th.equal(b1.priorities, b2.priorities) and th.equal(b1.max_priority, b2.max_priority)
        assert not th.equal(b1.priorities, th.ones_like(b1.priorities))


def test_priorities_from_lambda_td():
    s, buf = _loop_system(5, True)
    L = s.learner
    th.manual_seed(3)
    p0 = buf.priorities.clone()
    params = (np_params(s.mac.agent), np_params(L.mixer))     # the step updates them; the targets used these
    L.train_from_buffer(buf, 8, t_env=0, episode_num=0)
    th.cuda.synchronize()
    st = L._stage
    it = {k: v.cpu().numpy() for k, v in L.intermediates(st).items()}
    ids = st.ids.cpu().numpy()
    td, m = it["td"].astype(np.float64), it["mask"][..., 0].astype(np.float64)[..., None]
    new = (np.abs(td * m).sum(axis=(1, 2)) / m.sum(axis=(1, 2)) + 1e-6) ** 0.6
    want = p0.cpu().numpy().astype(np.float64)
    for b, i in enumerate(ids):
        want[i] = new[b]
    assert np.allclose(buf.priorities.cpu().numpy(), want, rtol=2e-6, atol=0)
    ref = _oracle(s, 0.6, params, batch=np_batch(st), weights=st.weights.cpu().numpy().astype(np.float64),
                  argmax_override=it["argmax"].astype(np.int64))     # the double-Q choices are checked elsewhere
    assert_close(it["targets"], ref["targets"], TOL, "targets of the sampled batch")


def test_masked_padding_equals_truncation():
    """Episodes that terminate inside the window: masked padding and truncation give the same update."""
    outs = []
    for truncate in (False, True):
        s, buf = _loop_system(11, False)
        th.manual_seed(5)
        np.random.seed(5)
        for i in range(3):
            s.learner.train_from_buffer(buf, 8, t_env=i, episode_num=0, truncate=truncate)
        th.cuda.synchronize()
        outs.append((_flat_params(s), s.learner.optimiser.flat_sq.cpu().numpy()))
    assert_close(outs[0][0], outs[1][0], TOL, "parameters")
    assert rel_err(outs[0][1], outs[1][1]) < 1e-4


# ---------------------------------------------------------------------------------------------- data-parallel
def test_unnormalised_halves_through_peer_exchange_equal_full_batch():
    s = _system(5, 16, 61, "qmix", 0.6, seed=17)
    L = s.learner
    ref = _oracle(s, 0.6)
    p0 = _flat_params(s)
    bufs = []
    for lo, hi in ((0, 8), (8, 16)):
        half = s.batch[lo:hi]
        bs, cfg, f = L._prepare(half)
        cfg.unnormalized = 1
        n_total = L._grad.numel()
        buf = th.zeros(n_total + DP_TAIL, device=DEV)
        with nat.on_device(DEV):
            nat.check(nat.lib().mal_learner_forward(C.byref(bs), C.byref(cfg), C.byref(L._plan), nat.ptr(f["agent"]),
                                                    nat.ptr(f["tagent"]), nat.ptr(f["mixer"]), nat.ptr(f["tmixer"]),
                                                    nat.ptr(L._ws), nat.current_stream()), "mal_learner_forward")
            nat.check(nat.lib().mal_learner_backward(C.byref(bs), C.byref(cfg), C.byref(L._plan), nat.ptr(f["agent"]),
                                                     nat.ptr(f["mixer"]), nat.ptr(L._ws), nat.ptr(buf),
                                                     nat.current_stream()), "mal_learner_backward")
        buf[n_total:n_total + DP_RAW].copy_(L.scalars()[nat.SC_RAW0:nat.SC_RAW0 + DP_RAW])
        bufs.append(buf)
    n_agent = L._plan.n_agent_params
    agent = th.from_numpy(p0[:n_agent].astype(np.float32)).to(DEV)
    mixer = th.from_numpy(p0[n_agent:].astype(np.float32)).to(DEV)
    sq = th.zeros(n_total, device=DEV)
    grad = th.zeros(n_total, device=DEV)
    tail = th.zeros(DP_TAIL, device=DEV)
    scalars = th.zeros(64, device=DEV)
    scratch = th.zeros((n_total + 255) // 256, device=DEV)
    ptrs = (C.c_void_p * 2)(*[b.data_ptr() for b in bufs])
    a = s.args
    nat.check(nat.lib().mal_peer_allreduce_clip_rmsprop(ptrs, 2, nat.ptr(agent), n_agent, nat.ptr(mixer), n_total - n_agent,
                                                        nat.ptr(grad), nat.ptr(tail), DP_TAIL, nat.ptr(sq), a.lr,
                                                        a.optim_alpha, a.optim_eps, a.grad_norm_clip, nat.ptr(scalars),
                                                        nat.ptr(scratch), 0, nat.current_stream()),
              "mal_peer_allreduce_clip_rmsprop")
    th.cuda.synchronize()
    norm, (g_clip,) = O.clip_grad_norm([_ref_flat(ref)], a.grad_norm_clip)
    assert abs(float(scalars[nat.SC_GRAD_NORM]) - norm) <= TOL * norm
    assert_close(grad.cpu().numpy(), g_clip, TOL, "all-reduced gradient")
    raw = tail.cpu().numpy()
    assert abs(raw[0] / raw[4] - ref["loss"]) <= TOL * ref["loss"]
    assert abs(raw[3] / (raw[4] * 5) - ref["stats"]["target_mean"]) <= TOL * max(1.0, abs(ref["stats"]["target_mean"]))
    p1, _ = O.rmsprop_update(p0, g_clip, np.zeros(n_total), a.lr, a.optim_alpha, a.optim_eps)
    assert_close(np.concatenate([agent.cpu().numpy(), mixer.cpu().numpy()]), p1, TOL, "parameters after the step")
