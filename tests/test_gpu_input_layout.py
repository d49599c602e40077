"""Agent inputs with obs_last_action / obs_agent_id switched off, on the GPU: the learner step on every path that reads
fc1's input, act-select and the fused rollout step, against the numpy reference of tests/input_layout_ref.py."""
import numpy as np
import pytest
import torch as th

from oracle import np_oracle as O
from tests.gpu_helpers import seeded_system, np_params, np_batch, split_grad
from tests.helpers import assert_close, rel_err
from tests.input_layout_ref import LAYOUTS, build_inputs, d_in, learner_forward_backward, OracleMAC
from tests.test_gpu_learner import TOL, _FLAVOURS, _discrete_choices

pytestmark = pytest.mark.gpu
DEV = "cuda"
NEW_LAYOUTS = [l for l in LAYOUTS if l != (True, True)]


def _lib():
    from ma_league_b200 import _native as nat
    return nat, nat.lib()


class options:
    """`with options(fuse_agent_in=0, ...)`: library options of this thread, restored to their defaults afterwards."""
    DEFAULTS = dict(fuse_agent_in=1, tc_pipelined=1, rec_tc=1, fc1_fused=1, reduce_tc=1, actsel_lat=1)

    def __init__(self, **kv):
        self.kv = kv

    def __enter__(self):
        nat, lib = _lib()
        for k, v in self.kv.items():
            nat.check(lib.mal_set_option(k.encode(), v), "mal_set_option")

    def __exit__(self, *exc):
        nat, lib = _lib()
        for k in self.kv:
            nat.check(lib.mal_set_option(k.encode(), self.DEFAULTS[k]), "mal_set_option")
        return False


def _system(N, B, TT, mixer, layout, seed, **kw):
    last, aid = layout
    s = seeded_system(N, B, TT, mixer, True, seed=seed, obs_last_action=last, obs_agent_id=aid, **kw)
    A, OBS = 6 + N, 8 + 8 * N
    assert s.mac.agent.fc1.weight.shape[1] == d_in(OBS, A, N, last, aid)
    return s


def _check(s, mixer, layout):
    """Forward intermediates, loss and every gradient against the fp64 reference at 1e-5; discrete choices (double-Q
    arg-max, ReLU / abs derivatives) may differ only on verified near-ties (as in test_gpu_learner)."""
    nat, lib = _lib()
    last, aid = layout
    before = {k: lib.mal_stat(k.encode()) for k in _FLAVOURS}
    grads = split_grad(s.learner.forward_backward(s.batch), s.learner)
    th.cuda.synchronize()
    ran = {k: lib.mal_stat(k.encode()) - before[k] for k in _FLAVOURS}
    it = {k: v.cpu().numpy() for k, v in s.learner.intermediates(s.batch).items()}
    L = s.learner
    args = (np_params(s.mac.agent), np_params(L.target_mac.agent), np_params(L.mixer) if mixer == "qmix" else None,
            np_params(L.target_mixer) if mixer == "qmix" else None, np_batch(s.batch))
    kw = dict(mixer=mixer, double_q=True, gamma=s.args.gamma, dtype=np.float64, last_action=last, agent_id=aid)
    ref = learner_forward_backward(*args, **kw)
    assert_close(it["hout"], ref["hout"], TOL, "hidden states")
    assert_close(it["chosen"], ref["chosen"], TOL, "chosen")
    flips = np.argwhere(it["argmax"].astype(np.int64) != ref["argmax"])
    if len(flips):
        oq = ref["mac_out"][:, 1:].copy()
        oq[np_batch(s.batch)["avail_actions"][:, 1:] == 0] = O.NEG_MASK
        for b, t, n in flips:
            row = oq[b, t, n]
            gap = abs(row[ref["argmax"][b, t, n]] - row[it["argmax"][b, t, n]])
            assert gap <= 1e-5 * max(1.0, np.abs(row[row > O.NEG_MASK]).max()), ("argmax flip without a near-tie", b, t, n)
        assert len(flips) <= 1 + it["argmax"].size // 100000
    discrete, n_diff = _discrete_choices(it, ref, mixer)
    if len(flips) or n_diff:
        ref = learner_forward_backward(*args, argmax_override=it["argmax"].astype(np.int64), discrete=discrete, **kw)
    assert_close(it["q_tot"], ref["q_tot"], TOL, "q_tot")
    assert_close(it["target_q_tot"], ref["target_q_tot"], TOL, "target_q_tot")
    assert abs(it["scalars"][1] - ref["loss"]) <= TOL * abs(ref["loss"])
    for k, v in ref["agent_grads"].items():
        assert_close(grads["agent." + k], v, TOL, "grad " + k)
    for k, v in ref["mixer_grads"].items():
        assert_close(grads["mixer." + k], v, TOL, "grad mixer " + k)
    return ran, ref


def _after_step_matches(s, mixer, ref):
    """train() (clip + RMSprop included) after _check on the same batch: parameters against the reference update of the
    gradients _check verified, at 1e-5."""
    L = s.learner
    names = ["agent." + k for k in np_params(s.mac.agent)] + (["mixer." + k for k in np_params(L.mixer)] if mixer == "qmix" else [])
    p0 = [v for v in np_params(s.mac.agent).values()] + ([v for v in np_params(L.mixer).values()] if mixer == "qmix" else [])
    grads = list(ref["agent_grads"].values()) + list(ref["mixer_grads"].values())
    _, clipped = O.clip_grad_norm(grads, s.args.grad_norm_clip)
    L.train(s.batch, 0, 0)
    th.cuda.synchronize()
    got = list(np_params(s.mac.agent).values()) + (list(np_params(L.mixer).values()) if mixer == "qmix" else [])
    for n, v, g, new in zip(names, p0, clipped, got):
        ref_new, _ = O.rmsprop_update(v.astype(np.float64), g, np.zeros_like(g), s.args.lr, s.args.optim_alpha, s.args.optim_eps)
        assert rel_err(new, ref_new) <= TOL, ("param " + n, rel_err(new, ref_new))   # norm-wise


# ---------------------------------------------------------------------------------------------------------- learner
@pytest.mark.parametrize("layout", NEW_LAYOUTS)
@pytest.mark.parametrize("N,B,TT,mixer", [
    (5, 32, 21, "qmix"), (5, 32, 21, "vdn"),       # d_in <= 64 (5v5: 48 / 53 / 59 columns)
    (10, 32, 9, "qmix"), (10, 32, 9, "vdn"),       # 64 < d_in <= 128 (10v10: 88 / 98 / 104)
])
def test_learner_against_reference(N, B, TT, mixer, layout):
    s = _system(N, B, TT, mixer, layout, seed=300 + N)
    ran, ref = _check(s, mixer, layout)
    assert ran["agent_in_fused"] == 1                 # OBS % 4 == 0: the fused input GEMM takes fc1
    _after_step_matches(s, mixer, ref)


@pytest.mark.parametrize("layout", NEW_LAYOUTS)
def test_learner_wide_input_k_reduce_fc1(layout):
    """d_in > 128 at 20v20 dimensions (168 / 188 / 194 columns; 194 = 3 x 64 + 2 leaves a two-column one-hot remainder
    to epilogue 1 of the fused input GEMM, 168 has no one-hot tail at all) with the fc1 gradient in k_reduce_fc1."""
    s = _system(20, 4, 6, "qmix", layout, seed=320)
    with options(reduce_tc=2, tc_pipelined=2):
        ran, _ = _check(s, "qmix", layout)
    assert ran["reduce_fc1"] >= 1 and ran["agent_in_fused"] == 1


@pytest.mark.parametrize("layout", NEW_LAYOUTS)
@pytest.mark.parametrize("opts,expect", [
    (dict(fuse_agent_in=0), dict(agent_in_fused=0, linear_tc=1)),                 # k_linear_tc fc1 + W_ih
    (dict(fuse_agent_in=0, tc_pipelined=2), dict(agent_in_fused=0, linear_tc2=1)),  # k_linear_tc2
    (dict(rec_tc=2), dict(agent_in_fused=1, rec_tc=1)),                            # tiled gi for the tensor-core recurrence
    (dict(reduce_tc=2, fc1_fused=0), dict(reduce_tc_swap=1, reduce_fc1=0)),        # k_reduce_tc3 SWAP over d_in > 64
    (dict(reduce_tc=0), dict(reduce_ffma=1, reduce_fc1=0)),                        # k_reduce_group
], ids=["linear_tc", "linear_tc2", "rec_tc", "reduce_tc_swap", "reduce_group"])
def test_learner_forced_paths(opts, expect, layout):
    s = _system(10, 32, 9, "qmix", layout, seed=340)
    with options(**opts):
        ran, _ = _check(s, "qmix", layout)
    for k, v in expect.items():
        assert (ran[k] >= 1) == bool(v), (k, ran)


@pytest.mark.parametrize("layout", NEW_LAYOUTS)
@pytest.mark.parametrize("N,B,TT,mixer", [(5, 8, 9, "qmix"), (10, 6, 12, "vdn")])
def test_dqn_agent_learner(N, B, TT, mixer, layout):
    s = _system(N, B, TT, mixer, layout, seed=360 + N, agent="dqn")
    assert type(s.mac.agent).__name__ == "DQNAgentNetwork"
    _, ref = _check(s, mixer, layout)
    _after_step_matches(s, mixer, ref)


@pytest.mark.parametrize("layout", [(False, True), (False, False)])
def test_cuda_graph_replay_equals_eager(layout):
    def run(graphs):
        s = _system(3, 4, 9, "qmix", layout, seed=21, learner_log_interval=0)
        s.learner.use_graphs = graphs
        s2 = _system(3, 4, 9, "qmix", layout, seed=22)
        for i in range(8):
            s.learner.train(s.batch if i % 2 == 0 else s2.batch, t_env=i, episode_num=i)
        th.cuda.synchronize()
        if graphs:
            assert sum(1 for v in s.learner._graphs.values() if v) == 2
        return np_params(s.mac.agent), np_params(s.learner.mixer), s.learner.optimiser.flat_sq.cpu().numpy(), \
            {k: v[0] for k, v in s.logger.stats.items()}
    a, b = run(True), run(False)
    for x, y in zip(a[:2], b[:2]):
        for k in x:
            assert np.array_equal(x[k], y[k]), k
    assert np.array_equal(a[2], b[2]) and a[3] == b[3]


# ---------------------------------------------------------------------------------------------------------- act-select
def _same_choice(got, ref, q, greedy):
    """Actions equal, except a greedy pick on a genuine near-tie of the fp64 Q-values."""
    for idx in np.argwhere(got != ref):
        qi = q[tuple(idx)]
        assert greedy[tuple(idx)] == 1 and abs(qi[got[tuple(idx)]] - qi[ref[tuple(idx)]]) <= 1e-5 * max(1.0, np.abs(qi).max()), idx
    assert (got != ref).sum() <= 1 + got.size // 10000


@pytest.mark.parametrize("layout", NEW_LAYOUTS)
@pytest.mark.parametrize("bs,agent", [(1, "rnn"), (32, "rnn"), (256, "rnn"), (1024, "rnn"), (32, "dqn")])
def test_select_actions_against_reference(bs, agent, layout):
    """One launch per select_actions call; bs = 1 / 32 take k_agent_step_lat, 256 k_agent_step (more CTAs than SMs),
    1024 k_agent_step_stream, the DQN agent its own step; injected (u, e) draws, epsilon 0.525."""
    nat, lib = _lib()
    last, aid = layout
    N, TT, T_ENV = 5, 4, 25000
    s = _system(N, bs, TT, "vdn", layout, seed=bs, agent=agent, var_len=False)   # every step filled: avail rows non-empty
    mac = s.mac
    A = mac.n_actions
    assert mac._fusable()
    p = {k: v.astype(np.float64) for k, v in np_params(mac.agent).items()}
    b = np_batch(s.batch)
    gen = th.Generator().manual_seed(bs + 1)
    mac.init_hidden(bs)
    h = np.zeros((bs * N, 64))
    for t in range(TT):
        u, e = th.rand(bs, N, generator=gen), th.empty(bs * N, A).exponential_(generator=gen)
        n0 = lib.mal_launch_count()
        acts, greedy = mac.select_actions(s.batch, t_ep=t, t_env=T_ENV, u=u, e=e)
        th.cuda.synchronize()
        assert lib.mal_launch_count() - n0 == 1
        inp = build_inputs(b["obs"].astype(np.float64), b["actions_onehot"].astype(np.float64), t, last, aid)
        q, h, _ = (O.dqn_step(p, inp) if agent == "dqn" else O.drqn_step(p, inp, h))
        q = q.reshape(bs, N, A)
        eps = mac.action_selector.epsilon
        ra, rg = O.eps_greedy_select(q, b["avail_actions"][:, t], eps, u.numpy(), e.numpy())
        assert np.array_equal(greedy.cpu().numpy(), rg), t
        _same_choice(acts.cpu().numpy(), ra, q, rg)
        if agent == "rnn":
            assert_close(mac.hidden_states.reshape(bs * N, 64).cpu().numpy(), h, 1e-5, "hidden t=%d" % t)


@pytest.mark.parametrize("layout", NEW_LAYOUTS)
def test_philox_stream_matches_torch_cuda_generator(layout):
    """rng_mode 1 (no injected draws): the fused select consumes torch's CUDA generator exactly like the reference's
    rand_like + Categorical.sample on the same Q-values (action_selectors.py:52-61)."""
    from torch.distributions import Categorical
    bs, N = 32, 5
    s = _system(N, bs, 3, "vdn", layout, seed=7, var_len=False)
    mac = s.mac
    mac.init_hidden(bs)
    h = mac.hidden_states
    for t in range(3):
        th.manual_seed(99 + t)
        a, g = mac.select_actions(s.batch, t_ep=t, t_env=30000)
        h_sel = mac.hidden_states
        mac.hidden_states = h
        q = mac.forward(s.batch, t)                              # the same step without the selection tail
        assert th.allclose(mac.hidden_states, h_sel, rtol=1e-6, atol=1e-6)
        h = mac.hidden_states
        avail = s.batch["avail_actions"][:, t]
        eps = mac.action_selector.epsilon
        th.manual_seed(99 + t)
        masked = q.clone()
        masked[avail == 0.0] = -float("inf")
        pick_random = (th.rand_like(q[:, :, 0]) < eps).long()
        ref_a = pick_random * Categorical(avail.float()).sample().long() + (1 - pick_random) * masked.max(dim=2)[1]
        assert th.equal(a, ref_a) and th.equal(g, 1 - pick_random)


# ---------------------------------------------------------------------------------------------------------- rollout
@pytest.mark.parametrize("layout", NEW_LAYOUTS)
@pytest.mark.parametrize("n_teams", [1, 2])
def test_fused_rollout_against_the_reference_loop(n_teams, layout):
    """BatchedEpisodeStepper through the one-launch rollout step (one launch per team and timestep) leaves, match by match,
    exactly the episode batch of the reference loop (rollout_oracle) with the switched agent input."""
    import ma_league_b200 as M
    from ma_league_b200.steppers import BatchedEpisodeStepper, SyntheticVecEnv
    from ma_league_b200.synthetic import make_args, make_scheme
    from oracle import rollout_oracle as RO
    nat, lib = _lib()
    last, aid = layout
    N, A, OBS, S, LIMIT, B, T_ENV = 3, 9, 32, 48, 12, 5, 25000
    th.manual_seed(3)
    args = make_args(N, A, S, mixer="vdn", device=DEV, batch_size_run=1, obs_last_action=last, obs_agent_id=aid)
    scheme, groups, pre = make_scheme(N, A, OBS, S)
    buf = M.ReplayBuffer(scheme, groups, 8, LIMIT + 1, preprocess=pre, device=DEV)
    macs = [M.mac_REGISTRY["basic"](buf.scheme, groups, args) for _ in range(n_teams)]
    assert all(m._rollout_fusable() for m in macs)
    env = SyntheticVecEnv(B, N, A, OBS, S, LIMIT, n_teams=n_teams, seed=11, device=DEV, min_len=3)
    gen = th.Generator().manual_seed(5)
    U = [[th.rand(B, N, generator=gen) for _ in range(LIMIT + 1)] for _ in range(n_teams)]
    E = [[th.empty(B * N, A).exponential_(generator=gen) for _ in range(LIMIT + 1)] for _ in range(n_teams)]
    st = BatchedEpisodeStepper(args, None, env, sync_every=LIMIT + 1, fuse=True)
    st.initialize(scheme, groups, pre, macs[0], macs[1] if n_teams == 2 else None)
    st.t_env = T_ENV
    for m in macs:
        m.action_selector.validate = False
    n0 = lib.mal_launch_count()
    out = st.run(test_mode=False, draws=lambda k, t: (U[k][t], E[k][t]))
    assert lib.mal_launch_count() - n0 == n_teams * (LIMIT + 1)
    batches, info = out[:-1], out[-1]
    lens = env.lengths.cpu().numpy()
    for b in range(B):
        penv = RO.PlaybackEnv(env._obs[:, b].cpu().numpy(), env._state[:, b].cpu().numpy(), env._avail[:, b].cpu().numpy(),
                              env._noise[:, b].cpu().numpy(), lens[b], LIMIT)
        omacs = [OracleMAC(np_params(m.agent), N, A, dtype=np.float64, last_action=last, agent_id=aid,
                           draws=(lambda t, k=k: (U[k][t][b].numpy(), E[k][t].view(B, N, A)[b].numpy())))
                 for k, m in enumerate(macs)]
        ref_batches, _, ref_steps = RO.run_episode(penv, omacs, (N, A, OBS, S), t_env=T_ENV, test_mode=False)
        assert ref_steps == lens[b] == int(info["episode_steps"][b])
        for k in range(n_teams):
            for key, ref in ref_batches[k].items():
                got = batches[k][key][b].cpu().numpy()
                if key == "reward":
                    assert np.allclose(got, ref, rtol=1e-6, atol=1e-6), (key, b, k)
                else:
                    assert np.array_equal(got, ref), (key, b, k)
