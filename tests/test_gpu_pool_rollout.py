"""Per-match policies on the GPU: one pooled launch over B matches, match b playing row ids[b] of a [K, P] agent table.

Each match must get bit for bit what the plain step computes over the WHOLE batch with its policy (same variant band,
same injected draws), and whole rollouts must equal the reference loop oracle played match by match with that match's
parameters."""
import ctypes as C

import numpy as np
import pytest
import torch as th

import ma_league_b200 as M
from ma_league_b200 import _native as nat
from ma_league_b200.components.action_selectors import make_select_struct
from ma_league_b200.league import DeviceAgentPool, cross_play_returns
from ma_league_b200.steppers import BatchedEpisodeStepper, SyntheticVecEnv
from ma_league_b200.synthetic import make_args, make_scheme
from oracle import np_oracle as O
from tests.gpu_helpers import np_params
from tests.helpers import assert_close
from tests.input_layout_ref import LAYOUTS, OracleMAC

pytestmark = pytest.mark.gpu
DEV = "cuda"


def _table(K, d_in, A, seed):
    g = th.Generator().manual_seed(seed)
    P = nat.lib().mal_agent_param_count(d_in, A)
    return (th.randn(K, P, generator=g) * 0.15).to(DEV), P


def _unflat(row, d_in, A):
    shapes = [("fc1.weight", (64, d_in)), ("fc1.bias", (64,)), ("gru.weight_ih", (192, 64)), ("gru.weight_hh", (192, 64)),
              ("gru.bias_ih", (192,)), ("gru.bias_hh", (192,)), ("fc2.weight", (A, 64)), ("fc2.bias", (A,))]
    out, o = {}, 0
    r = row.detach().cpu().double().numpy()
    for k, s in shapes:
        n = int(np.prod(s))
        out[k] = r[o:o + n].reshape(s)
        o += n
    return out


def _inputs(bs, N, A, OBS, seed):
    g = th.Generator().manual_seed(seed)
    obs = th.randn(bs, N, OBS, generator=g).to(DEV)
    last = th.nn.functional.one_hot(th.randint(0, A, (bs, N), generator=g), A).float().to(DEV)
    h = (th.randn(bs * N, 64, generator=g) * 0.5).to(DEV)
    avail = (th.rand(bs, N, A, generator=g) < 0.6).int()
    avail[..., 0] = 1
    u = th.rand(bs, N, generator=g)
    e = th.empty(bs * N, A).exponential_(generator=g)
    return obs, last, h, avail.to(DEV), u, e


def _step(table_or_row, pool, bs, N, A, OBS, obs, last, h, avail, u=None, e=None, eps=0.5, seed=None):
    rows = bs * N
    q = th.empty(rows, A, device=DEV)
    h_out = th.empty(rows, 64, device=DEV)
    out = th.empty(2, rows, dtype=th.long, device=DEV)
    if seed is not None:
        th.manual_seed(seed)
    s, keep = make_select_struct(avail, eps, out[0], out[1], None, u, e)
    lib = nat.lib()
    common = (rows, N, OBS, A, 0, obs.data_ptr(), N * OBS, last.data_ptr(), N * A, h.data_ptr(), h_out.data_ptr(),
              q.data_ptr(), C.byref(s), nat.current_stream(0))
    if pool is None:
        nat.check(lib.mal_agent_step(table_or_row.data_ptr(), *common), "mal_agent_step")
    else:
        K, sched = pool
        nat.check(lib.mal_agent_step_pool(table_or_row.data_ptr(), table_or_row.stride(0), K, sched.data_ptr(), *common),
                  "mal_agent_step_pool")
    th.cuda.synchronize()
    return q, h_out, out[0]


def _schedule(ids, N, K, status=None):
    lib = nat.lib()
    nb = lib.mal_policy_schedule_bytes(len(ids), N, K)
    assert nb > 0
    sched = th.empty(nb // 4, dtype=th.int32, device=DEV)
    ids_d = th.as_tensor(ids, dtype=th.int32, device=DEV)
    nat.check(lib.mal_policy_schedule(ids_d.data_ptr(), len(ids), N, K, sched.data_ptr(),
                                      status.data_ptr() if status is not None else None, nat.current_stream(0)),
              "mal_policy_schedule")
    return sched


SHAPES = [(5, 1), (5, 5), (5, 32), (5, 400), (20, 1024)]     # (N, bs): latency, latency, latency, register, stream kernel


def _dims(N):
    return 6 + N, 8 + 8 * N            # A, OBS (SURVEY.md section 8 config table)


@pytest.mark.parametrize("N,bs", SHAPES)
@pytest.mark.parametrize("K,mode", [(1, "random"), (3, "random"), (8, "random"), (8, "equal")])
def test_pooled_step_equals_plain_step_per_match(N, bs, K, mode):
    A, OBS = _dims(N)
    d_in = OBS + A + N
    table, P = _table(K, d_in, A, seed=K + bs)
    obs, last, h, avail, u, e = _inputs(bs, N, A, OBS, seed=bs)
    g = th.Generator().manual_seed(100 + bs)
    if mode == "equal":
        ids = [K - 1] * bs
    else:
        ids = th.randint(0, K, (bs,), generator=g).tolist()
        if K > 1:
            ids = [i if i != 1 else 0 for i in ids]            # policy 1 plays no match
    sched = _schedule(ids, N, K)
    used = int(sched[0])
    assert used <= (bs * N + 7) // 8 + min(K, bs) - 1
    qp, hp, ap = _step(table, (K, sched), bs, N, A, OBS, obs, last, h, avail, u, e)
    ids_t = th.tensor(ids)
    for k in sorted(set(ids)):
        row = table[k].clone()                                   # 16-byte aligned copy, the plain entry's contract
        q1, h1, a1 = _step(row, None, bs, N, A, OBS, obs, last, h, avail, u, e)
        m = (ids_t == k).repeat_interleave(N).to(DEV)
        assert th.equal(qp[m], q1[m]) and th.equal(hp[m], h1[m]) and th.equal(ap[m], a1[m]), k
    # fp64 oracle, a few matches
    inp = np.concatenate([obs.cpu().double().numpy().reshape(bs * N, OBS), last.cpu().double().numpy().reshape(bs * N, A),
                          np.tile(np.eye(N), (bs, 1))], 1)
    for b in sorted({0, bs // 2, bs - 1}):
        sl = slice(b * N, (b + 1) * N)
        qo, ho, _ = O.drqn_step(_unflat(table[ids[b]], d_in, A), inp[sl], h[sl].cpu().double().numpy())
        assert_close(qp[sl].cpu().numpy(), qo, 1e-5, "q")
        assert_close(hp[sl].cpu().numpy(), ho, 1e-5, "h")


@pytest.mark.parametrize("N,bs", [(5, 32), (5, 400), (20, 1024)])
def test_one_policy_with_philox_draws_is_the_plain_step(N, bs):
    A, OBS = _dims(N)
    table, P = _table(1, OBS + A + N, A, seed=9)
    obs, last, h, avail, _, _ = _inputs(bs, N, A, OBS, seed=3)
    sched = _schedule([0] * bs, N, 1)
    qp, hp, ap = _step(table, (1, sched), bs, N, A, OBS, obs, last, h, avail, seed=1234)
    q1, h1, a1 = _step(table[0].clone(), None, bs, N, A, OBS, obs, last, h, avail, seed=1234)
    assert th.equal(qp, q1) and th.equal(hp, h1) and th.equal(ap, a1)


def test_out_of_range_id_sets_status_and_reads_nothing_outside_the_table():
    N, bs, K = 5, 6, 3
    A, OBS = _dims(N)
    table, P = _table(K, OBS + A + N, A, seed=1)
    obs, last, h, avail, u, e = _inputs(bs, N, A, OBS, seed=2)
    status = th.zeros(1, dtype=th.int32, device=DEV)
    ids = [0, 7, 2, -1, 1, 2]
    sched = _schedule(ids, N, K, status)
    assert int(status) == 1
    qp, hp, ap = _step(table, (K, sched), bs, N, A, OBS, obs, last, h, avail, u, e)
    ok = th.tensor([i in range(K) for i in ids]).repeat_interleave(N).to(DEV)
    for k in range(K):
        q1, h1, _ = _step(table[k].clone(), None, bs, N, A, OBS, obs, last, h, avail, u, e)
        m = th.tensor([i == k for i in ids]).repeat_interleave(N).to(DEV)
        assert th.equal(qp[m], q1[m])
    assert ok.sum() == 4 * N
    th.cuda.synchronize()


# ------------------------------------------------------------------ controllers and the stepper
N, A, OBS, S, LIMIT = 3, 9, 32, 48, 12


def _macs(n, seed, **over):
    th.manual_seed(seed)
    args = make_args(N, A, S, mixer="vdn", device=DEV, batch_size_run=1, **over)
    scheme, groups, pre = make_scheme(N, A, OBS, S)
    buf = M.ReplayBuffer(scheme, groups, 8, LIMIT + 1, preprocess=pre, device=DEV)
    return args, scheme, groups, pre, [M.mac_REGISTRY["basic"](buf.scheme, groups, args) for _ in range(n)]


@pytest.mark.parametrize("layout", LAYOUTS)
@pytest.mark.parametrize("n_teams", [1, 2])
@pytest.mark.parametrize("fuse", [True, False])
def test_pooled_rollout_against_the_reference_loop_oracle(layout, n_teams, fuse):
    from oracle import rollout_oracle as RO
    last, aid = layout
    K, B, T_ENV = 4, 7, 25000                                    # epsilon = 0.525
    args, scheme, groups, pre, macs = _macs(n_teams + K, 3, obs_last_action=last, obs_agent_id=aid)
    players, pol = macs[:n_teams], macs[n_teams:]
    table = th.stack([m.agent.flat_params().detach().clone() for m in pol])
    g = th.Generator().manual_seed(8)
    ids = [th.randint(0, K, (B,), generator=g).tolist() for _ in range(n_teams)]
    for m, i in zip(players, ids):
        m.set_match_policies(table, i)
    env = SyntheticVecEnv(B, N, A, OBS, S, LIMIT, n_teams=n_teams, seed=11, device=DEV, min_len=3)
    U = [[th.rand(B, N, generator=g) for _ in range(LIMIT + 1)] for _ in range(n_teams)]
    E = [[th.empty(B * N, A).exponential_(generator=g) for _ in range(LIMIT + 1)] for _ in range(n_teams)]
    st = BatchedEpisodeStepper(args, None, env, sync_every=1, fuse=fuse)
    st.initialize(scheme, groups, pre, players[0], players[1] if n_teams == 2 else None)
    st.t_env = T_ENV
    out = st.run(test_mode=False, draws=lambda k, t: (U[k][t], E[k][t]))
    batches, info = out[:-1], out[-1]
    lens = env.lengths.cpu().numpy()
    for b in range(B):
        penv = RO.PlaybackEnv(env._obs[:, b].cpu().numpy(), env._state[:, b].cpu().numpy(), env._avail[:, b].cpu().numpy(),
                              env._noise[:, b].cpu().numpy(), lens[b], LIMIT)
        omacs = [OracleMAC(np_params(pol[ids[k][b]].agent), N, A, dtype=np.float64, last_action=last, agent_id=aid,
                           draws=(lambda t, k=k: (U[k][t][b].numpy(), E[k][t].view(B, N, A)[b].numpy())))
                 for k in range(n_teams)]
        ref_batches, _, ref_steps = RO.run_episode(penv, omacs, (N, A, OBS, S), t_env=T_ENV, test_mode=False)
        assert ref_steps == lens[b] == int(info["episode_steps"][b])
        for k in range(n_teams):
            for key, ref in ref_batches[k].items():
                got = batches[k][key][b].cpu().numpy()
                if key == "reward":
                    assert np.allclose(got, ref, rtol=1e-6, atol=1e-6), (key, b, k)
                else:
                    assert np.array_equal(got, ref), (key, b, k)


def test_two_pooled_teams_launch_count():
    args, scheme, groups, pre, macs = _macs(2, 4)
    table = th.stack([macs[0].agent.flat_params().detach(), macs[1].agent.flat_params().detach()])
    n0 = nat.lib().mal_launch_count()
    macs[0].set_match_policies(table, [0, 1, 1, 0])
    macs[1].set_match_policies(table, [1, 1, 0, 0])
    assert nat.lib().mal_launch_count() - n0 == 2
    env = SyntheticVecEnv(4, N, A, OBS, S, LIMIT, n_teams=2, seed=2, device=DEV, min_len=LIMIT)
    st = BatchedEpisodeStepper(args, None, env, sync_every=4)
    st.initialize(scheme, groups, pre, macs[0], macs[1])
    for m in macs:
        m.action_selector.validate = False
    n0 = nat.lib().mal_launch_count()
    st.run(test_mode=True)
    assert nat.lib().mal_launch_count() - n0 == 2 * (LIMIT + 1)


def test_cross_play_equals_single_pair_runs():
    K, reps = 3, 2
    args, scheme, groups, pre, macs = _macs(2 + K, 5)
    home, away, pol = macs[0], macs[1], macs[2:]
    table = th.stack([m.agent.flat_params().detach().clone() for m in pol])
    n = K * K * reps
    env_ids = list(range(n))
    env = SyntheticVecEnv(n, N, A, OBS, S, LIMIT, n_teams=2, seed=3, device=DEV, env_ids=env_ids, min_len=3)
    st = BatchedEpisodeStepper(args, None, env)
    st.initialize(scheme, groups, pre, home, away)
    ret = cross_play_returns(st, home, away, table, reps)
    assert ret.shape == (K, K) and home.match_policies is None and away.match_policies is None
    for i in range(K):
        for j in range(K):
            m = [(i * K + j) * reps + r for r in range(reps)]
            home.load_state_dict(pol[i].agent.state_dict())
            away.load_state_dict(pol[j].agent.state_dict())
            env1 = SyntheticVecEnv(reps, N, A, OBS, S, LIMIT, n_teams=2, seed=3, device=DEV, env_ids=m, min_len=3)
            st1 = BatchedEpisodeStepper(args, None, env1)
            st1.initialize(scheme, groups, pre, home, away)
            _, _, info = st1.run(test_mode=True)
            assert th.equal(ret[i, j], info["episode_returns"][0].view(1, 1, reps).mean(dim=2)[0, 0]), (i, j)


def test_clearing_restores_the_own_agent_path():
    args, scheme, groups, pre, macs = _macs(2, 6)
    mac, other = macs
    pool = DeviceAgentPool(other)
    pool.sync()
    B = 4
    env = SyntheticVecEnv(B, N, A, OBS, S, LIMIT, n_teams=1, seed=1, device=DEV, min_len=3)
    st = BatchedEpisodeStepper(args, None, env)
    st.initialize(scheme, groups, pre, mac)
    ref, _ = st.run(test_mode=True)
    ref = {k: v.clone() for k, v in ref.data.transition_data.items()}
    mac.set_match_policies(pool.pool, [0] * B)
    pooled, _ = st.run(test_mode=True)                           # plays `other`
    mac.set_match_policies(None)
    again, _ = st.run(test_mode=True)
    for k, v in ref.items():
        assert th.equal(again[k], v), k
    st2 = BatchedEpisodeStepper(args, None, env)
    st2.initialize(scheme, groups, pre, other)
    ob, _ = st2.run(test_mode=True)
    for k in ref:
        assert th.equal(pooled[k], ob[k]), k
    # a pool.sync() between runs takes effect at the next step
    mac.set_match_policies(pool.pool, [0] * B)
    with th.no_grad():
        for p in other.agent.parameters():
            p.mul_(0.5)
    pool.sync()
    p2, _ = st.run(test_mode=True)
    o2, _ = st2.run(test_mode=True)
    for k in ref:
        assert th.equal(p2[k], o2[k]), k


def test_rejections():
    args, scheme, groups, pre, macs = _macs(1, 7)
    mac = macs[0]
    P = mac.agent.flat_params().numel()
    with pytest.raises(ValueError, match="architectures differ"):
        mac.set_match_policies(th.zeros(2, P + 1, device=DEV), [0, 1])
    with pytest.raises(ValueError):
        mac.set_match_policies(th.zeros(2, P, device=DEV), [0, 2])
    with pytest.raises(ValueError):
        mac.set_match_policies(th.zeros(2, P, device=DEV), th.tensor([-1, 0], device=DEV))
    with pytest.raises(nat.MalError):
        mac.set_match_policies(th.zeros(2, P), [0, 1])
    mac.set_match_policies(th.zeros(2, P, device=DEV), [0, 1, 1])
    with pytest.raises(nat.MalError):
        mac.init_hidden(4)
    mac.init_hidden(3)
    # forward under autograd_forward with grad mode on
    ag_args, scheme2, groups2, _, (mac2,) = _macs(1, 7, autograd_forward=True)
    mac2.set_match_policies(th.zeros(2, P, device=DEV), [0, 1])
    mac2.init_hidden(2)
    eb = M.EpisodeBatch(scheme2, groups2, 2, LIMIT + 1, preprocess=pre, device=DEV)
    with pytest.raises(nat.MalError):
        mac2.forward(eb, 0)
    with th.no_grad():
        assert mac2.forward(eb, 0).shape == (2, N, A)
    # the dqn agent and an ensemble with members
    _, _, _, _, (dqn,) = _macs(1, 7, agent="dqn")
    with pytest.raises(nat.MalError):
        dqn.set_match_policies(th.zeros(2, dqn.agent.flat_params().numel(), device=DEV), [0, 1])
    args_e, scheme_e, groups_e, _, _ = _macs(0, 7)
    ens = M.EnsembleMAC(M.ReplayBuffer(scheme_e, groups_e, 2, LIMIT + 1, preprocess=pre, device=DEV).scheme, groups_e, args_e)
    ens.load_state_dict(ensemble={1: ens.agent.state_dict()})
    with pytest.raises(nat.MalError):
        ens.set_match_policies(th.zeros(2, P, device=DEV), [0, 1])
