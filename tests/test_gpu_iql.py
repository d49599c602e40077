"""Independent Q-learners (`mixer: None`) through the CUDA learner step, against the fp64 IQL reference of
tests/iql_ref.py (q_learner.py:34-125 with self.mixer = None: per-agent TD errors, the mask broadcast over agents)."""
import os

import numpy as np
import pytest
import torch as th
import torch.distributed as dist
import torch.multiprocessing as mp

import ma_league_b200 as M
from ma_league_b200.synthetic import fill_episode_batch, synth_episode_data
from oracle import np_oracle as O
from tests import iql_ref as R
from tests.gpu_helpers import build_system, np_params, np_batch
from tests.helpers import assert_close, rel_err
from tests.test_data_parallel import _free_port
from tests.test_gpu_learner import _FLAVOURS, _discrete_choices

pytestmark = pytest.mark.gpu
TOL = 1e-5
STATS = ("loss", "grad_norm", "td_error_abs", "q_taken_mean", "target_mean")


def iql_system(N, B, TT, double_q=True, seed=0, device="cuda", last_action=True, agent_id=True, **kw):
    """seeded_system without a mixer: A = 6 + N, OBS = 8 + 8N, S = 16N, a perturbed target agent, variable lengths."""
    A, OBS, S = 6 + N, 8 + 8 * N, 16 * N
    th.manual_seed(seed)
    s = build_system(N, A, OBS, S, B, TT, None, double_q, device, obs_last_action=last_action, obs_agent_id=agent_id, **kw)
    gen = th.Generator().manual_seed(seed + 1)
    with th.no_grad():
        for p in s.learner.target_mac.parameters():
            p.add_(0.05 * th.randn(p.shape, generator=gen).to(device))
    data, lens = synth_episode_data(B, TT, N, A, OBS, S, gen, var_len=True, device=device)
    lens[0] = TT - 1
    s["batch"] = fill_episode_batch(M.EpisodeBatch(s.scheme, s.groups, B, TT, preprocess=s.pre, device=device), data, lens)
    s["layout"] = (last_action, agent_id)
    return s


def agent_grads(flat, learner):
    out, off = {}, 0
    for k, p in learner.mac.agent.named_parameters():
        out[k] = flat[off:off + p.numel()].view(p.shape).cpu().numpy().copy()
        off += p.numel()
    assert off == flat.numel()
    return out


def oracle(s, params, batch=None, **kw):
    """The fp64 IQL reference (tests/iql_ref.py) for this system's agent-input layout."""
    last, aid = s.layout
    return R.learner_forward_backward(params, np_params(s.learner.target_mac.agent),
                                      np_batch(s.batch) if batch is None else batch, last_action=last, agent_id=aid,
                                      double_q=bool(s.args.double_q), gamma=s.args.gamma, dtype=np.float64, **kw)


def forward_against_oracle(s, params=None):
    """One forward + backward on the device against the oracle at `params` (default: the device's own parameters, read
    back): chosen, arg-max, target max, [B,T,N] targets / td, mask, loss, the statistics, the counter and every gradient.
    Near-ties of the double-Q arg-max and the fc1 ReLU are handled as in test_gpu_learner._check_against_oracle_full.
    Returns (mal_stat flavour counts, oracle result)."""
    lib = M._native.lib()
    before = {k: lib.mal_stat(k.encode()) for k in _FLAVOURS + ("gru_balanced",)}
    grads = agent_grads(s.learner.forward_backward(s.batch), s.learner)
    th.cuda.synchronize()
    ran = {k: lib.mal_stat(k.encode()) - v for k, v in before.items()}
    it = {k: v.cpu().numpy() for k, v in s.learner.intermediates(s.batch).items()}
    p = np_params(s.mac.agent) if params is None else params
    ref = oracle(s, p)
    B, T, N = ref["chosen"].shape
    assert it["q_tot"].shape == it["targets"].shape == it["td"].shape == (B, T, N)
    assert_close(it["hout"], ref["hout"], TOL, "hidden states")
    assert_close(it["chosen"], ref["chosen"], TOL, "chosen")
    flips = np.argwhere(it["argmax"].astype(np.int64) != ref["argmax"])
    if len(flips):
        oq = ref["mac_out"][:, 1:].copy()
        oq[np_batch(s.batch)["avail_actions"][:, 1:] == 0] = O.NEG_MASK
        for b, t, n in flips:
            row = oq[b, t, n]
            gap = abs(row[ref["argmax"][b, t, n]] - row[it["argmax"][b, t, n]])
            assert gap <= 1e-5 * max(1.0, np.abs(row[row > O.NEG_MASK]).max()), ("argmax flip without a near-tie", b, t, n, gap)
        assert len(flips) <= 1 + it["argmax"].size // 100000, "%d argmax flips" % len(flips)
    discrete, n_diff = _discrete_choices(it, ref, None)
    if len(flips) or n_diff:
        ref = oracle(s, p, argmax_override=it["argmax"].astype(np.int64), discrete=discrete)
    assert_close(it["target_max"], ref["target_max"], TOL, "target_max")
    assert_close(it["mask"], ref["mask"], 0, "mask")
    assert np.array_equal(it["q_tot"], it["chosen"]) and np.array_equal(it["target_q_tot"], it["target_max"])
    assert_close(it["targets"], ref["targets"], TOL, "targets")
    assert_close(it["td"], ref["td"], TOL, "td")
    sc, st = it["scalars"], ref["stats"]
    assert abs(sc[M._native.SC_LOSS] - ref["loss"]) <= TOL * abs(ref["loss"])
    assert sc[M._native.SC_MASK_SUM] == st["mask_sum"] == N * ref["mask"].sum()
    for i, k in ((M._native.SC_TD_ABS, "td_error_abs"), (M._native.SC_Q_TAKEN, "q_taken_mean"),
                 (M._native.SC_TARGET, "target_mean")):
        assert abs(sc[i] - st[k]) <= TOL * max(1.0, abs(st[k])), (k, sc[i], st[k])
    assert int(sc[6:7].view(np.int32)[0]) == st["trained_steps"] == N * np.count_nonzero(ref["mask"])
    for k, v in ref["agent_grads"].items():
        assert_close(grads[k], v, TOL, "grad " + k)
    return ran, ref


def two_steps_against_oracle(s):
    """forward_against_oracle, then two train() steps (graphs on) chained through the oracle from the same start:
    parameters and square_avg after each step, the five logged statistics and the trained-step counter."""
    L, a = s.learner, s.args
    a.learner_log_interval = 0
    p = {k: v.astype(np.float64) for k, v in np_params(s.mac.agent).items()}
    sq = np.zeros(sum(v.size for v in p.values()))
    steps = 0
    ran = None
    for i in range(2):
        r, ref = forward_against_oracle(s, p)
        ran = ran or r
        g = np.concatenate([v.ravel() for v in ref["agent_grads"].values()])
        norm, (g_clip,) = O.clip_grad_norm([g], a.grad_norm_clip)
        p0 = np.concatenate([v.ravel() for v in p.values()])
        p1, sq = O.rmsprop_update(p0, g_clip, sq, a.lr, a.optim_alpha, a.optim_eps)
        L.train(s.batch, t_env=i, episode_num=0)
        th.cuda.synchronize()
        logged = {k[len("home_qlearner_"):]: v[0] for k, v in s.logger.stats.items()}
        want = dict(loss=ref["loss"], grad_norm=norm, **{k: ref["stats"][k] for k in STATS[2:]})
        for k in STATS:
            assert abs(logged[k] - want[k]) <= TOL * max(1.0, abs(want[k])), (i, k, logged[k], want[k])
        got = np.concatenate([v.ravel() for v in np_params(s.mac.agent).values()])
        assert_close(got, p1, TOL, "parameters after step %d" % (i + 1))
        assert_close(got - p0, p1 - p0, 1e-3, "update of step %d" % (i + 1))
        assert rel_err(L.optimiser.flat_sq.cpu().numpy(), sq) < 1e-4, "square_avg after step %d" % (i + 1)
        steps += ref["stats"]["trained_steps"]
        off = 0
        for k, v in p.items():
            p[k] = p1[off:off + v.size].reshape(v.shape)
            off += v.size
    assert s.mac.agent.trained_steps == steps
    assert all(q.grad is not None for q in L.parameters())
    return ran


# ---------------------------------------------------------------------------------------------- shapes and variations
@pytest.mark.parametrize("N,B,TT,agent,double_q,layout", [
    (3, 32, 201, "rnn", True, (True, True)),         # BASELINE.json 3v3 / 5v5 / 10v10 shapes, default heuristics
    (5, 32, 201, "rnn", True, (True, True)),
    (10, 128, 201, "rnn", True, (True, True)),
    (20, 16, 24, "rnn", True, (True, True)),         # 20v20 widths (d_in = 214) at a short T
    (2, 1, 3, "rnn", True, (True, True)),            # tiny
    (5, 32, 201, "dqn", True, (True, True)),
    (3, 8, 40, "dqn", False, (True, True)),
    (4, 8, 33, "rnn", False, (True, True)),
    (5, 16, 40, "rnn", True, (False, False)),        # both agent-input switches off
    (10, 4, 12, "dqn", True, (False, True)),
])
def test_iql_learner_against_oracle(N, B, TT, agent, double_q, layout):
    s = iql_system(N, B, TT, double_q, seed=100 + N + TT, agent=agent, last_action=layout[0], agent_id=layout[1])
    assert s.learner.mixer is None and s.learner.target_mixer is None
    ran = two_steps_against_oracle(s)
    if agent == "rnn" and (N, B) == (5, 32):
        assert ran["gru_balanced"] == 1, ran          # 320 chains > 2 x SMs: nothing beside the recurrence, balanced
    if (N, B) == (10, 128):
        assert ran["agent_in_fused"] == 1 and ran["reduce_ffma"] == 0, ran


@pytest.mark.parametrize("bwd_tc", [0, 1])
@pytest.mark.parametrize("N,B,TT", [(5, 32, 41), (3, 96, 7)])
def test_tensor_core_recurrence_forced(N, B, TT, bwd_tc):
    lib = M._native.lib()
    M._native.check(lib.mal_set_option(b"rec_tc", 2), "mal_set_option")
    M._native.check(lib.mal_set_option(b"rec_tc_bwd", bwd_tc), "mal_set_option")
    try:
        ran, _ = forward_against_oracle(iql_system(N, B, TT, True, seed=60 + N))
    finally:
        M._native.check(lib.mal_set_option(b"rec_tc", 1), "mal_set_option")
        M._native.check(lib.mal_set_option(b"rec_tc_bwd", 0), "mal_set_option")
    assert ran["rec_tc"] >= 1 and (ran["rec_tc_bwd"] >= 1) == bool(bwd_tc), ran


@pytest.mark.parametrize("graphs", [False, True])
def test_balanced_recurrence_default_is_bit_identical_to_unbalanced(graphs):
    """IQL, like VDN, runs nothing beside the forward recurrence, so the default takes the balanced schedule: parameters,
    optimiser state, statistics and the counter are bit-identical to gru_balance = 0, eagerly and through graphs."""
    lib = M._native.lib()

    def run(balance):
        M._native.check(lib.mal_set_option(b"gru_balance", balance), "mal_set_option")
        try:
            s = iql_system(5, 32, 201, True, seed=37, learner_log_interval=0)
            s.learner.use_graphs = graphs
            n0 = lib.mal_stat(b"gru_balanced")
            for i in range(4):
                s.learner.train(s.batch, t_env=i, episode_num=i)
            th.cuda.synchronize()
            return np_params(s.mac.agent), s.learner.optimiser.flat_sq.cpu().numpy(), \
                {k: v[0] for k, v in s.logger.stats.items()}, s.mac.agent.trained_steps, lib.mal_stat(b"gru_balanced") - n0
        finally:
            M._native.check(lib.mal_set_option(b"gru_balance", 1), "mal_set_option")
    a, b = run(1), run(0)
    assert a[4] >= 1 and b[4] == 0, (a[4], b[4])
    for k in a[0]:
        assert np.array_equal(a[0][k], b[0][k]), k
    assert np.array_equal(a[1], b[1]) and a[2] == b[2] and a[3] == b[3]


def test_cuda_graph_replay_equals_eager_launches():
    def run(graphs):
        s = iql_system(3, 4, 9, True, seed=21, learner_log_interval=0)
        s.learner.use_graphs = graphs
        s2 = iql_system(3, 4, 9, True, seed=22)
        for i in range(8):
            s.learner.train(s.batch if i % 2 == 0 else s2.batch, t_env=i, episode_num=i)
        th.cuda.synchronize()
        if graphs:
            assert sum(1 for v in s.learner._graphs.values() if v) == 2
        return np_params(s.mac.agent), s.learner.optimiser.flat_sq.cpu().numpy(), \
            {k: v[0] for k, v in s.logger.stats.items()}, s.mac.agent.trained_steps
    a, b = run(True), run(False)
    for k in a[0]:
        assert np.array_equal(a[0][k], b[0][k]), k
    assert np.array_equal(a[1], b[1]) and a[2] == b[2] and a[3] == b[3]


def test_train_from_buffer_against_oracle():
    """The fused input pipeline (sample into the staging batch, padding masked) against the oracle on the sampled ids,
    truncated as the reference does (ma_experiment.py:231-241)."""
    clip = 0.5
    s = iql_system(3, 6, 14, True, seed=33, buffer_size=24, learner_log_interval=0, clip=clip)
    gen = th.Generator().manual_seed(78)
    for _ in range(4):
        data, lens = synth_episode_data(6, 14, 3, 9, 32, 48, gen, var_len=True, device="cuda")
        lens = th.clamp(lens, max=10)
        data["terminated"].zero_()
        data["terminated"][th.arange(6), lens - 1] = 1
        s.buf.insert_episode_batch(fill_episode_batch(
            M.EpisodeBatch(s.scheme, s.groups, 6, 14, preprocess=s.pre, device="cuda"), data, lens))
    host_buf = np_batch(s.buf)
    L, a = s.learner, s.args
    for truncate in (False, True):
        p0 = np_params(s.mac.agent)
        sq0 = L.optimiser.flat_sq.cpu().numpy().astype(np.float64)
        np.random.seed(9)
        ids = np.random.choice(s.buf.episodes_in_buffer, 6, replace=False)
        np.random.seed(9)
        L.train_from_buffer(s.buf, 6, t_env=0, episode_num=0, truncate=truncate)
        th.cuda.synchronize()
        smp = {k: v[ids] for k, v in host_buf.items()}
        mt = O.max_t_filled(smp["filled"])
        ref = oracle(s, p0, {k: v[:, :mt] for k, v in smp.items()})
        g = np.concatenate([v.ravel() for v in ref["agent_grads"].values()])
        norm, (g_clip,) = O.clip_grad_norm([g], clip)
        st = {k: v[0] for k, v in s.logger.stats.items()}
        assert abs(st["home_qlearner_loss"] - ref["loss"]) <= TOL * abs(ref["loss"])
        assert abs(st["home_qlearner_grad_norm"] - norm) <= TOL * norm
        assert abs(st["home_qlearner_q_taken_mean"] - ref["stats"]["q_taken_mean"]) <= TOL * max(1, abs(ref["stats"]["q_taken_mean"]))
        assert_close(L._grad.cpu().numpy(), g_clip, TOL, "clipped gradient")
        flat0 = np.concatenate([v.ravel() for v in p0.values()]).astype(np.float64)
        p_ref, sq_ref = O.rmsprop_update(flat0, g_clip, sq0, a.lr, a.optim_alpha, a.optim_eps)
        assert_close(np.concatenate([v.ravel() for v in np_params(s.mac.agent).values()]), p_ref, TOL, "parameters")
        assert_close(L.optimiser.flat_sq.cpu().numpy(), sq_ref, TOL, "square_avg")


# ---------------------------------------------------------------------------------------------- data-parallel
def _dp_worker(rank, world, port, out, nccl, fused):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dev = "cuda:%d" % (rank if nccl else 0)
    th.cuda.set_device(dev)
    if nccl:
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=th.device(dev))
    else:
        dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        s = iql_system(3, 8, 12, True, seed=5, device=dev, data_parallel=True, learner_log_interval=0, dp_fused=fused)
        B = s.batch.batch_size
        lo, hi = rank * B // world, (rank + 1) * B // world
        for i in range(3):
            s.learner.train(s.batch[lo:hi], t_env=i, episode_num=i)
        th.cuda.synchronize()
        out.put((rank, np_params(s.mac.agent), {k: v[0] for k, v in s.logger.stats.items()}, s.mac.agent.trained_steps,
                 bool(getattr(s.learner, "_dp_sym", None)), getattr(s.learner, "_dp_sym_error", "")))
        dist.barrier()
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("nccl,fused", [(False, False), (True, False), (True, True)])
def test_dp_two_ranks_equal_full_batch(nccl, fused):
    """Ranks all-reduce un-normalised gradients and raw sums; the global normaliser is the expanded mask sum
    N * mask.sum() of the whole batch, so two half batches land on one full-batch step."""
    if nccl and th.cuda.device_count() < 2:
        pytest.skip("needs two GPUs (gradient all-reduce over NCCL / NVLink)")
    ctx = mp.get_context("spawn")
    out = ctx.SimpleQueue()
    port = _free_port()
    procs = [ctx.Process(target=_dp_worker, args=(r, 2, port, out, nccl, fused)) for r in range(2)]
    for p in procs:
        p.start()
    res = sorted([out.get(), out.get()], key=lambda r: r[0])
    for p in procs:
        p.join(300)
        assert p.exitcode == 0
    s = iql_system(3, 8, 12, True, seed=5, device="cuda:0", learner_log_interval=0)
    for i in range(3):
        s.learner.train(s.batch, t_env=i, episode_num=i)
    ref = np_params(s.mac.agent)
    for _, pa, stats, steps, was_fused, err in res:
        assert was_fused == fused, err
        for k in ref:
            assert_close(pa[k], ref[k], TOL, "dp agent " + k)
        for k, v in s.logger.stats.items():
            assert abs(stats[k] - v[0]) <= TOL * max(1.0, abs(v[0])), (k, stats[k], v[0])
        assert steps == s.mac.agent.trained_steps
    for k in ref:
        assert np.array_equal(res[0][1][k], res[1][1][k]), k


# ---------------------------------------------------------------------------------------------- targets, checkpoints
def test_update_targets_and_checkpoint_roundtrip(tmp_path):
    s = iql_system(3, 4, 8, True, seed=2)
    L = s.learner
    L.args.target_update_interval = 1
    before = np_params(L.target_mac.agent)
    L.train(s.batch, t_env=0, episode_num=1)
    assert any("Updated" in m for m in s.logger.infos)
    after, online = np_params(L.target_mac.agent), np_params(s.mac.agent)
    for k in after:
        assert np.array_equal(after[k], online[k]) and not np.array_equal(after[k], before[k])
    L.save_models(str(tmp_path))
    assert sorted(f.name for f in tmp_path.iterdir()) == ["home_qlearner_agent.th", "home_qlearner_opt.th"]
    s2 = iql_system(3, 4, 8, True, seed=3)
    s2.learner.load_models(str(tmp_path))
    for k, v in online.items():
        assert np.array_equal(v, np_params(s2.mac.agent)[k])
        assert np.array_equal(v, np_params(s2.learner.target_mac.agent)[k])
    assert th.equal(L.optimiser.flat_sq, s2.learner.optimiser.flat_sq)
    L.train(s.batch, 1, 1)
    s2.learner.train(s.batch, 1, 1)
    for k, v in np_params(s.mac.agent).items():
        assert np.array_equal(v, np_params(s2.mac.agent)[k])
