"""Adam in the fused learner step (`args.optimizer: "adam"`, mal_learner_step_adam / k_clip_adam) on the device, against
the fp64 reference of tests/adam_ref.py: three chained steps (so that the bias corrections change) for QMIX (2 and 1
layers), VDN and IQL, both agents and both double_q settings, with the 1-step target and with TD(lambda); a stock fp32
torch.optim.Adam fed the same clipped gradients; eager against graph replay and re-capture when weight_decay changes;
prioritized replay through train_from_buffer; a frozen agent; a checkpoint round trip; the launch count; the stand-alone
and peer-exchange entry points; and the two-rank data-parallel run against the full batch.

The reference step starts from the device's gradient: the TD(lambda) cases first check it against the fp64 oracle of
tests/td_lambda_ref.py, the 1-step cases rely on tests/test_gpu_learner.py and tests/test_gpu_iql.py for that.  Adam's
first steps are close to lr * sign(g), so an element whose gradient is near eps would turn the gradient's fp32 rounding
into a parameter difference of order lr: the optimiser is compared on the same gradient."""
import ctypes as C
import multiprocessing as mp
import os

import numpy as np
import pytest
import torch as th
import torch.distributed as dist

import ma_league_b200 as M
from ma_league_b200 import _native as nat
from ma_league_b200.learners.q_learner import DP_TAIL
from tests import adam_ref as R
from tests.gpu_helpers import np_params
from tests.helpers import assert_close, rel_err
from tests.test_data_parallel import _free_port
from tests.test_gpu_td_lambda import _fill, _flat_params, _nets, _per_buffer, _system, against_oracle

pytestmark = pytest.mark.gpu
DEV = "cuda"
TOL = 1e-5
LR = 1e-3


def _adam_system(N, B, TT, mixer, lam=None, layers=2, agent="rnn", double_q=True, seed=0, weight_decay=0.0, **kw):
    return _system(N, B, TT, mixer, lam, layers, agent, double_q, seed=seed, optimizer="adam", lr=LR,
                   weight_decay=weight_decay, **kw)


def _adam_state(s):
    """(exp_avg, exp_avg_sq, step, ticket) of the flat device state."""
    st = s.learner.optimiser.flat_state
    P = (st.numel() - 2) // 2
    h = st.cpu()
    return h[:P].numpy(), h[P:2 * P].numpy(), float(h[2 * P]), int(h[2 * P + 1:].view(th.int32)[0])


def _split(s, p):
    out, off = [], 0
    for n in _nets(s):
        d = {}
        for k, v in np_params(n).items():
            d[k] = p[off:off + v.size].reshape(v.shape)
            off += v.size
        out.append(d)
    return out[0], (out[1] if s.mixer else None)


def chained(s, lam, steps=3, n_frozen=0):
    """train() (graphs on: eager, capture, replay) `steps` times, chained through adam_ref from the same start."""
    L, a = s.learner, s.args
    wd = L.optimiser.param_groups[0]["weight_decay"]
    p = _flat_params(s)
    m, v, t = np.zeros_like(p), np.zeros_like(p), 0
    for i in range(steps):
        if lam is None:
            L.forward_backward(s.batch)
        else:
            against_oracle(s, lam, _split(s, p))               # the device gradient against the fp64 oracle at TOL
        g = L._grad.cpu().numpy().astype(np.float64)
        norm, _, p, m, v, t = R.clip_adam(p, g, m, v, t, a.lr, a.grad_norm_clip, n_frozen, weight_decay=wd)
        L.train(s.batch, t_env=i, episode_num=0)
        th.cuda.synchronize()
        logged = s.logger.stats["home_qlearner_grad_norm"][0]
        assert abs(logged - norm) <= TOL * norm, (i, logged, norm)
        assert_close(_flat_params(s), p, TOL, "parameters after step %d" % (i + 1))
        em, ev, step, ticket = _adam_state(s)
        assert_close(em, m, TOL, "exp_avg after step %d" % (i + 1))
        # exp_avg_sq is quadratic in the gradient: twice the gradient's relative error
        assert_close(ev, v, 2 * TOL, "exp_avg_sq after step %d" % (i + 1))
        assert step == t == L.optimiser._steps and ticket == 0
    return p, m, v


CASES = [  # N, B, TT, mixer, layers, agent, double_q, lambda, weight_decay
    (3, 32, 201, "qmix", 2, "rnn", True, None, 0.0),
    (5, 32, 201, "qmix", 2, "rnn", True, None, 1e-4),
    (10, 128, 201, "qmix", 2, "rnn", True, None, 0.0),
    (20, 16, 24, "qmix", 2, "rnn", True, None, 0.0),
    (5, 32, 201, "qmix", 1, "rnn", False, None, 0.0),
    (5, 32, 201, "vdn", 2, "rnn", True, None, 0.0),
    (5, 32, 201, None, 2, "rnn", True, None, 1e-4),
    (20, 16, 24, None, 2, "dqn", False, None, 0.0),
    (5, 32, 201, "qmix", 2, "dqn", True, None, 0.0),
    (5, 32, 201, "qmix", 2, "rnn", True, 0.6, 0.0),
    (10, 32, 201, "vdn", 2, "rnn", False, 0.6, 1e-4),
    (5, 32, 201, None, 2, "rnn", True, 0.6, 0.0),
]


@pytest.mark.parametrize("N,B,TT,mixer,layers,agent,double_q,lam,wd", CASES)
def test_adam_step_against_reference(N, B, TT, mixer, layers, agent, double_q, lam, wd):
    s = _adam_system(N, B, TT, mixer, lam, layers, agent, double_q, seed=300 + N + TT, weight_decay=wd)
    chained(s, lam)


def test_matches_stock_torch_adam_fp32():
    s = _adam_system(5, 32, 201, "qmix", seed=3, weight_decay=1e-4)
    L = s.learner
    params = L.parameters()
    copies = [p.detach().clone() for p in params]
    stock = th.optim.Adam(copies, lr=LR, weight_decay=1e-4)
    for i in range(3):
        L.train(s.batch, i, 0)
        for c, p in zip(copies, params):
            c.grad = p.grad.clone()                                # the clipped gradient the fused step used
        stock.step()
        th.cuda.synchronize()
        flat = lambda ts: th.cat([x.detach().reshape(-1) for x in ts]).cpu().numpy()
        assert_close(flat(params), flat(copies), 1e-6, "parameters after step %d" % (i + 1))
        em, ev, step, _ = _adam_state(s)
        assert_close(em, flat([stock.state[c]["exp_avg"] for c in copies]), 1e-6, "exp_avg")
        assert_close(ev, flat([stock.state[c]["exp_avg_sq"] for c in copies]), 1e-6, "exp_avg_sq")
        assert step == float(stock.state[copies[0]]["step"]) == i + 1
    sd = L.optimiser.state_dict()
    ref = stock.state_dict()
    assert sd["param_groups"] == ref["param_groups"]
    for k, st in ref["state"].items():
        assert float(sd["state"][k]["step"]) == float(st["step"]) and sd["state"][k]["step"].device == st["step"].device


def _state(s):
    return [v.clone() for n in _nets(s) for v in n.state_dict().values()] + \
        [s.learner.optimiser.flat_state.clone(), s.learner.scalars()[:nat.SC_STATUS].clone()]


@pytest.mark.parametrize("mixer", ["qmix", None])
def test_graph_replay_bit_identical_to_eager_and_recapture_on_weight_decay(mixer):
    outs = []
    for graphs in (False, True):
        s = _adam_system(5, 8, 61, mixer, seed=4)
        s.learner.use_graphs = graphs
        for i in range(4):                                     # eager, capture (which performs the step), replay, replay
            s.learner.train(s.batch, i, 0)
        th.cuda.synchronize()
        assert s.learner.n_graph_captures == (1 if graphs else 0)
        assert s.learner.n_graph_replays == (2 if graphs else 0)
        assert _adam_state(s)[2:] == (4.0, 0) and s.learner.optimiser._steps == 4
        outs.append(_state(s))
    for x, y in zip(*outs):
        assert th.equal(x, y)
    # weight_decay changes: its own key (eager, capture, replay), each step against the reference with the new value
    L, a = s.learner, s.args
    replays, captures = L.n_graph_replays, L.n_graph_captures
    L.optimiser.param_groups[0]["weight_decay"] = 1e-2
    for i in range(3):
        p = _flat_params(s)
        m, v, t, _ = _adam_state(s)
        g = L.forward_backward(s.batch).cpu().numpy().astype(np.float64)
        _, _, p1, m1, _, t1 = R.clip_adam(p, g, m.astype(np.float64), v.astype(np.float64), int(t), a.lr,
                                          a.grad_norm_clip, weight_decay=1e-2)
        _, _, p0, _, _, _ = R.clip_adam(p, g, m.astype(np.float64), v.astype(np.float64), int(t), a.lr,
                                        a.grad_norm_clip, weight_decay=0.0)
        L.train(s.batch, 9 + i, 0)
        th.cuda.synchronize()
        got = _flat_params(s)
        assert_close(got, p1, TOL, "parameters with weight_decay")
        assert np.linalg.norm(got - p1) < 0.1 * np.linalg.norm(p1 - p0)   # the new value is applied, not the old one
        assert_close(_adam_state(s)[0], m1, TOL, "exp_avg with weight_decay")
        assert _adam_state(s)[2] == t1
    assert L.n_graph_captures == captures + 1 and L.n_graph_replays == replays + 1


def test_launch_count_equals_rmsprop_step():
    counts = {}
    for opt in ("rmsprop", "adam"):
        s = _system(5, 8, 61, "qmix", None, seed=5, optimizer=opt)
        s.learner.use_graphs = False
        s.learner.train(s.batch, 0, 0)
        th.cuda.synchronize()
        n0 = nat.lib().mal_launch_count()
        s.learner.train(s.batch, 1, 0)
        th.cuda.synchronize()
        counts[opt] = nat.lib().mal_launch_count() - n0
    assert counts["adam"] == counts["rmsprop"], counts


def test_frozen_agent_state_stays_zero():
    s = _adam_system(5, 16, 61, "qmix", seed=9)
    s.mac.freeze_agent_weights()
    agent0 = np_params(s.mac.agent)
    n_agent = sum(v.size for v in agent0.values())
    chained(s, None, n_frozen=n_agent)
    em, ev, _, _ = _adam_state(s)
    assert not em[:n_agent].any() and not ev[:n_agent].any() and em[n_agent:].any()
    for k, v in np_params(s.mac.agent).items():
        assert np.array_equal(v, agent0[k]), k
    assert not s.learner._grad[:n_agent].any()


@pytest.mark.parametrize("per", [False, True])
def test_train_from_buffer_equals_manual_loop(per):
    """Uniform and prioritized replay (importance weights, TD(lambda) targets) through train_from_buffer, graphs on,
    against the same steps done by hand with eager launches: bit-identical parameters, Adam state and priorities."""
    def system():
        s = _system(5, 8, 31, "qmix", 0.6, seed=9, open_ended=False, optimizer="adam", lr=LR)
        buf = _per_buffer(s, 64, 31) if per else M.ReplayBuffer(s.scheme, s.groups, 64, 31, preprocess=s.pre, device=DEV)
        _fill(s, buf, 8, 8, 31, 16, 5, short=20)
        return s, buf
    (s1, b1), (s2, b2) = system(), system()
    th.manual_seed(77)
    np.random.seed(77)
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
    assert _adam_state(s1)[2] == 4.0
    if per:
        assert th.equal(b1.priorities, b2.priorities) and th.equal(b1.max_priority, b2.max_priority)


def test_checkpoint_round_trip_continues_identically(tmp_path):
    s1 = _adam_system(5, 8, 61, "qmix", seed=12, weight_decay=1e-4)
    for i in range(2):
        s1.learner.train(s1.batch, i, 0)
    s1.learner.save_models(str(tmp_path))
    s2 = _adam_system(5, 8, 61, "qmix", seed=13)
    s2.learner.load_models(str(tmp_path))
    L1, L2 = s1.learner, s2.learner
    assert L2.optimiser._steps == 2 and _adam_state(s2)[2] == 2.0
    assert L2.optimiser.param_groups[0]["weight_decay"] == 1e-4          # the checkpoint brings its own value
    assert th.equal(L1.optimiser.flat_state, L2.optimiser.flat_state)
    L2.target_mac.agent.load_state_dict(L1.target_mac.agent.state_dict())   # load_models does not restore targets
    L2.target_mixer.load_state_dict(L1.target_mixer.state_dict())
    for i in range(2, 5):
        L1.train(s1.batch, i, 0)
        L2.train(s1.batch, i, 0)
    th.cuda.synchronize()
    for x, y in zip(_state(s1), _state(s2)):
        assert th.equal(x, y)
    assert _adam_state(s2)[2] == 5.0


# ---------------------------------------------------------------------------------------------- stand-alone entry points
def _hyper(clip, wd=0.0):
    return nat.AdamHyper(LR, 0.9, 0.999, 1e-8, wd, clip)


@pytest.mark.parametrize("clip", [1e3, 0.5])
@pytest.mark.parametrize("n_frozen", [0, 30000])
def test_clip_adam_with_denominator(clip, n_frozen):
    n_agent, n_mixer = 40000, 61000                        # several hundred blocks share the step ticket
    P = n_agent + n_mixer
    rng = np.random.default_rng(7)
    p = rng.standard_normal(P).astype(np.float32)
    agent, mixer = th.from_numpy(p[:n_agent].copy()).to(DEV), th.from_numpy(p[n_agent:].copy()).to(DEV)
    state = th.zeros(nat.adam_state_floats(P), device=DEV)
    scalars = th.zeros(64, device=DEV)
    scratch = th.zeros((P + 255) // 256, device=DEV)
    denom = th.tensor([37.0], device=DEV)
    ref_p, m, v, t = p.astype(np.float64), np.zeros(P), np.zeros(P), 0
    h = _hyper(clip, 1e-4)
    for i in range(3):
        G = (rng.standard_normal(P) * 20).astype(np.float32)
        grad = th.from_numpy(G.copy()).to(DEV)
        nat.check(nat.lib().mal_clip_adam(nat.ptr(agent), n_agent, nat.ptr(mixer), n_mixer, nat.ptr(grad), nat.ptr(state),
                                          C.byref(h), nat.ptr(scalars), nat.ptr(scratch), nat.ptr(denom), n_frozen,
                                          nat.current_stream()), "mal_clip_adam")
        th.cuda.synchronize()
        norm, g_clip, ref_p, m, v, t = R.clip_adam(ref_p, G.astype(np.float64) / 37.0, m, v, t, LR, clip, n_frozen,
                                                   weight_decay=1e-4)
        assert (norm > clip) == (clip < 1.0)
        assert abs(float(scalars[nat.SC_GRAD_NORM]) - norm) <= TOL * norm
        assert_close(grad.cpu().numpy(), g_clip, TOL, "clipped gradient")
        got = np.concatenate([agent.cpu().numpy(), mixer.cpu().numpy()])
        assert_close(got, ref_p, 1e-6, "parameters")
        assert np.array_equal(got[:n_frozen], p[:n_frozen])
        hs = state.cpu()
        assert_close(hs[:P].numpy(), m, TOL, "exp_avg")
        assert_close(hs[P:2 * P].numpy(), v, 2 * TOL, "exp_avg_sq")
        assert float(hs[2 * P]) == t == i + 1 and int(hs[2 * P + 1:].view(th.int32)[0]) == 0
        assert not hs[:n_frozen].any()
    bad = nat.AdamHyper(LR, 1.0, 0.999, 1e-8, 0.0, clip)
    assert nat.lib().mal_clip_adam(nat.ptr(agent), n_agent, nat.ptr(mixer), n_mixer, nat.ptr(grad), nat.ptr(state),
                                   C.byref(bad), nat.ptr(scalars), nat.ptr(scratch), None, 0, nat.current_stream()) != 0


@pytest.mark.parametrize("world", [2, 4])
def test_peer_allreduce_clip_adam_one_device_fake_peers(world):
    """`mal_peer_allreduce_clip_adam` takes raw peer pointers, so W "ranks" can live on ONE device: every fake rank's
    buffer holds an un-normalised gradient and its raw statistic sums (element 4: its mask sum)."""
    n_agent, n_mixer = 3000, 5000
    P = n_agent + n_mixer
    rng = np.random.default_rng(world)
    bufs, acc, den = [], np.zeros(P), 0.0
    for r in range(world):
        g = (rng.standard_normal(P) * 5).astype(np.float32)
        tail = np.zeros(DP_TAIL, np.float32)
        tail[4] = 10.0 + r
        acc += g
        den += tail[4]
        bufs.append(th.from_numpy(np.concatenate([g, tail])).to(DEV))
    p = rng.standard_normal(P).astype(np.float32)
    agent, mixer = th.from_numpy(p[:n_agent].copy()).to(DEV), th.from_numpy(p[n_agent:].copy()).to(DEV)
    state = th.zeros(nat.adam_state_floats(P), device=DEV)
    grad, tail_out = th.full((P,), 7.0, device=DEV), th.zeros(DP_TAIL, device=DEV)
    scalars, scratch = th.zeros(64, device=DEV), th.zeros((P + 255) // 256, device=DEV)
    ptrs = (C.c_void_p * world)(*[b.data_ptr() for b in bufs])
    h = _hyper(1.0)
    ref_p, m, v, t = p.astype(np.float64), np.zeros(P), np.zeros(P), 0
    for i in range(2):
        nat.check(nat.lib().mal_peer_allreduce_clip_adam(ptrs, world, nat.ptr(agent), n_agent, nat.ptr(mixer), n_mixer,
                                                         nat.ptr(grad), nat.ptr(tail_out), DP_TAIL, nat.ptr(state),
                                                         C.byref(h), nat.ptr(scalars), nat.ptr(scratch), 0,
                                                         nat.current_stream()), "mal_peer_allreduce_clip_adam")
        th.cuda.synchronize()
        norm, g_clip, ref_p, m, v, t = R.clip_adam(ref_p, acc / den, m, v, t, LR, 1.0)
        assert abs(float(scalars[nat.SC_GRAD_NORM]) - norm) <= TOL * norm
        assert abs(float(tail_out[4]) - den) == 0
        assert_close(grad.cpu().numpy(), g_clip, TOL, "all-reduced clipped gradient")
        assert_close(np.concatenate([agent.cpu().numpy(), mixer.cpu().numpy()]), ref_p, 1e-6, "parameters")
        hs = state.cpu()
        assert_close(hs[:P].numpy(), m, TOL, "exp_avg")
        assert float(hs[2 * P]) == t == i + 1


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
        from tests.gpu_helpers import seeded_system
        s = seeded_system(3, 8, 12, "qmix", True, seed=5, device=dev, data_parallel=True, learner_log_interval=0,
                          dp_fused=fused, optimizer="adam", lr=LR)
        B = s.batch.batch_size
        lo, hi = rank * B // world, (rank + 1) * B // world
        for i in range(3):
            s.learner.train(s.batch[lo:hi], t_env=i, episode_num=i)
        th.cuda.synchronize()
        out.put((rank, np_params(s.mac.agent), np_params(s.learner.mixer), s.learner.optimiser.flat_state.cpu().numpy(),
                 s.learner._grad.cpu().numpy(), bool(getattr(s.learner, "_dp_sym", None)),
                 getattr(s.learner, "_dp_sym_error", "")))
        dist.barrier()
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("nccl,fused", [(False, False), (True, False), (True, True)])
def test_dp_adam_two_ranks_equals_full_batch(nccl, fused):
    """The exchanged, clipped gradient equals the full batch's at TOL and the replicas stay bit-identical.  The parameters
    are compared norm-wise: an element whose gradient is near eps gets an update close to lr * sign(g) from Adam, so the
    rounding difference between two halves and the full batch can move that one element by a fraction of lr."""
    from tests.gpu_helpers import seeded_system
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
    s = seeded_system(3, 8, 12, "qmix", True, seed=5, device="cuda:0", learner_log_interval=0, optimizer="adam", lr=LR)
    for i in range(3):
        s.learner.train(s.batch, t_env=i, episode_num=i)
    ref_a, ref_m = np_params(s.mac.agent), np_params(s.learner.mixer)
    ref_state = s.learner.optimiser.flat_state.cpu().numpy()
    ref_grad = s.learner._grad.cpu().numpy()
    P = (ref_state.size - 2) // 2
    for _, pa, pm, state, grad, was_fused, err in res:
        assert was_fused == fused, err
        assert_close(grad, ref_grad, TOL, "dp clipped gradient of the last step")
        for k in ref_a:
            assert rel_err(pa[k], ref_a[k]) <= TOL, "dp agent " + k
        for k in ref_m:
            assert rel_err(pm[k], ref_m[k]) <= TOL, "dp mixer " + k
        assert rel_err(state[:P], ref_state[:P]) <= TOL, "dp exp_avg"
        assert state[2 * P] == 3.0 and state[2 * P + 1:].view(np.int32)[0] == 0
    for i in (1, 2, 3):                                  # replicas: same reduced gradient, same update on every rank
        a, b = res[0][i], res[1][i]
        assert all(np.array_equal(a[k], b[k]) for k in a) if isinstance(a, dict) else np.array_equal(a, b)
