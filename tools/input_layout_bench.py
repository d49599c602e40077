"""Cost of the agent-input switches (obs_last_action / obs_agent_id): ms per learner step and per fused rollout timestep
for the four layouts of each workload, one JSON line per (workload, layout), in the spirit of bench.py.

    python tools/input_layout_bench.py [--workload qmix_5v5_b32 ...] [--steps 60] [--warmup 10] [--rollout-limit 200]

Learner: QLearner.train() on rotating pre-built batches (CUDA graphs on, as in bench.py), K steps between one pair of
CUDA events; the four batches are not flushed from L2 between steps.  Rollout: one
BatchedEpisodeStepper.run() of B matches (the workload's B, full-length episodes) through the one-launch rollout step,
wall time around the synchronised run divided by the stored timesteps.  The GPU name and power limit are printed with
every line."""
import argparse
import json
import os
import subprocess
import sys
import time

import torch as th

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

LAYOUTS = [(True, True), (False, True), (True, False), (False, False)]   # (obs_last_action, obs_agent_id)


class NullLog:
    def log_stat(self, *x): pass
    def info(self, *x): pass


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power = [x.strip() for x in out.split(",")]
        return name, power
    except Exception:                                   # noqa: BLE001 -- the numbers are still printed, unlabelled
        return th.cuda.get_device_name(), "unknown"


def learner_ms(M, N, A, OBS, S, B, TT, mixer, last, aid, steps, warmup, device):
    from ma_league_b200.synthetic import make_args, make_scheme, synth_episode_data, fill_episode_batch
    th.manual_seed(1000)
    args = make_args(N, A, S, mixer=mixer, double_q=True, device=device, batch_size=B, obs_last_action=last,
                     obs_agent_id=aid)
    scheme, groups, pre = make_scheme(N, A, OBS, S)
    buf = M.ReplayBuffer(scheme, groups, B, TT, preprocess=pre, device=device)
    mac = M.mac_REGISTRY["basic"](buf.scheme, groups, args)
    learner = M.learner_REGISTRY["q"](mac, buf.scheme, NullLog(), args, name="home")
    learner.build_optimizer()
    gen = th.Generator().manual_seed(7)
    batches = []
    for _ in range(4):
        data, lens = synth_episode_data(B, TT, N, A, OBS, S, gen, var_len=True, device=device)
        lens[0] = TT - 1
        batches.append(fill_episode_batch(M.EpisodeBatch(scheme, groups, B, TT, preprocess=pre, device=device), data, lens))
    for i in range(2 * len(batches) + warmup):         # eager, graph capture, then warm replays
        learner.train(batches[i % len(batches)], t_env=i, episode_num=0)
    th.cuda.synchronize()
    e0, e1 = th.cuda.Event(enable_timing=True), th.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(steps):
        learner.train(batches[i % len(batches)], t_env=i, episode_num=0)
    e1.record()
    th.cuda.synchronize()
    return e0.elapsed_time(e1) / steps, mac.agent.fc1.weight.shape[1]


def rollout_ms(M, N, A, OBS, S, B, mixer, last, aid, limit, device):
    from ma_league_b200.steppers import BatchedEpisodeStepper, SyntheticVecEnv
    from ma_league_b200.synthetic import make_args, make_scheme
    th.manual_seed(1000)
    args = make_args(N, A, S, mixer=mixer, device=device, batch_size_run=B, obs_last_action=last, obs_agent_id=aid)
    scheme, groups, pre = make_scheme(N, A, OBS, S)
    buf = M.ReplayBuffer(scheme, groups, B, limit + 1, preprocess=pre, device=device)
    mac = M.mac_REGISTRY["basic"](buf.scheme, groups, args)
    mac.action_selector.validate = False
    assert mac._rollout_fusable()
    env = SyntheticVecEnv(B, N, A, OBS, S, limit, n_teams=1, seed=3, device=device, min_len=limit)
    st = BatchedEpisodeStepper(args, None, env, sync_every=limit + 1)
    st.initialize(scheme, groups, pre, mac, None)
    st.run(test_mode=True)                             # warm-up episode
    th.cuda.synchronize()
    times = []
    for _ in range(3):
        t0 = time.perf_counter()
        st.run(test_mode=True)
        th.cuda.synchronize()
        times.append((time.perf_counter() - t0) * 1e3 / (limit + 1))
    return min(times)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workload", action="append", default=None)
    ap.add_argument("--steps", type=int, default=60)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--rollout-limit", dest="rollout_limit", type=int, default=200)
    a = ap.parse_args()
    workloads = a.workload or ["qmix_5v5_b32", "vdn_5v5_b32", "qmix_10v10_b128"]
    assert th.cuda.is_available(), "input_layout_bench measures on the GPU"
    import ma_league_b200 as M
    from ma_league_b200 import _native as nat
    from ma_league_b200.synthetic import CONFIGS, dims
    nat.build()
    device = "cuda"
    name, power = gpu_info()
    for w in workloads:
        c = CONFIGS[w]
        d = dims(c["N"])
        N, A, OBS, S, B = d["N"], d["A"], d["OBS"], d["S"], c["B"]
        for last, aid in LAYOUTS:
            ms, d_in = learner_ms(M, N, A, OBS, S, B, 201, c["mixer"], last, aid, a.steps, a.warmup, device)
            r_ms = rollout_ms(M, N, A, OBS, S, B, c["mixer"], last, aid, a.rollout_limit, device)
            print(json.dumps(dict(workload=w, obs_last_action=last, obs_agent_id=aid, d_in=d_in,
                                  learner_ms_per_step=round(ms, 4), rollout_ms_per_timestep=round(r_ms, 4),
                                  steps=a.steps, rollout_timesteps=a.rollout_limit + 1, gpu=name, power_limit=power)),
                  flush=True)


if __name__ == "__main__":
    main()
