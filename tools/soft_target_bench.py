"""Soft target updates in the fused learner step: ms per `QLearner.train` step (graph replay) in hard mode on steps
where no copy fires, against `args.target_update_interval_or_tau = 0.01` (the blend inside the optimiser kernel), and
the per-kernel time of `k_clip_rmsprop` against `k_clip_rmsprop_soft`.

    python tools/soft_target_bench.py [--reps 7] [--steps 20] [--out FILE] [--workloads qmix_5v5_b32,...]

For each workload (T = 200, variable episode lengths, RMSprop) two learners with identical parameters train on the same
batch, one in each mode; they are timed alternately in one process, `--steps` steps per run between CUDA events, median
over `--reps` runs, each replaying its own captured graph.  Then `--steps` eager steps of each learner under
`mal_profile_begin` / `mal_profile_end` give the mean time of the optimiser kernel.  One JSON line per case with the GPU
name and power limit.
"""
import argparse
import json
import os
import statistics
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import torch as th  # noqa: E402

import ma_league_b200 as M  # noqa: E402
from ma_league_b200 import _native as nat  # noqa: E402
from ma_league_b200.synthetic import CONFIGS, dims, synth_episode_data, fill_episode_batch  # noqa: E402
from tests.gpu_helpers import build_system  # noqa: E402
from tools.td_lambda_bench import events_ms, gpu_info  # noqa: E402

DEV = "cuda"
TT = 201
MODES = (("hard", None, "k_clip_rmsprop"), ("soft", 0.01, "k_clip_rmsprop_soft"))   # hard: episode 0 never copies


def cases(wl, reps, steps, emit):
    c = CONFIGS[wl]
    d = dims(c["N"])
    N, A, OBS, S, B = d["N"], d["A"], d["OBS"], d["S"], c["B"]
    learners, batch = {}, None
    for opt, tau, _ in MODES:
        th.manual_seed(0)                                      # identical parameters for both learners
        s = build_system(N, A, OBS, S, B, TT, c["mixer"], True, target_update_interval_or_tau=tau)
        if batch is None:
            data, lens = synth_episode_data(B, TT, N, A, OBS, S, th.Generator().manual_seed(1), var_len=True, device=DEV)
            batch = fill_episode_batch(M.EpisodeBatch(s.scheme, s.groups, B, TT, preprocess=s.pre, device=DEV), data, lens)
        learners[opt] = s.learner
    t = [0]

    def step(opt):
        def f():
            t[0] += 1
            learners[opt].train(batch, t_env=t[0], episode_num=0)
        return f
    for opt, _, _ in MODES:
        for _ in range(3):                                     # eager, capture, replay
            step(opt)()
    th.cuda.synchronize()
    n_params = learners["soft"]._grad.numel()
    runs = {opt: [] for opt, _, _ in MODES}
    for _ in range(reps):
        for opt, _, _ in MODES:
            runs[opt].append(events_ms(step(opt), steps))
    base = statistics.median(runs["hard"])
    for opt, v in runs.items():
        med = statistics.median(v)
        emit(dict(case="train", workload=wl, mode=opt, T=TT - 1, params=n_params, ms_per_step=round(med, 4),
                  vs_hard=round(med / base - 1.0, 4), runs=[round(x, 4) for x in v]))
    for opt, _, kernel in MODES:
        learners[opt].use_graphs = False
        step(opt)()
        th.cuda.synchronize()
        nat.profile_begin()
        for _ in range(steps):
            step(opt)()
        th.cuda.synchronize()
        prof = nat.profile_end()
        n, ms = prof[kernel]
        emit(dict(case="kernel_eager", workload=wl, mode=opt, kernel=kernel, params=n_params, launches=n,
                  us_per_launch=round(ms * 1e3 / n, 2),
                  step_kernels_us=round(sum(v for _, v in prof.values()) * 1e3 / steps, 1)))
    del learners, batch
    th.cuda.empty_cache()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--workloads", default="qmix_5v5_b32,vdn_5v5_b32,qmix_10v10_b128,qmix_20v20_b1024")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    name, pl = gpu_info()

    def emit(d):
        d = dict(d, gpu=name, power_limit_w=pl)
        line = json.dumps(d)
        print(line, flush=True)
        if a.out:
            with open(a.out, "a") as f:
                f.write(line + "\n")
    for wl in a.workloads.split(","):
        steps = a.steps if not wl.endswith("b1024") else max(3, a.steps // 4)
        cases(wl, a.reps, steps, emit)


if __name__ == "__main__":
    main()
