"""TD(lambda) targets: ms per `QLearner.train` step (graph replay) with 1-step targets and with `td_lambda = 0.6`.

    python tools/td_lambda_bench.py [--reps 7] [--steps 20] [--out FILE] [--workloads qmix_5v5_b32,...]

For each workload (T = 200, variable episode lengths) the two settings are timed alternately in one process on the same
learner and batch, `--steps` steps per run between CUDA events, median over `--reps` runs; each setting replays its own
captured graph.  Then one eager step of each setting under `mal_profile_begin` / `mal_profile_end` gives the time of
the mixing / target kernels.  One JSON line per case with the GPU name and power limit.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import torch as th  # noqa: E402

import ma_league_b200 as M  # noqa: E402
from ma_league_b200 import _native as nat  # noqa: E402
from ma_league_b200.synthetic import CONFIGS, dims, synth_episode_data, fill_episode_batch  # noqa: E402
from tests.gpu_helpers import build_system  # noqa: E402

DEV = "cuda"
TT = 201
SETTINGS = (("one_step", None), ("td_lambda_0.6", 0.6))
KERNELS = ("k_mix_td", "k_mix_tq", "k_td_lambda", "k_mix_td_lambda")


def gpu_info():
    name = th.cuda.get_device_name(0)
    try:
        pl = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader,nounits", "-i", "0"],
                            capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception:
        pl = "unknown"
    return name, pl


def events_ms(fn, n):
    e0, e1 = th.cuda.Event(enable_timing=True), th.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        fn()
    e1.record()
    th.cuda.synchronize()
    return e0.elapsed_time(e1) / n


def cases(wl, reps, steps, emit):
    c = CONFIGS[wl]
    d = dims(c["N"])
    N, A, OBS, S, B = d["N"], d["A"], d["OBS"], d["S"], c["B"]
    th.manual_seed(0)
    s = build_system(N, A, OBS, S, B, TT, c["mixer"], True)
    data, lens = synth_episode_data(B, TT, N, A, OBS, S, th.Generator().manual_seed(1), var_len=True, device=DEV)
    batch = fill_episode_batch(M.EpisodeBatch(s.scheme, s.groups, B, TT, preprocess=s.pre, device=DEV), data, lens)
    L = s.learner
    t = [0]

    def step(lam):
        def f():
            s.args.td_lambda = lam
            t[0] += 1
            L.train(batch, t_env=t[0], episode_num=0)
        return f
    for _, lam in SETTINGS:
        for _ in range(3):                                     # eager, capture, replay
            step(lam)()
    th.cuda.synchronize()
    runs = {name: [] for name, _ in SETTINGS}
    for _ in range(reps):
        for name, lam in SETTINGS:
            runs[name].append(events_ms(step(lam), steps))
    base = statistics.median(runs["one_step"])
    for name, v in runs.items():
        med = statistics.median(v)
        emit(dict(case="train", workload=wl, returns=name, T=TT - 1, ms_per_step=round(med, 4),
                  vs_one_step=round(med / base - 1.0, 4), runs=[round(x, 4) for x in v]))
    L.use_graphs = False
    for name, lam in SETTINGS:
        step(lam)()
        th.cuda.synchronize()
        nat.profile_begin()
        step(lam)()
        th.cuda.synchronize()
        prof = nat.profile_end()
        ks = {k: round(ms * 1e3, 2) for k, (n, ms) in prof.items() if k.startswith(KERNELS)}
        emit(dict(case="kernels_eager", workload=wl, returns=name, us=ks,
                  step_kernels_us=round(sum(ms for _, ms in prof.values()) * 1e3, 1)))
    del s, L, batch
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
