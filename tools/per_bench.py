"""Prioritized episode replay: ms per `train_from_buffer` step with a uniform and a prioritized buffer, and the sampler and
priority-update kernels alone.

    python tools/per_bench.py [--reps 5] [--steps 20] [--out FILE] [--workloads qmix_5v5_b32,...]

Learner cases (buffer of 5000 episodes, T = 200, graphs on, masked form): for each workload the uniform ReplayBuffer and
the PrioritizedReplayBuffer are timed alternately in one process, `--steps` steps per run between CUDA events, median over
`--reps` runs.  Kernel cases: mal_per_sample (B = 32 and 1024) and mal_per_update (B = 32, T = 200) at buffers of 5000,
50000 and 10^6 slots, 200 launches between CUDA events.  One JSON line per case with the GPU name and power limit.
"""
import argparse
import ctypes as C
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
SIZE = 5000


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


def learner_cases(wl, reps, steps, emit):
    c = CONFIGS[wl]
    d = dims(c["N"])
    N, A, OBS, S, B = d["N"], d["A"], d["OBS"], d["S"], c["B"]
    th.manual_seed(0)
    s = build_system(N, A, OBS, S, B, TT, c["mixer"], True, buffer_size=SIZE)
    uni = s.buf
    per = M.PrioritizedReplayBuffer(s.scheme, s.groups, SIZE, TT, preprocess=s.pre, device=DEV)
    gen = th.Generator().manual_seed(1)
    chunk = 250
    for _ in range(SIZE // chunk):
        data, lens = synth_episode_data(chunk, TT, N, A, OBS, S, gen, var_len=True, device=DEV)
        data["terminated"].zero_()
        data["terminated"][th.arange(chunk), lens - 1] = 1
        eb = fill_episode_batch(M.EpisodeBatch(s.scheme, s.groups, chunk, TT, preprocess=s.pre, device=DEV), data, lens)
        uni.insert_episode_batch(eb)
        per.insert_episode_batch(eb)
    L = s.learner
    t = [0]

    def step(buf):
        def f():
            t[0] += 1
            L.train_from_buffer(buf, B, t_env=t[0], episode_num=0)
        return f
    runs = {"uniform": [], "per": []}
    for name, buf in (("uniform", uni), ("per", per)):
        for _ in range(3):
            step(buf)()
    th.cuda.synchronize()
    for _ in range(reps):
        for name, buf in (("uniform", uni), ("per", per)):
            runs[name].append(events_ms(step(buf), steps))
    for name, v in runs.items():
        emit(dict(case="train_from_buffer", workload=wl, buffer=name, buffer_size=SIZE, T=TT - 1,
                  ms_per_step=round(statistics.median(v), 4), runs=[round(x, 4) for x in v]))
    del s, uni, per
    th.cuda.empty_cache()


def kernel_cases(emit):
    lib = nat.lib()
    st = nat.current_stream()
    gen = th.Generator().manual_seed(2)
    for n in (5000, 50000, 10 ** 6):
        p = (th.rand(n, generator=gen) + 0.01).to(DEV)
        for B in (32, 1024):
            ids = th.empty(B, dtype=th.long, device=DEV)
            w = th.empty(B, dtype=th.float32, device=DEV)
            u = th.rand(B, device=DEV)

            def samp():
                nat.check(lib.mal_per_sample(nat.ptr(p), n, B, 0.4, nat.ptr(u), 0, 0, nat.ptr(ids), nat.ptr(w), None, st))
            samp()
            emit(dict(case="mal_per_sample", buffer_size=n, B=B, us_per_launch=round(events_ms(samp, 200) * 1e3, 2)))
        B, T = 32, 200
        ids = th.randint(0, n, (B,), device=DEV)
        td = th.randn(B * T, device=DEV)
        mask = th.ones(B * T, device=DEV)
        mx = th.ones(1, device=DEV)

        def upd():
            nat.check(lib.mal_per_update(nat.ptr(td), nat.ptr(mask), B, T, 1, nat.ptr(ids), 0.6, 1e-6, nat.ptr(p), n,
                                         nat.ptr(mx), st))
        upd()
        emit(dict(case="mal_per_update", buffer_size=n, B=B, T=T, us_per_launch=round(events_ms(upd, 200) * 1e3, 2)))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--workloads", default="qmix_5v5_b32,qmix_10v10_b128,qmix_20v20_b1024")
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
    kernel_cases(emit)
    for wl in a.workloads.split(","):
        steps = a.steps if not wl.endswith("b1024") else max(3, a.steps // 4)
        learner_cases(wl, a.reps, steps, emit)


if __name__ == "__main__":
    main()
