"""ms per rollout timestep of a two-team league rollout in which the away team plays K different opponents.

    python tools/pool_rollout_bench.py [--reps 5] [--limit 60] [--out FILE]

Workloads 5v5 bs=32 and 10v10 bs=128 (SyntheticVecEnv, every match lasts `limit` steps), K in {1, 4, 8, 32}; the home
team plays its own agent, match b's away team plays opponent b % K of a [K, P] table.  Three cases, timed alternately in
one process (median over --reps runs of the whole episode, ms per timestep = run time / (limit + 1)):
    pooled  one stepper run, away controller with set_match_policies(table, ids): one launch per team and timestep
    split   today's workaround: K stepper runs of bs/K matches, the away agent loaded with one opponent per run
    single  one stepper run, both teams on their own agent (the floor)
One JSON line per (workload, K, case) with the GPU name and power limit.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import torch as th  # noqa: E402

import ma_league_b200 as M  # noqa: E402
from ma_league_b200.league import DeviceAgentPool  # noqa: E402
from ma_league_b200.steppers import BatchedEpisodeStepper, SyntheticVecEnv  # noqa: E402
from ma_league_b200.synthetic import make_args, make_scheme  # noqa: E402

DEV = "cuda"


def gpu_info():
    name = th.cuda.get_device_name(0)
    try:
        pl = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader,nounits", "-i", "0"],
                            capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception:
        pl = "unknown"
    return name, pl


def stepper(args, scheme, groups, pre, n, N, A, OBS, S, limit, home, away):
    env = SyntheticVecEnv(n, N, A, OBS, S, limit, n_teams=2, seed=1, device=DEV, min_len=limit)
    st = BatchedEpisodeStepper(args, None, env, sync_every=8)
    st.initialize(scheme, groups, pre, home, away)
    return st


def timed(fn):
    th.cuda.synchronize()
    t0 = time.perf_counter()
    fn()
    th.cuda.synchronize()
    return time.perf_counter() - t0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--limit", type=int, default=60)
    ap.add_argument("--out", default=None)
    o = ap.parse_args()
    if not th.cuda.is_available():
        raise SystemExit("pool_rollout_bench needs a CUDA device")
    gpu, power = gpu_info()
    lines = []
    for N, bs in [(5, 32), (10, 128)]:
        A, OBS, S = 6 + N, 8 + 8 * N, 16 * N
        th.manual_seed(0)
        args = make_args(N, A, S, mixer="qmix", device=DEV, batch_size_run=bs)
        scheme, groups, pre = make_scheme(N, A, OBS, S)
        sch = M.ReplayBuffer(scheme, groups, 2, o.limit + 1, preprocess=pre, device=DEV).scheme
        home, away = M.BasicMAC(sch, groups, args), M.BasicMAC(sch, groups, args)
        for m in (home, away):
            m.action_selector.validate = False
        for K in [1, 4, 8, 32]:
            opponents = [M.BasicMAC(sch, groups, args) for _ in range(K)]
            table = th.stack([m.agent.flat_params().detach().clone() for m in opponents])
            pool = DeviceAgentPool(away)
            pool.pool = table                      # the league table the split runs load from (load_into)
            ids = th.arange(bs) % K
            big = stepper(args, scheme, groups, pre, bs, N, A, OBS, S, o.limit, home, away)
            small = stepper(args, scheme, groups, pre, bs // K, N, A, OBS, S, o.limit, home, away)

            def pooled():
                away.set_match_policies(table, ids)
                big.run(test_mode=True)
                away.set_match_policies(None)

            def split():
                for k in range(K):
                    pool.load_into(away, k)
                    small.run(test_mode=True)

            def single():
                big.run(test_mode=True)
            cases = {"pooled": pooled, "split": split, "single": single}
            for fn in cases.values():
                fn()                               # warm-up: module loads, allocator
            times = {c: [] for c in cases}
            for _ in range(o.reps):
                for c, fn in cases.items():
                    times[c].append(timed(fn))
            for c in cases:
                ms = 1e3 * statistics.median(times[c]) / (o.limit + 1)
                rec = dict(tool="pool_rollout_bench", workload="%dv%d_b%d" % (N, N, bs), K=K, case=c,
                           ms_per_timestep=round(ms, 4), runs=o.reps, limit=o.limit, gpu=gpu, power_limit_w=power)
                lines.append(json.dumps(rec))
                print(lines[-1], flush=True)
    if o.out:
        with open(o.out, "a") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
