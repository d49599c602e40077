"""Cost of independent Q-learners (`mixer: None`) against VDN and QMIX: ms per learner step at the same shapes, one JSON
line per (workload, mixer), in the spirit of bench.py.

    python tools/iql_bench.py [--workload 5v5_b32 ...] [--steps 200] [--warmup 10] [--rounds 3]

QLearner.train() on four rotating pre-built batches shared by the three learners of a shape (CUDA graphs on, as in
bench.py), K steps between one pair of CUDA events; the batches are not flushed from L2 between steps.  The three
mixers are timed alternately (IQL, VDN, QMIX, IQL, ...) for `--rounds` rounds in one process, so that a drift of the
machine shows in every mixer alike; each line carries every round and their median.  The GPU name and power limit are
printed with every line."""
import argparse
import json
import os
import statistics
import subprocess
import sys

import torch as th

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

WORKLOADS = {"5v5_b32": (5, 32), "10v10_b128": (10, 128), "20v20_b1024": (20, 1024)}
MIXERS = [("iql", None), ("vdn", "vdn"), ("qmix", "qmix")]


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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workload", action="append", default=None, choices=sorted(WORKLOADS))
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--rounds", type=int, default=3)
    a = ap.parse_args()
    assert th.cuda.is_available(), "iql_bench measures on the GPU"
    import ma_league_b200 as M
    from ma_league_b200.synthetic import dims, make_args, make_scheme, synth_episode_data, fill_episode_batch
    device, TT = "cuda", 201
    name, power = gpu_info()
    for w in a.workload or ["5v5_b32", "10v10_b128", "20v20_b1024"]:
        N, B = WORKLOADS[w]
        d = dims(N)
        A, OBS, S = d["A"], d["OBS"], d["S"]
        scheme, groups, pre = make_scheme(N, A, OBS, S)
        gen = th.Generator().manual_seed(7)
        batches = []
        for _ in range(4):
            data, lens = synth_episode_data(B, TT, N, A, OBS, S, gen, var_len=True, device=device)
            lens[0] = TT - 1
            batches.append(fill_episode_batch(M.EpisodeBatch(scheme, groups, B, TT, preprocess=pre, device=device), data, lens))
        learners = {}
        buf = M.ReplayBuffer(scheme, groups, 1, TT, preprocess=pre, device=device)   # the processed scheme
        for tag, mixer in MIXERS:
            th.manual_seed(1000)
            args = make_args(N, A, S, mixer=mixer, double_q=True, device=device, batch_size=B)
            mac = M.mac_REGISTRY["basic"](buf.scheme, groups, args)
            learner = M.learner_REGISTRY["q"](mac, buf.scheme, NullLog(), args, name="home")
            learner.build_optimizer()
            for i in range(2 * len(batches) + a.warmup):   # eager, graph capture, then warm replays
                learner.train(batches[i % len(batches)], t_env=i, episode_num=0)
            learners[tag] = learner
        th.cuda.synchronize()
        runs = {tag: [] for tag, _ in MIXERS}
        e0, e1 = th.cuda.Event(enable_timing=True), th.cuda.Event(enable_timing=True)
        for _ in range(a.rounds):
            for tag, _ in MIXERS:
                learner = learners[tag]
                e0.record()
                for i in range(a.steps):
                    learner.train(batches[i % len(batches)], t_env=i, episode_num=0)
                e1.record()
                th.cuda.synchronize()
                runs[tag].append(round(e0.elapsed_time(e1) / a.steps, 4))
        for tag, _ in MIXERS:
            print(json.dumps(dict(workload=w, mixer=tag, N=N, B=B, T=TT - 1,
                                  learner_ms_per_step=round(statistics.median(runs[tag]), 4), rounds=runs[tag],
                                  steps=a.steps, gpu=name, power_limit=power)), flush=True)
        del learners, batches
        th.cuda.empty_cache()


if __name__ == "__main__":
    main()
