"""Cost of training through the modules with torch autograd (`args.autograd_forward`): ms per training step, one JSON line
per (workload, case), in the spirit of bench.py.

    python tools/autograd_bench.py [--workload qmix_5v5_b32 ...] [--steps 5] [--warmup 2] [--rounds 3] [--out FILE]

Cases, on the same seeded batch (T = 200), timed alternately for `--rounds` rounds in one process:
  modules     the reference's q_learner.py:36-105 op sequence (tests/autograd_ref.py) over BasicMAC + QMixer with the
              switch on, then clip_grad_norm_ and a stock RMSprop step;
  torch_port  oracle/torch_port's eager op sequence (TorchPortLearner.train) on the same GPU;
  fused       QLearner.train (CUDA graphs on), for context.
Each case runs K steps between a device synchronise before and after; the GPU name and power limit go into every line."""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import torch as th

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

WORKLOADS = {"qmix_5v5_b32": (5, 32), "qmix_10v10_b128": (10, 128)}


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power = [x.strip() for x in out.split(",")]
        return name, power
    except Exception:                                   # noqa: BLE001 -- the numbers are still printed, unlabelled
        return th.cuda.get_device_name(), "unknown"


def build(N, B):
    from oracle import torch_port as TP
    from tests.autograd_ref import reference_loss
    from tests.gpu_helpers import np_batch, np_params, seeded_system

    s = seeded_system(N, B, 201, "qmix", autograd_forward=True)
    L, eb, a = s.learner, s.batch, s.args
    params = list(L.mac.parameters()) + list(L.mixer.parameters())
    opt = th.optim.RMSprop(params, lr=a.lr, alpha=a.optim_alpha, eps=a.optim_eps)

    def modules_step():
        L.mac.init_hidden(B)
        L.target_mac.init_hidden(B)
        loss, _ = reference_loss({k: eb[k] for k in ("reward", "actions", "terminated", "filled", "avail_actions", "state", "obs")},
                                 lambda t: L.mac.forward(eb, t), lambda t: L.target_mac.forward(eb, t),
                                 L.mixer, L.target_mixer, double_q=a.double_q, gamma=a.gamma)
        opt.zero_grad()
        loss.backward()
        th.nn.utils.clip_grad_norm_(params, a.grad_norm_clip)
        opt.step()

    nb = {k: th.from_numpy(v).cuda() for k, v in np_batch(eb).items()}
    port = TP.TorchPortLearner(np_params(L.mac.agent), np_params(L.target_mac.agent), np_params(L.mixer),
                               np_params(L.target_mixer), mixer="qmix", double_q=a.double_q, gamma=a.gamma, lr=a.lr,
                               alpha=a.optim_alpha, eps=a.optim_eps, clip=a.grad_norm_clip, device="cuda")

    def port_step():
        port.train(nb)

    fused = seeded_system(N, B, 201, "qmix")

    def fused_step():
        fused.learner.train(fused.batch, 0, 0)

    return {"modules": modules_step, "torch_port": port_step, "fused": fused_step}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workload", nargs="*", default=list(WORKLOADS))
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not th.cuda.is_available():
        raise SystemExit("autograd_bench.py measures on the GPU; no CUDA device found")
    name, power = gpu_info()
    for w in args.workload:
        N, B = WORKLOADS[w]
        cases = build(N, B)
        for f in cases.values():
            for _ in range(args.warmup):
                f()
        times = {k: [] for k in cases}
        for _ in range(args.rounds):
            for k, f in cases.items():
                th.cuda.synchronize()
                t0 = time.perf_counter()
                for _ in range(args.steps):
                    f()
                th.cuda.synchronize()
                times[k].append(1e3 * (time.perf_counter() - t0) / args.steps)
        for k, v in times.items():
            line = json.dumps(dict(workload=w, case=k, ms_per_step=statistics.median(v), rounds=v, steps=args.steps,
                                   gpu=name, power_limit=power))
            print(line)
            if args.out:
                with open(args.out, "a") as fh:
                    fh.write(line + "\n")


if __name__ == "__main__":
    main()
