#!/usr/bin/env python
"""Benchmark of the hot path on BASELINE.json's metric: QMIX train transitions/sec (B=32, T=200) + act-select.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload NAME] [--dump-outputs DIR]

One JSON line on stdout (rank 0).  `--dump-outputs DIR` also writes what the last timed step returned to its caller
(statistics, gradient, updated parameters) as DIR/<name>.npy; the inputs are seeded, so two builds run with the same
arguments can be compared output for output.  A "step" is one QLearner.train() on one sampled batch of synthetic episodes
(SURVEY.md 8d).  `value` = transitions/s with the batch resident in HBM; `e2e` = the same through the public API
with the batch in pinned HOST memory (H2D copy of the step's inputs + D2H read of the loss inside the timed region).
Multi-GPU = league sharding: every rank owns an independent learner + replay buffer (weak scaling, no collective
on the data path); timing is max-over-ranks of CUDA-event time.  Under WORLD_SIZE > 1 the line also carries `dp`:
the strong-scaling data-parallel leg of BASELINE.json configs[4] (QMIX 20v20, global B=1024 split over the ranks,
gradients meeting in the fused peer-memory all-reduce / in NCCL).
`--impl reference` times the reference's CPU implementation (oracle/torch_port.py, the same ATen op sequence;
/root/reference itself is pure Python and does not exist on the GPU box) on the host cores, rank 0 only.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np   # noqa: E402
import torch as th   # noqa: E402

METRIC = "qmix_train_transitions_per_sec"
UNIT = "transitions/s"
T_STEPS = 200   # transitions per episode (201 stored steps)


def workload_dims(name):
    from ma_league_b200.synthetic import CONFIGS, dims
    c = CONFIGS[name]
    d = dims(c["N"])
    d.update(B=c["B"], mixer=c["mixer"], TT=T_STEPS + 1)
    return d


def workload_string(name):
    """The ONE description of a workload both arms print (the driver compares the strings)."""
    d = workload_dims(name)
    mixer = "QMIX (2-layer hypernet E=32 HE=64)" if d["mixer"] == "qmix" else "VDN"
    return "%s: %s, double-Q, B=%d, T=%d, N=%d, A=%d, OBS=%d, S=%d, H=64" % (
        name, mixer, d["B"], d["TT"] - 1, d["N"], d["A"], d["OBS"], d["S"])


# ------------------------------------------------------------------------------------------------ clocks
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.p = None
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(index), "--query-gpu=" + self.Q,
                                       "--format=csv,noheader,nounits", "-lms", "50"], stdout=subprocess.PIPE,
                                      stderr=subprocess.DEVNULL, text=True)
            time.sleep(0.3)      # let the first samples start before the timed region
        except Exception:
            self.p = None

    def stop(self):
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.p.terminate()
        try:
            out = self.p.communicate(timeout=5)[0]
        except Exception:
            self.p.kill()
            out = ""
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in out.splitlines():
            f = [x.strip() for x in line.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for n, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


# ------------------------------------------------------------------------------------------------ algorithmic bytes
def kernel_bytes(d, mixer, B=None):
    """Algorithmic bytes per launch of each learner kernel (DESIGN.md section 4); M1 = TT*B*N rows, BT = B*T.
    `B` = the batch THIS launch processes (a data-parallel rank's shard, not the global batch)."""
    B = d["B"] if B is None else B
    TT, N, A, OBS, S = d["TT"], d["N"], d["A"], d["OBS"], d["S"]
    T, R = TT - 1, B * N
    M1, BT = TT * R, B * T
    E, HE = 32, 64
    ld1, ld2 = 2 * HE + 2 * E, E * N + E
    f = 4
    P = 64 * (OBS + A + N) + 64 + 2 * 192 * 64 + 2 * 192 + 64 * A + A
    out = {
        "k_linear_group:fc1": M1 * (OBS + A) * f + 2 * M1 * 64 * f,
        "k_agent_in_tc": 2 * M1 * (OBS + A + 64 + 192) * f,
        "k_linear_group:w_ih": 2 * M1 * (64 + 192) * f,
        "k_gru_fwd": M1 * (2 * 192 + 2 * 64 + 256) * f,
        "k_q_head": M1 * (2 * 64 * f + A * 4 + 8) + 3 * BT * N * f,
        "k_gru_bwd": M1 * (256 + 64 + 64 + 256) * f,
        "k_linear_group:dx": M1 * (192 + 64 + 64) * f,
        "k_reduce_group:agent_dense": M1 * (256 + 64 + 64) * f,
        "k_reduce_gru": M1 * (256 + 64 + 64) * f,
        "k_reduce_group:agent_fc1": M1 * (64 + (OBS + A)) * f,
        "k_fc2_grad": T * R * (64 * f + 12),
    }
    if mixer == "qmix":
        P += (S * HE + HE + HE * E * N + E * N) + (S * HE + HE + HE * E + E) + (S * E + E) + (S * E + E + E + 1)
        out.update({
            "k_linear_group:mixer_l1": 2 * BT * (S + ld1) * f,
            "k_linear_group:mixer_l2": 2 * BT * (2 * HE + ld2) * f,
            "k_mix_td": BT * (2 * (ld1 - 2 * HE + ld2) + ld2 + 2 * E + 3 * N + 12) * f + BT * N * 64 * f,
            "k_linear_group:mixer_bwd_dh": BT * (ld2 + 2 * HE + 2 * HE) * f,
            "k_reduce_group:mixer_dense": BT * (ld2 + 2 * HE) * f,
            "k_reduce_group:mixer_state": BT * (ld1 + S) * f,
        })
    else:
        out["k_mix_td"] = BT * (3 * N + 12) * f + BT * N * 64 * f
    out["k_clip_rmsprop"] = 20 * P
    out["k_update"] = 24 * P
    for k in list(out):                       # the tensor-core variants of the reductions move the same bytes
        if k.startswith("k_reduce_group:"):
            out["k_reduce_tc:" + k.split(":")[1]] = out[k]
    return out


def load_traffic(workload):
    """DRAM bytes per launch (dram__bytes_read.sum + dram__bytes_write.sum) from the committed ncu --set full summary of
    THIS workload (profiles/traffic.json: {workload: {kernel: bytes}}; the flat r01 form is the 5v5 capture)."""
    try:
        t = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
    except Exception:
        return {}
    if workload in t and isinstance(t[workload], dict):
        return t[workload]
    if all(not isinstance(v, dict) for v in t.values()) and workload == "qmix_5v5_b32":
        return t
    return {}


def hbm_peak():
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    src = "MEASURED_PEAKS.json hbm_gbs (measured)" if "hbm_gbs" in peaks else "B200_PROFILING.md fallback 6650"
    return peak, src


class NullLog:
    def log_stat(self, *x): pass
    def info(self, *x): pass


def dist_max(x, world, device):
    if world > 1:
        t = th.tensor([x], dtype=th.float64, device=device)
        th.distributed.all_reduce(t, op=th.distributed.ReduceOp.MAX)
        return float(t.item())
    return x


def barrier(world, device):
    if world > 1:
        th.distributed.barrier()
    th.cuda.synchronize(device)


def gpu_synth_batch(M, scheme, groups, pre, B, TT, N, A, OBS, S, device, seed):
    """Synthetic episodes of SURVEY.md 8(d) generated ON the device (the 20v20 / B=1024 batch is 3.9 GB)."""
    from ma_league_b200.synthetic import fill_episode_batch
    g = th.Generator(device=device).manual_seed(seed)
    T = TT - 1
    avail = (th.rand(B, TT, N, A, generator=g, device=device) < 0.7).int()
    avail[..., 0] = 1
    e = th.empty(B, TT, N, A, device=device).exponential_(generator=g)
    actions = (avail.float() / e).argmax(-1, keepdim=True)
    del e
    lens = th.randint(max(T // 2, 1), T + 1, (B,), generator=g, device=device)
    lens[0] = T
    term = th.zeros(B, TT, 1, dtype=th.uint8, device=device)
    term[th.arange(B, device=device), lens - 1] = 1
    data = {"state": th.randn(B, TT, S, generator=g, device=device), "obs": th.randn(B, TT, N, OBS, generator=g, device=device),
            "actions": actions, "avail_actions": avail, "reward": th.randn(B, TT, 1, generator=g, device=device),
            "terminated": term}
    eb = M.EpisodeBatch(scheme, groups, B, TT, preprocess=pre, device=device)
    return fill_episode_batch(eb, data, lens)


# ------------------------------------------------------------------------------------------------ our arm
def run_ours(a, rank, world, device):
    import ma_league_b200 as M
    from ma_league_b200 import _native as nat
    from ma_league_b200.synthetic import make_args, make_scheme, synth_episode_data, fill_episode_batch
    nat.build()
    lib = nat.lib()
    for kv in a.opt:
        k, v = kv.split("=")
        nat.check(lib.mal_set_option(k.encode(), int(v)), "mal_set_option")
    d = workload_dims(a.workload)
    N, A, OBS, S, B, TT = d["N"], d["A"], d["OBS"], d["S"], d["B"], d["TT"]
    if a.buffer_size <= B:                              # sample() of a buffer holding exactly one batch returns views of the buffer itself
        a.buffer_size = B + max(B // 2, 1)
    th.manual_seed(1000 + rank)
    np.random.seed(1000 + rank)
    B_global = B
    if a.dp:
        assert B % world == 0, "--dp needs the batch to divide by the number of ranks"
        B = B // world                                   # this rank's shard of the global batch
        th.manual_seed(1000)                             # replicas start from identical parameters
    args = make_args(N, A, S, mixer=d["mixer"], double_q=True, device=device, batch_size=B, buffer_size=a.buffer_size,
                     data_parallel=bool(a.dp), dp_fused=not a.dp_nccl)
    scheme, groups, pre = make_scheme(N, A, OBS, S)
    buf = M.ReplayBuffer(scheme, groups, a.buffer_size, TT, preprocess=pre, device=device)
    mac = M.mac_REGISTRY[args.mac](buf.scheme, groups, args)
    learner = M.learner_REGISTRY[args.learner](mac, buf.scheme, NullLog(), args, name="home")
    learner.build_optimizer()

    # device-resident replay buffer pre-filled with synthetic episodes (every rank its own matchup data)
    gen = th.Generator().manual_seed(7 + rank)
    chunk = 256
    for s0 in range(0, a.buffer_size, chunk):
        n = min(chunk, a.buffer_size - s0)
        data, lens = synth_episode_data(n, TT, N, A, OBS, S, gen, var_len=True, device=device)
        lens[0] = TT - 1
        eb = fill_episode_batch(M.EpisodeBatch(scheme, groups, n, TT, preprocess=pre, device=device), data, lens)
        buf.insert_episode_batch(eb)

    # NB pre-sampled batches whose total size exceeds L2 (126 MB): inputs come from HBM on every step
    rb = buf._layout.record_bytes
    nb = max(4, -(-160 * 2 ** 20 // (B * rb)))
    batches, parents = [], []
    for _ in range(nb):
        smp = buf.sample(B)
        smp._storage.view(B, rb)[0].copy_(buf._storage.view(a.buffer_size, rb)[0])   # one full-length episode
        mt = int(smp.max_t_filled())
        assert mt == TT, mt
        parents.append(smp)
        batches.append(smp[:, :mt])                    # ma_experiment.py:235-236
    transitions = B * (TT - 1)

    # ---------------- value: batch resident in HBM
    # untimed: every rotating batch is seen twice (eager, then CUDA-graph capture) before the W warm-up steps
    for i in range(2 * nb):
        learner.train(batches[i % nb], t_env=i, episode_num=0)
    for i in range(a.warmup):
        learner.train(batches[i % nb], t_env=i, episode_num=0)
    barrier(world, device)
    launches0 = lib.mal_launch_count()
    sampler = ClockSampler(int(os.environ.get("LOCAL_RANK", 0)) if world > 1 else th.cuda.current_device())
    ev0, ev1 = th.cuda.Event(enable_timing=True), th.cuda.Event(enable_timing=True)
    barrier(world, device)
    wall0 = time.perf_counter()
    ev0.record()
    for i in range(a.steps):                           # EXACTLY K steps between one pair of CUDA events
        learner.train(batches[i % nb], t_env=i, episode_num=0)
    ev1.record()
    barrier(world, device)
    wall = time.perf_counter() - wall0
    clocks = sampler.stop()
    launches = lib.mal_launch_count() - launches0
    dev_ms = dist_max(ev0.elapsed_time(ev1), world, device)
    wall = dist_max(wall, world, device)
    ms_per_step = dev_ms / a.steps
    value = world * transitions / (ms_per_step * 1e-3)
    if a.dump_outputs and rank == 0:                    # before the passes below train the learner further
        dump_outputs(a.dump_outputs, learner)

    # ---------------- per-kernel profile (same steps again, CUDA events around every launch on its own stream)
    peak, peak_src = hbm_peak()
    # kernels timed ALONE: the step normally runs 2-3 kernel chains concurrently (fork/join side streams), where a
    # launch's event time includes queueing for SM resources behind its neighbours; the profile pass serialises them
    lib.mal_set_option(b"overlap", 0)
    learner.use_graphs = False              # replayed graphs bypass the per-launch events
    th.cuda.synchronize(device)
    nat.profile_begin()
    for i in range(a.steps):
        learner.train(batches[i % nb], t_env=i, episode_num=0)
    prof = nat.profile_end()
    lib.mal_set_option(b"overlap", 1)
    learner.use_graphs = True
    kb = kernel_bytes(d, d["mixer"], B)     # B = this rank's rows (its shard in --dp mode)
    traffic = load_traffic(a.workload)
    kern = []
    tot_ms = sum(ms for _, ms in prof.values())
    serial_ms_per_step = tot_ms / a.steps
    for name, (n, ms) in sorted(prof.items(), key=lambda kv: -kv[1][1]):
        per = ms / n
        byts = kb.get(name)
        kern.append({"kernel": name, "launches_per_step": round(n / a.steps, 2), "us_per_launch": round(per * 1e3, 2),
                     "us_per_step": round(ms / a.steps * 1e3, 2), "share": round(ms / tot_ms, 4),
                     "algo_gbs": round(byts / (per * 1e-3) / 1e9, 1) if byts else None,
                     "frac_of_hbm_peak": round(byts / (per * 1e-3) / 1e9 / peak, 4) if byts else None,
                     "dram_bytes_ncu": traffic.get(name.split(":")[0]) if ":" not in name else traffic.get(name, traffic.get(name.split(":")[0]))})
    top = kern[0]
    roofline = {"kernel": top["kernel"], "bound": "hbm", "achieved": top["algo_gbs"], "peak": peak, "unit": "GB/s",
                "frac": top["frac_of_hbm_peak"], "traffic": top["dram_bytes_ncu"],
                "peak_source": peak_src, "us_per_launch": top["us_per_launch"],
                "algorithmic_bytes_per_launch": kb.get(top["kernel"]),
                "note": "dominant kernel of the step; at B=32 it is the serial 201-step GRU recurrence, which is "
                        "latency-bound (cycles per timestep), not bandwidth-bound; memory-bound kernels are listed "
                        "under hbm_kernels"}

    # ---------------- e2e: batch in pinned host memory, H2D + train + D2H every step
    # The host keeps the sampled batches as compact WIRE records (EpisodeBatch.to_wire: no derivable fields, narrow flags);
    # every step copies its wire batch H2D (copy stream, double-buffered), expands it on the device into the staging batch
    # (EpisodeBatch.load_wire, one launch), trains, and reads the loss back.  `full_records` = the same loop shipping the
    # full packed records (the round-1 method), for comparison.
    if a.learner_only:                                  # profiling runs (tools/profile_round.sh): the learner step only
        return {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": a.steps, "warmup": a.warmup,
                "ms_per_step": ms_per_step, "config": {"workload": workload_string(a.workload)}, "learner_only": True,
                "gpu_launches": int(launches), "clocks": clocks, "roofline": roofline, "kernels": kern}
    n_pin = nb if B * rb * nb < 2 ** 31 else 2         # bound pinned host memory on the big workloads
    wb = parents[0].wire_bytes()
    stage = [M.EpisodeBatch(scheme, groups, B, TT, preprocess=pre, device=device) for _ in range(2)]
    copy_stream = th.cuda.Stream(device=device)
    out_ring = [th.empty(8, dtype=th.float32).pin_memory() for _ in range(2)]

    def e2e_variant(use_wire):
        if use_wire:
            pinned = [p_.to_wire().cpu().pin_memory() for p_ in parents[:n_pin]]
            land = [th.empty(B, wb, dtype=th.uint8, device=device) for _ in range(2)]
        else:
            pinned = [p_._storage.cpu().pin_memory() for p_ in parents[:n_pin]]
            land = [st_._storage for st_ in stage]
        ready = [th.cuda.Event(), th.cuda.Event()]
        consumed = [th.cuda.Event(), th.cuda.Event()]
        done = [th.cuda.Event(), th.cuda.Event()]

        def prefetch(i):
            slot = i % 2
            with th.cuda.stream(copy_stream):
                copy_stream.wait_event(consumed[slot])
                land[slot].copy_(pinned[i % n_pin], non_blocking=True)
                ready[slot].record(copy_stream)

        def e2e_steps(k, t0, pipelined):
            """Every step: H2D of its batch (copy stream, double-buffered), [unpack,] train, D2H of its loss/statistics.
            pipelined: the host waits for step i's result after it has enqueued step i+1 (a training loop that logs the
            previous step's loss); otherwise it synchronises on every step before enqueueing the next one."""
            prefetch(t0)
            cur = th.cuda.current_stream(device)
            last = float("nan")
            for i in range(t0, t0 + k):
                slot = i % 2
                if i + 1 < t0 + k:
                    prefetch(i + 1)
                cur.wait_event(ready[slot])
                if use_wire:
                    stage[slot].load_wire(land[slot])
                learner.train(stage[slot], t_env=i, episode_num=0)
                consumed[slot].record()
                out_ring[slot].copy_(learner.scalars()[:8], non_blocking=True)
                done[slot].record()
                if not pipelined:
                    done[slot].synchronize()           # this step's loss is on the host
                    last = float(out_ring[slot][1])
                elif i > t0:
                    done[slot ^ 1].synchronize()       # the previous step's loss is on the host
                    last = float(out_ring[slot ^ 1][1])
            done[(t0 + k - 1) % 2].synchronize()
            return float(out_ring[(t0 + k - 1) % 2][1]) if pipelined else last

        for c in consumed:
            c.record()
        # the H2D copy alone (pinned -> device on the copy stream): the e2e step cannot be shorter than this
        hs, he = th.cuda.Event(enable_timing=True), th.cuda.Event(enable_timing=True)
        with th.cuda.stream(copy_stream):
            land[0].copy_(pinned[0], non_blocking=True)
            hs.record(copy_stream)
            for _ in range(8):
                land[0].copy_(pinned[0], non_blocking=True)
            he.record(copy_stream)
        copy_stream.synchronize()
        h2d_ms = hs.elapsed_time(he) / 8
        res = {}
        k_e2e = max(a.steps, 100) if B * rb < 64 * 2 ** 20 else a.steps      # a longer window for the small (sub-ms) steps
        last_loss = float("nan")
        for pipelined in (False, True):
            e2e_steps(max(a.warmup, 3), 0, pipelined)
            barrier(world, device)
            t0 = time.perf_counter()
            last_loss = e2e_steps(k_e2e, 100, pipelined)
            barrier(world, device)
            res[pipelined] = dist_max(time.perf_counter() - t0, world, device)
        assert np.isfinite(last_loss)
        nbytes = B * (wb if use_wire else rb)
        return {"value": world * transitions * k_e2e / res[True], "unit": UNIT, "h2d_bytes_per_step": nbytes,
                "d2h_bytes_per_step": 32, "ms_per_step": res[True] / k_e2e * 1e3, "steps": k_e2e,
                "h2d_copy_alone_ms": round(h2d_ms, 4), "h2d_gbs": round(nbytes / (h2d_ms * 1e-3) / 1e9, 1),
                "sync_every_step": {"value": world * transitions * k_e2e / res[False], "ms_per_step": res[False] / k_e2e * 1e3,
                                    "how": "same, but the host synchronises on each step's loss before enqueueing the next step"}}

    how_common = ("double-buffered H2D on a copy stream -> %sQLearner.train -> loss D2H; every step's loss is read on the host, one "
                  "step behind the enqueue (the host enqueues step i+1, then waits for step i's result)")
    ev = {"wire_records": e2e_variant(True), "full_records": e2e_variant(False)}
    ev["wire_records"]["how"] = ("pinned host batch as compact wire records (EpisodeBatch.to_wire: %d of %d bytes per episode) -> " % (wb, rb)) + \
        how_common % "EpisodeBatch.load_wire (device unpack, one launch) -> "
    ev["full_records"]["how"] = "pinned host batch as full packed records -> " + how_common % ""
    # both are public-API paths; the headline is the faster one on THIS run (the wire form wins when the H2D copy is the
    # bottleneck, i.e. several GPUs sharing the host's PCIe / memory bandwidth; the extra unpack launch loses when it is not)
    best = max(ev, key=lambda k: ev[k]["value"])
    e2e = dict(ev[best])
    e2e["path"] = best
    other = "full_records" if best == "wire_records" else "wire_records"
    e2e["alternative"] = dict(ev[other], path=other)

    extra = {}
    # ---------------- M1': the learner-side input pipeline (sample + truncate + train), ma_experiment.py:231-241
    if not a.dp:
        try:
            extra["m1_prime"] = measure_m1_prime(a, M, learner, buf, B, TT, world, device)
        except Exception as ex:
            extra["m1_prime_error"] = repr(ex)

    # ---------------- second headline metric: act-select agent-steps/s (public API, default RNG = torch's Philox stream)
    extra["act_select"] = {}
    for bs in (1, B, 1024):
        eb = M.EpisodeBatch(scheme, groups, bs, TT, preprocess=pre, device=device)
        for r_ in range(0, bs, a.buffer_size):
            n_ = min(a.buffer_size, bs - r_)
            eb._storage[r_ * rb:(r_ + n_) * rb].copy_(buf._storage[:n_ * rb])
        for validate in (True, False):
            # validate=True is the DEFAULT (the reference's Categorical raises ValueError on an all-zero avail row, which
            # costs a device->host sync per call); validate_avail=False skips that check
            mac.action_selector.validate = validate
            mac.init_hidden(bs)
            for i in range(10):
                mac.select_actions(eb, t_ep=1 + i % 100, t_env=i)
            th.cuda.synchronize(device)
            reps = 200
            s_, e_ = th.cuda.Event(enable_timing=True), th.cuda.Event(enable_timing=True)
            w0 = time.perf_counter()
            s_.record()
            for i in range(reps):
                mac.select_actions(eb, t_ep=1 + i % 100, t_env=i)
            e_.record()
            th.cuda.synchronize(device)
            api_us = (time.perf_counter() - w0) / reps * 1e6
            nat.profile_begin()
            for i in range(50):
                mac.select_actions(eb, t_ep=1 + i % 100, t_env=i)
            pk = nat.profile_end()["k_agent_step"]
            extra["act_select"]["bs%d_%s" % (bs, "validate_default" if validate else "validate_off")] = {
                "agent_steps_per_s": round(bs * N * reps / (s_.elapsed_time(e_) * 1e-3), 1),
                "api_us_per_call": round(api_us, 2), "kernel_us": round(pk[1] / pk[0] * 1e3, 2),
                "kernel_agent_steps_per_s": round(bs * N / (pk[1] / pk[0] * 1e-3), 1)}
    mac.action_selector.validate = True

    # ---------------- the rollout loop around act-select (SURVEY.md 8 f1): B lock-step matches, device-resident batches
    try:
        from ma_league_b200.steppers import BatchedEpisodeStepper, SyntheticVecEnv
        env = SyntheticVecEnv(B, N, A, OBS, S, TT - 1, n_teams=1, seed=3, device=device, min_len=TT - 1)
        roll = {}
        for fuse, validate in ((True, False), (True, True), (False, False)):
            mac.action_selector.validate = validate
            stp = BatchedEpisodeStepper(args, None, env, sync_every=50, fuse=fuse)
            stp.initialize(scheme, groups, pre, mac)
            stp.run(test_mode=False)
            th.cuda.synchronize(device)
            l0 = lib.mal_launch_count()
            w0 = time.perf_counter()
            stp.run(test_mode=False)
            th.cuda.synchronize(device)
            dt = time.perf_counter() - w0
            roll["%s_validate_%s" % ("fused_step" if fuse else "separate_calls", "default" if validate else "off")] = {
                "agent_steps_per_s": round(B * N * (TT - 1) / dt, 1), "env_steps_per_s": round(B * (TT - 1) / dt, 1),
                "ms_per_timestep": round(dt / (TT - 1) * 1e3, 4), "our_launches_per_timestep": round((lib.mal_launch_count() - l0) / TT, 2)}
        mac.action_selector.validate = True
        roll["what"] = ("BatchedEpisodeStepper.run over %d timesteps: fused_step = ONE launch per timestep (pre-transition update + "
                        "previous reward/terminated + act-select + actions/one-hot), separate_calls = update / select_actions / "
                        "update; the synthetic environment's own step (3 small torch ops) is inside the timed loop" % (TT - 1))
        extra["rollout_loop_bs%d" % B] = roll
    except Exception as ex:                                  # the extra leg must never take the headline down
        extra["rollout_loop_error"] = repr(ex)

    # ---------------- memory-bound kernels against the HBM roofline (kernel time from CUDA events around the launch)
    hbm = []
    ids = [th.as_tensor(np.random.choice(a.buffer_size, B, replace=False), device=device) for _ in range(20)]
    for i in ids[:3]:
        buf[i]
    th.cuda.synchronize(device)
    w0 = time.perf_counter()
    nat.profile_begin()
    for i in ids:
        buf[i]
    pk = nat.profile_end()["k_record_copy_tma"]
    api_us = (time.perf_counter() - w0) / len(ids) * 1e6
    us = pk[1] / pk[0] * 1e3
    hbm.append({"kernel": "k_record_copy_tma", "what": "ReplayBuffer.sample(%d) gather" % B, "bytes": 2 * B * rb,
                "us": round(us, 2), "gbs": round(2 * B * rb / (us * 1e-6) / 1e9, 1),
                "frac_of_hbm_peak": round(2 * B * rb / (us * 1e-6) / 1e9 / peak, 4), "api_us_per_call": round(api_us, 1)})
    nbig = min(a.buffer_size, 768)
    big_ids = th.as_tensor(np.random.choice(a.buffer_size, nbig, replace=False), device=device)
    buf[big_ids]
    nat.profile_begin()
    for _ in range(5):
        buf[big_ids]
    pk = nat.profile_end()["k_record_copy_tma"]
    us = pk[1] / pk[0] * 1e3
    hbm.append({"kernel": "k_record_copy_tma", "what": "gather of %d episodes (> L2)" % nbig, "bytes": 2 * nbig * rb,
                "us": round(us, 2), "gbs": round(2 * nbig * rb / (us * 1e-6) / 1e9, 1),
                "frac_of_hbm_peak": round(2 * nbig * rb / (us * 1e-6) / 1e9 / peak, 4)})
    for k in kern:
        if k["kernel"].split(":")[0] in ("k_mix_td", "k_q_head", "k_clip_rmsprop", "k_update", "k_fc2_grad") or \
                k["kernel"] == "k_linear_group:mixer_l1":
            hbm.append({"kernel": k["kernel"], "what": "learner step", "us": k["us_per_launch"], "gbs": k["algo_gbs"],
                        "algorithmic_bytes": kb.get(k["kernel"]), "dram_bytes_ncu": k["dram_bytes_ncu"],
                        "frac_of_hbm_peak": k["frac_of_hbm_peak"]})

    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": a.steps, "warmup": a.warmup,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong" if a.dp else "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": workload_string(a.workload),
                       "transitions_per_step": transitions,
                       "parallelism": ("data-parallel x%d: global batch %d split over the ranks, %s" % (
                           world, B_global, "NCCL all_reduce of gradient + statistic sums" if a.dp_nccl or not getattr(learner, "_dp_sym", None)
                           else "peer-memory all-reduce fused into the clip+RMSprop prologue")) if a.dp
                       else "league-sharded x%d: one independent matchup per GPU (no collective)" % world,
                       "l2": "inputs rotate over %d sampled batches (%.0f MB) > 126 MB L2" % (nb, nb * B * rb / 2 ** 20),
                       "replay_buffer_episodes": a.buffer_size,
                       "math": "fp32; batched projections on tcgen05 3xTF32 (fp32-accurate), recurrences fp32 FFMA2",
                       "launch": "one CUDA graph per batch address set (captured on the 2nd sighting, replayed after)"},
            "e2e": e2e, "e2e_sync_every_step": e2e["sync_every_step"],
            "gpu_launches": int(launches), "launches_per_step": launches / a.steps,
            "wall_ms_per_step": wall / a.steps * 1e3, "sum_of_kernels_ms_per_step": serial_ms_per_step, "clocks": clocks, "roofline": roofline, "kernels": kern,
            "hbm_kernels": hbm}
    line.update(extra)
    return line


def dump_outputs(out_dir, learner):
    """What QLearner.train() leaves its caller after a step, as float32 .npy files: the logged statistics (mask sum,
    loss, |td| mean, q_taken mean, target mean, grad norm), the clipped gradient (p.grad) and the updated parameters."""
    from ma_league_b200 import _native as nat
    flat = lambda ts: th.cat([t.detach().reshape(-1) for t in ts])      # noqa: E731
    arrays = {"train_stats": learner.scalars()[nat.SC_MASK_SUM:nat.SC_GRAD_NORM + 1],
              "grad": flat(p.grad for p in learner.parameters()),
              "agent_params": flat(learner.mac.parameters())}
    mixer_params = list(learner.mixer.parameters())                    # VDN has none
    if mixer_params:
        arrays["mixer_params"] = flat(mixer_params)
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.float().cpu().numpy())


def measure_m1_prime(a, M, learner, buf, B, TT, world, device):
    """M1' = B*T / t(sample + truncate + train): (i) the reference's exact call sequence through this repo's API
    (`sample` -> new storage every step -> `max_t_filled()` host sync -> slice -> `train`, ma_experiment.py:231-241),
    where the step's CUDA graph only replays when the caching allocator hands back a block seen before; (ii) the fused
    `train_from_buffer` (persistent staging batch, padding masked, no host sync)."""
    out = {}
    K = max(a.steps, 40)
    transitions = B * (TT - 1)
    for name in ("reference_sequence", "train_from_buffer"):
        def one(i):
            if name == "reference_sequence":
                smp = buf.sample(B)
                mt = smp.max_t_filled()
                learner.train(smp[:, :int(mt)], t_env=i, episode_num=0)
            else:
                learner.train_from_buffer(buf, B, t_env=i, episode_num=0)
        for i in range(max(a.warmup, 5)):
            one(i)
        barrier(world, device)
        r0, e0, c0 = learner.n_graph_replays, learner.n_eager_steps, learner.n_graph_captures
        t0 = time.perf_counter()
        for i in range(K):
            one(i)
        th.cuda.synchronize(device)
        dt = dist_max(time.perf_counter() - t0, world, device)
        out[name] = {"value": world * transitions * K / dt, "unit": UNIT, "ms_per_step": dt / K * 1e3, "steps": K,
                     "graph_replays": learner.n_graph_replays - r0, "eager_steps": learner.n_eager_steps - e0,
                     "graph_captures": learner.n_graph_captures - c0,
                     "transitions_counted": "B*T with T = %d (sampled episodes are shorter: the truncated step does less work)" % (TT - 1)}
    return out


# ------------------------------------------------------------------------------------------------ data-parallel leg
DP_WORKLOAD = "qmix_20v20_b1024"


def run_dp_leg(a, rank, world, device):
    """BASELINE.json configs[4]: QMIX 20v20, global B=1024, T=200, data-parallel over the ranks (strong scaling).
    Every rank trains on its B/world shard; gradients + statistic sums meet in (fused) the peer-memory all-reduce inside
    the optimiser prologue, or (nccl) one NCCL all_reduce.  Rank 0 also times the single-GPU step on the full batch, so
    the speed-up is measured inside one run.  Replicas are asserted bit-identical after the timed steps."""
    import ma_league_b200 as M
    from ma_league_b200 import _native as nat
    from ma_league_b200.synthetic import make_args, make_scheme
    d = workload_dims(DP_WORKLOAD)
    N, A, OBS, S, Bg, TT = d["N"], d["A"], d["OBS"], d["S"], d["B"], d["TT"]
    assert Bg % world == 0
    B = Bg // world
    scheme, groups, pre = make_scheme(N, A, OBS, S)
    K, W = a.dp_steps, 3
    out = {"workload": workload_string(DP_WORKLOAD), "global_batch": Bg, "batch_per_rank": B, "steps": K, "warmup": W,
           "scaling": "strong", "n_gpus": world}

    def build(batch_size, dp, fused):
        th.manual_seed(4242)                                 # identical initial parameters on every rank
        args = make_args(N, A, S, mixer="qmix", double_q=True, device=device, batch_size=batch_size, buffer_size=8,
                         data_parallel=dp, dp_fused=fused)
        holder = M.ReplayBuffer(scheme, groups, 1, TT, preprocess=pre, device=device)     # only for the derived scheme
        mac = M.mac_REGISTRY[args.mac](holder.scheme, groups, args)
        learner = M.learner_REGISTRY[args.learner](mac, holder.scheme, NullLog(), args, name="home")
        learner.build_optimizer()
        return mac, learner

    def timed(learner, batch, sync_world):
        for i in range(W):
            learner.train(batch, t_env=i, episode_num=0)
        if sync_world:
            barrier(world, device)
        else:
            th.cuda.synchronize(device)
        e0, e1 = th.cuda.Event(enable_timing=True), th.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(K):
            learner.train(batch, t_env=i, episode_num=0)
        e1.record()
        th.cuda.synchronize(device)
        ms = e0.elapsed_time(e1) / K
        return dist_max(ms, world, device) if sync_world else ms

    # ---- single-GPU reference time on the full batch (rank 0; the others wait at the barrier)
    n1_ms = None
    if rank == 0:
        full = gpu_synth_batch(M, scheme, groups, pre, Bg, TT, N, A, OBS, S, device, seed=99)
        mac1, l1 = build(Bg, False, False)
        n1_ms = timed(l1, full, False)
        del l1, mac1, full
        th.cuda.empty_cache()
    t = th.tensor([n1_ms or 0.0], dtype=th.float64, device=device)
    if world > 1:
        th.distributed.broadcast(t, 0)
    n1_ms = float(t.item())
    out["n1_ms_per_step"] = n1_ms
    out["n1_transitions_per_s"] = Bg * (TT - 1) / (n1_ms * 1e-3)
    if world == 1:
        out["modes"] = {}
        return out

    shard = gpu_synth_batch(M, scheme, groups, pre, B, TT, N, A, OBS, S, device, seed=100 + rank)
    peak, _ = hbm_peak()
    modes = {}
    for mode in ("fused", "nccl"):
        mac, learner = build(B, True, mode == "fused")
        ms = timed(learner, shard, True)
        # exchange time: CUDA events around (cross-rank barrier + peer all-reduce kernel + clip/RMSprop) resp.
        # (NCCL all_reduce + k_sumsq + clip/RMSprop); per-rank median, max over ranks
        learner.dp_profile = []
        for i in range(K):
            learner.train(shard, t_env=i, episode_num=0)
        th.cuda.synchronize(device)
        ex_us = statistics.median([e0.elapsed_time(e1) * 1e3 for e0, e1 in learner.dp_profile])
        learner.dp_profile = None
        nat.lib().mal_set_option(b"overlap", 0)             # kernels timed alone (no queueing behind side-stream neighbours)
        nat.profile_begin()
        for i in range(K):
            learner.train(shard, t_env=i, episode_num=0)
        prof = nat.profile_end()
        nat.lib().mal_set_option(b"overlap", 1)
        kb = kernel_bytes(d, "qmix", B)
        tot = sum(v[1] for v in prof.values())
        kern = [{"kernel": k, "us_per_launch": round(v[1] / v[0] * 1e3, 2), "share": round(v[1] / tot, 4),
                 "frac_of_hbm_peak": round(kb[k] / (v[1] / v[0] * 1e-3) / 1e9 / peak, 4) if k in kb else None}
                for k, v in sorted(prof.items(), key=lambda kv: -kv[1][1])[:8]]
        # replicas must be bit-identical: same reduced gradient, same update everywhere
        flat = th.cat([p.detach().reshape(-1) for p in learner.parameters()])
        sig = th.stack([flat.view(th.int32).to(th.int64).sum(), flat.double().sum().view(th.int64)])
        sigs = [th.zeros_like(sig) for _ in range(world)]
        th.distributed.all_gather(sigs, sig)
        identical = all(bool((s_ == sigs[0]).all()) for s_ in sigs)
        assert identical, "data-parallel replicas diverged (%s)" % mode
        used_fused = bool(getattr(learner, "_dp_sym", None))
        modes[mode] = {"ms_per_step": ms, "transitions_per_s": Bg * (TT - 1) / (ms * 1e-3),
                       "speedup_vs_n1": n1_ms / ms, "efficiency": n1_ms / ms / world,
                       "exchange_us": dist_max(ex_us, world, device),
                       "exchange_what": ("cross-rank barrier (symmetric-memory signal pads) + k_peer_allreduce_grad + k_clip_rmsprop"
                                         if used_fused else "NCCL all_reduce + k_sumsq + k_clip_rmsprop"),
                       "mode": "peer-memory all-reduce fused into the optimiser prologue" if used_fused else "NCCL all_reduce",
                       "fused_available": used_fused if mode == "fused" else None,
                       "fused_error": getattr(learner, "_dp_sym_error", None) if mode == "fused" and not used_fused else None,
                       "replicas_bit_identical": identical, "top_kernels": kern}
        del learner, mac
        th.cuda.empty_cache()
    out["modes"] = modes
    best = min(modes.values(), key=lambda m: m["ms_per_step"])
    out.update(ms_per_step=best["ms_per_step"], speedup_vs_n1=best["speedup_vs_n1"], exchange_us=best["exchange_us"],
               mode=best["mode"])
    # limiter: what is left of the per-rank step besides the ideal n1/world share
    ideal = n1_ms / world
    out["limiter"] = {"ideal_ms": ideal, "over_ideal_ms": best["ms_per_step"] - ideal, "exchange_ms": best["exchange_us"] * 1e-3,
                      "note": "over_ideal - exchange = per-rank kernel tail (kernels that do not shrink with B/world: "
                              "weight staging, launch latency, the serial 201-step recurrences)"}
    return out


# ------------------------------------------------------------------------------------------------ reference arm
def _port_learner(workload, device="cpu"):
    from oracle import np_oracle as O, torch_port as TP
    from ma_league_b200.synthetic import synth_episode_data
    d = workload_dims(workload)
    N, A, OBS, S, B, TT = d["N"], d["A"], d["OBS"], d["S"], d["B"], d["TT"]
    rng = np.random.default_rng(0)
    ap = O.init_params(O.agent_param_shapes(OBS + A + N, A), rng)
    mp = O.init_params(O.qmix_param_shapes(S, N), rng) if d["mixer"] == "qmix" else None
    L = TP.TorchPortLearner(ap, ap, mp, mp, mixer=d["mixer"], double_q=True, gamma=0.99, lr=5e-4, alpha=0.99, eps=1e-5,
                            clip=10, device=device)
    gen = th.Generator().manual_seed(0)
    data, lens = synth_episode_data(B, TT, N, A, OBS, S, gen, var_len=False)
    data["actions_onehot"] = th.from_numpy(O.onehot(data["actions"].numpy(), A))
    data["filled"] = th.ones(B, TT, 1, dtype=th.long)
    data = {k: v.to(device) for k, v in data.items()}
    return L, data, d, ap


def run_reference(a, bounded_s=None, workload=None, device="cpu"):
    """The reference's CPU path (torch port, all host threads).  Returns (value, ms_per_step, steps, cores, sample)."""
    workload = workload or a.workload
    cores = os.cpu_count() or 1
    th.set_num_threads(cores)
    L, data, d, _ = _port_learner(workload, device)
    B, TT = d["B"], d["TT"]
    warm, steps = a.warmup, a.steps
    if bounded_s is not None:
        warm, steps = (2, 1000) if bounded_s >= 4 else (1, 1000)
    sync = (lambda: th.cuda.synchronize()) if device != "cpu" else (lambda: None)
    for _ in range(warm):
        L.train(data)
    sync()
    t0 = time.perf_counter()
    done = 0
    for _ in range(steps):
        L.train(data)
        done += 1
        if bounded_s is not None and time.perf_counter() - t0 > bounded_s:
            break
    sync()
    el = time.perf_counter() - t0
    return B * (TT - 1) * done / el, el / done * 1e3, done, cores, \
        "%d full train steps (B=%d, T=%d) of oracle/torch_port.py on %s" % (
            done, B, TT - 1, "%d host threads" % cores if device == "cpu" else "cuda (PyTorch eager)")


def cpu_side_baselines(a):
    """BASELINE.md section 3 on the host cores: M2 act-select (bs=1, bs=B), replay insert/sample, M1' (sample + train)
    and M1 for configs 1-3 -- all through oracle/torch_port.py (the reference's ATen op sequence), bounded samples."""
    from oracle import torch_port as TP
    out = {}
    L, data, d, ap = _port_learner(a.workload)
    N, A, B, TT = d["N"], d["A"], d["B"], d["TT"]
    p = TP.to_params(ap, requires_grad=False)
    # ---- M2: BasicMAC.select_actions (agent step + epsilon-greedy with torch's CPU generator)
    for bs in (1, B):
        sub = {k: v[:bs] for k, v in data.items()}
        h = th.zeros(bs * N, 64)
        for i in range(5):
            _, _, h = TP.select_actions(p, sub, 1 + i, h, 0.3)
        reps = 300 if bs == 1 else 100
        t0 = time.perf_counter()
        for i in range(reps):
            _, _, h = TP.select_actions(p, sub, 1 + i % 100, h, 0.3)
        dt = time.perf_counter() - t0
        out["act_select_bs%d" % bs] = {"agent_steps_per_s": round(bs * N * reps / dt, 1), "us_per_call": round(dt / reps * 1e6, 1),
                                       "sample": "%d select_actions calls" % reps}
    # ---- replay: CPU-resident buffer of 256 episodes (per-key tensors), insert of 32 and sample(32)
    n_buf = 256
    bufd = {k: v[th.arange(n_buf) % B].clone() for k, v in data.items()}
    t0 = time.perf_counter()
    reps = 20
    for i in range(reps):
        TP.replay_sample(bufd, n_buf, B)
    dt = time.perf_counter() - t0
    row_bytes = sum(v[0].numel() * v.element_size() for v in data.values())
    out["replay_sample"] = {"ms_per_call": round(dt / reps * 1e3, 3), "gbs": round(2 * B * row_bytes / (dt / reps) / 1e9, 2),
                            "sample": "%d x sample(%d) from a %d-episode host buffer" % (reps, B, n_buf)}
    t0 = time.perf_counter()
    for i in range(reps):
        lo = (i * B) % (n_buf - B)
        for k, v in bufd.items():                       # insert_episode_batch: slice-assign per key (replay_buffer.py:22-41)
            v[lo:lo + B] = data[k]
    dt = time.perf_counter() - t0
    out["replay_insert"] = {"ms_per_call": round(dt / reps * 1e3, 3), "sample": "%d x insert of %d episodes" % (reps, B)}
    # ---- M1': sample + max_t_filled + truncate + train
    t0 = time.perf_counter()
    done = 0
    while done < 3 or time.perf_counter() - t0 < 2.0:
        smp = TP.replay_sample(bufd, n_buf, B)
        mt = int(smp["filled"].sum(1).max())
        L.train({k: v[:, :mt] for k, v in smp.items()})
        done += 1
        if done >= 20:
            break
    dt = time.perf_counter() - t0
    out["m1_prime"] = {"value": round(B * (TT - 1) * done / dt, 1), "unit": UNIT, "ms_per_step": round(dt / done * 1e3, 2),
                       "sample": "%d x (sample + truncate + train)" % done}
    # ---- M1 for the other CPU-affordable configs (bounded: ~2 s each)
    for wl in ("qmix_3v3_b32", "vdn_5v5_b32", "qmix_10v10_b128"):
        if wl == a.workload:
            continue
        try:
            v, ms, done, cores, sample = run_reference(a, bounded_s=2.0, workload=wl)
            out["m1_" + wl] = {"value": round(v, 1), "unit": UNIT, "ms_per_step": round(ms, 2), "sample": sample}
        except Exception as ex:
            out["m1_" + wl] = {"error": repr(ex)}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=60)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="qmix_5v5_b32")
    ap.add_argument("--buffer-size", dest="buffer_size", type=int, default=1024)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--learner-only", dest="learner_only", action="store_true", help="profiling runs: value + per-kernel table only")
    ap.add_argument("--dp", action="store_true", help="data-parallel mode (config 5): the batch is split over the ranks, "
                    "gradients meet in the fused peer-memory all-reduce (strong scaling)")
    ap.add_argument("--dp-nccl", dest="dp_nccl", action="store_true", help="with --dp: exchange through NCCL all_reduce instead")
    ap.add_argument("--no-dp-leg", action="store_true", help="skip the config-5 data-parallel leg that WORLD_SIZE > 1 runs adds")
    ap.add_argument("--dp-leg", action="store_true", help="run the config-5 leg also at one GPU (its single-GPU step time)")
    ap.add_argument("--dp-steps", dest="dp_steps", type=int, default=10)
    ap.add_argument("--opt", action="append", default=[], help="library switch name=int (mal_set_option), e.g. reduce_tc=0")
    ap.add_argument("--dump-outputs", dest="dump_outputs", metavar="DIR",
                    help="write the outputs of the last timed step as DIR/<name>.npy (float32)")
    a = ap.parse_args()
    if a.dump_outputs and a.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    a.warmup = max(a.warmup, 3)
    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))

    if a.impl == "reference":
        if rank != 0:
            return
        v, ms, done, cores, sample = run_reference(a)
        print(json.dumps({"impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": a.gpus,
                          "steps": done, "warmup": a.warmup, "ms_per_step": ms, "higher_is_better": True,
                          "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                          "config": {"workload": workload_string(a.workload), "where": "host CPU, %d threads" % cores},
                          "cpu_baseline": {"value": v, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
                          "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))
        return

    if not th.cuda.is_available():
        raise SystemExit("bench.py --impl ours needs a CUDA device (no CPU fallback)")
    th.cuda.set_device(local)
    device = "cuda:%d" % local
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        th.distributed.init_process_group("nccl", device_id=th.device(device))
    line = run_ours(a, rank, world, device)
    if (world > 1 and not a.no_dp_leg and not a.dp) or a.dp_leg:
        try:
            line["dp"] = run_dp_leg(a, rank, world, device)
        except Exception as ex:                                  # the extra leg must never take the headline down
            import traceback
            line["dp"] = {"error": repr(ex), "trace": traceback.format_exc()[-1500:]}
    if rank == 0:
        if world == 1 and not a.no_cpu_baseline:
            v, ms, done, cores, sample = run_reference(a, bounded_s=10.0)
            line["cpu_baseline"] = {"value": v, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample,
                                    "ms_per_step": ms}
            try:
                line["cpu_baseline"]["other"] = cpu_side_baselines(a)
            except Exception as ex:
                line["cpu_baseline"]["other_error"] = repr(ex)
            try:                                                 # optional bar: the same ATen op sequence in PyTorch eager on the GPU
                v, ms, done, _, sample = run_reference(a, bounded_s=3.0, device=device)
                line["gpu_eager_baseline"] = {"value": v, "unit": UNIT, "ms_per_step": ms, "kind": "port on cuda", "sample": sample}
            except Exception as ex:
                line["gpu_eager_baseline"] = {"error": repr(ex)}
        print(json.dumps(line), flush=True)
    if world > 1:
        th.distributed.barrier()
        th.distributed.destroy_process_group()


if __name__ == "__main__":
    main()
