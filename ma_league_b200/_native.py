"""ctypes binding of libmal_b200.so (C ABI: include/mal_b200.h).

This is the reference-side stub a maintainer would add (see INTEGRATION.md): plain pointers and sizes go
across the boundary, torch is only used by the callers for device memory and the current stream.
There is NO fallback: if the shared library is missing or a call fails, an exception is raised.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
import sys

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libmal_b200.so")
SRC = os.path.join(_HERE, "csrc", "mal_b200.cu")
ABI_VERSION = 6

MIXER_VDN, MIXER_QMIX2, MIXER_QMIX1, MIXER_NONE = 0, 1, 2, 3    # MIXER_NONE: independent Q-learners (IQL)
AGENT_RNN, AGENT_DQN = 0, 1
IN_NO_LAST_ACTION, IN_NO_AGENT_ID = 1, 2     # agent-input switches (mal_learner_cfg_t.agent_input, mal_rollout_io_t.agent_input)
RETURNS_ONE_STEP, RETURNS_TD_LAMBDA = 0, 1   # mal_learner_cfg_t.returns: 1-step or TD(lambda) targets
STEP_DENSE = 1                               # dense_input of mal_agent_step / mal_dqn_step: bit 0; bits 1..2 = IN_* << 1
SC_MASK_SUM, SC_LOSS, SC_TD_ABS, SC_Q_TAKEN, SC_TARGET, SC_GRAD_NORM, SC_MASK_COUNT, SC_STATUS = range(8)
SC_RAW0 = 8     # raw sums: sum mtd^2, sum |mtd|, sum q_tot*m, sum targets*m, sum m, count
HID = 64
MAX_ACTIONS = 32
MAX_EMBED = 32
MAX_POLICIES = 1024                          # n_policies cap of the per-match policy entries (MAL_MAX_POLICIES)


class MalError(RuntimeError):
    pass


class Field(C.Structure):
    _fields_ = [("ptr", C.c_void_p), ("sb", C.c_int64), ("st", C.c_int64)]


class Batch(C.Structure):
    _fields_ = [("B", C.c_int32), ("TT", C.c_int32), ("N", C.c_int32), ("A", C.c_int32), ("OBS", C.c_int32),
                ("S", C.c_int32), ("obs", Field), ("onehot", Field), ("actions", Field), ("avail", Field),
                ("state", Field), ("reward", Field), ("terminated", Field), ("filled", Field), ("weight", Field)]


class LearnerCfg(C.Structure):
    _fields_ = [("mixer", C.c_int32), ("double_q", C.c_int32), ("embed", C.c_int32), ("hyper_embed", C.c_int32),
                ("gamma", C.c_float), ("lr", C.c_float), ("alpha", C.c_float), ("eps", C.c_float),
                ("clip", C.c_float), ("save_q", C.c_int32), ("unnormalized", C.c_int32), ("freeze_agent", C.c_int32),
                ("agent_kind", C.c_int32), ("agent_input", C.c_int32), ("returns", C.c_int32), ("td_lambda", C.c_float),
                ("target_tau", C.c_double)]


_PLAN_FIELDS = ["total_bytes", "n_agent_params", "n_mixer_params", "x_on", "x_tg", "gi_on", "gi_tg", "h_on", "h_tg",
                "gates", "mac_out", "target_mac_out", "chosen", "target_max", "argmax", "mask", "y1_on", "y1_tg",
                "a2_on", "a2_tg", "q_tot", "target_q_tot", "targets", "td", "d_a2", "d_y1", "d_chosen", "d_g", "d_x",
                "dh_head", "partials", "partials_bytes", "scalars", "w_t"]


class AdamHyper(C.Structure):
    """mal_adam_t: the hyper-parameters of the Adam step (mal_learner_step_adam, mal_clip_adam)."""
    _fields_ = [("lr", C.c_double), ("beta1", C.c_double), ("beta2", C.c_double), ("eps", C.c_double),
                ("weight_decay", C.c_double), ("clip", C.c_float)]


class SoftTarget(C.Structure):
    """mal_soft_target_t: tau and the target flats of the soft target update (the *_soft optimiser entries)."""
    _fields_ = [("tau", C.c_double), ("target_agent", C.c_void_p), ("target_mixer", C.c_void_p)]


def adam_state_floats(n_params: int) -> int:
    """MAL_ADAM_STATE_FLOATS: exp_avg [P] | exp_avg_sq [P] | step (f32) | ticket (u32)."""
    return 2 * n_params + 2


class Plan(C.Structure):
    _fields_ = [(n, C.c_int64) for n in _PLAN_FIELDS]


class Select(C.Structure):
    _fields_ = [("avail", C.c_void_p), ("avail_sb", C.c_int64), ("epsilon", C.c_float), ("rng_mode", C.c_int32),
                ("u", C.c_void_p), ("e", C.c_void_p), ("seed", C.c_uint64), ("offset", C.c_uint64),
                ("actions", C.c_void_p), ("greedy", C.c_void_p), ("status", C.c_void_p)]


class RolloutIO(C.Structure):
    _fields_ = [("state_dim", C.c_int32),
                ("env_state", C.c_void_p), ("env_state_sb", C.c_int64), ("env_avail", C.c_void_p), ("env_avail_sb", C.c_int64),
                ("env_obs", C.c_void_p), ("env_obs_sb", C.c_int64), ("alive", C.c_void_p), ("prev_reward", C.c_void_p),
                ("prev_done", C.c_void_p), ("state_t", C.c_void_p), ("state_sb", C.c_int64), ("avail_t", C.c_void_p),
                ("avail_sb", C.c_int64), ("obs_t", C.c_void_p), ("obs_sb", C.c_int64), ("filled_t", C.c_void_p),
                ("filled_sb", C.c_int64), ("actions_t", C.c_void_p), ("actions_sb", C.c_int64), ("onehot_t", C.c_void_p),
                ("onehot_sb", C.c_int64), ("onehot_tm1", C.c_void_p), ("onehot_tm1_sb", C.c_int64),
                ("reward_tm1", C.c_void_p), ("reward_sb", C.c_int64), ("term_tm1", C.c_void_p), ("term_sb", C.c_int64),
                ("agent_input", C.c_int32)]


RED_A_DENSE, RED_A_AGENT_IN, RED_A_STATE = 0, 1, 2   # mal_red_prob_t loaders (mal_debug_reduce a_kind)
RED_FFMA, RED_TC_MN0, RED_TC_MN1, RED_TC_MN2, RED_TC3 = range(5)   # mal_debug_reduce flavour


class RedProb(C.Structure):
    """mal_red_prob_t: one problem of mal_debug_reduce."""
    _fields_ = [("M", C.c_int64), ("rows_per_chunk", C.c_int64), ("K", C.c_int32), ("Nout", C.c_int32),
                ("shift", C.c_int32), ("dY", C.c_void_p), ("ldy", C.c_int64), ("A", C.c_void_p), ("lda", C.c_int64),
                ("part_w", C.c_void_p), ("part_b", C.c_void_p)]


class WireLayout(C.Structure):
    _fields_ = [(n, C.c_int64) for n in ("record_bytes", "off_state", "off_obs", "off_reward", "off_actions", "off_avail",
                                         "off_flags")]


_PROTOS = {
    "mal_version": (C.c_int, []),
    "mal_last_error": (C.c_char_p, []),
    "mal_launch_count": (C.c_uint64, []),
    "mal_count_launches": (None, [C.c_uint64]),
    "mal_profile_begin": (C.c_int, []),
    "mal_profile_end": (C.c_int, [C.c_char_p, C.c_int64]),
    "mal_profile_end_timeline": (C.c_int, [C.c_char_p, C.c_int64]),
    "mal_set_option": (C.c_int, [C.c_char_p, C.c_int]),
    "mal_stat": (C.c_uint64, [C.c_char_p]),
    "mal_debug_linear": (C.c_int, [C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_int64, C.c_void_p, C.c_int64,
                                   C.c_int32, C.c_void_p, C.c_int32, C.c_void_p, C.c_int64, C.c_void_p, C.c_int64,
                                   C.c_int32, C.c_void_p]),
    "mal_debug_reduce": (C.c_int, [C.c_int32, C.c_int32, C.c_int32, C.POINTER(RedProb), C.POINTER(Batch), C.c_int32,
                                   C.c_void_p]),
    "mal_debug_reduce_gru": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_int64] +
                             [C.c_void_p] * 7),
    "mal_debug_reduce_fc1": (C.c_int, [C.POINTER(Batch), C.c_int32, C.c_void_p, C.c_int64, C.c_int64, C.c_void_p,
                                       C.c_void_p, C.c_void_p]),
    "mal_debug_fc2_grad": (C.c_int, [C.POINTER(Batch), C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p,
                                     C.c_void_p]),
    "mal_agent_param_count":(C.c_int64, [C.c_int32, C.c_int32]),
    "mal_agent_param_count_kind": (C.c_int64, [C.c_int32, C.c_int32, C.c_int32]),
    "mal_dqn_step": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_int64,
                               C.c_void_p, C.c_int64, C.c_void_p, C.POINTER(Select), C.c_void_p]),
    "mal_mixer_param_count": (C.c_int64, [C.c_int32] * 5),
    "mal_learner_plan": (C.c_int, [C.POINTER(Batch), C.POINTER(LearnerCfg), C.POINTER(Plan)]),
    "mal_learner_forward": (C.c_int, [C.POINTER(Batch), C.POINTER(LearnerCfg), C.POINTER(Plan), C.c_void_p,
                                      C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "mal_learner_backward": (C.c_int, [C.POINTER(Batch), C.POINTER(LearnerCfg), C.POINTER(Plan), C.c_void_p,
                                       C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "mal_clip_rmsprop": (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_float,
                                   C.c_float, C.c_float, C.c_float, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]),
    "mal_peer_allreduce_clip_rmsprop": (C.c_int, [C.POINTER(C.c_void_p), C.c_int32, C.c_void_p, C.c_int64, C.c_void_p,
                                                  C.c_int64, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_float,
                                                  C.c_float, C.c_float, C.c_float, C.c_void_p, C.c_void_p, C.c_int64,
                                                  C.c_void_p]),
    "mal_learner_step": (C.c_int, [C.POINTER(Batch), C.POINTER(LearnerCfg), C.POINTER(Plan), C.c_void_p, C.c_void_p,
                                   C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "mal_learner_step_adam": (C.c_int, [C.POINTER(Batch), C.POINTER(LearnerCfg), C.POINTER(Plan), C.c_void_p, C.c_void_p,
                                        C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(AdamHyper), C.c_void_p,
                                        C.c_void_p]),
    "mal_clip_adam": (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p,
                                C.POINTER(AdamHyper), C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]),
    "mal_peer_allreduce_clip_adam": (C.c_int, [C.POINTER(C.c_void_p), C.c_int32, C.c_void_p, C.c_int64, C.c_void_p,
                                               C.c_int64, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p,
                                               C.POINTER(AdamHyper), C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]),
    "mal_clip_rmsprop_soft": (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_float,
                                        C.c_float, C.c_float, C.c_float, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64,
                                        C.POINTER(SoftTarget), C.c_void_p]),
    "mal_peer_allreduce_clip_rmsprop_soft": (C.c_int, [C.POINTER(C.c_void_p), C.c_int32, C.c_void_p, C.c_int64,
                                                       C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_int32,
                                                       C.c_void_p, C.c_float, C.c_float, C.c_float, C.c_float,
                                                       C.c_void_p, C.c_void_p, C.c_int64, C.POINTER(SoftTarget),
                                                       C.c_void_p]),
    "mal_clip_adam_soft": (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p,
                                     C.POINTER(AdamHyper), C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64,
                                     C.POINTER(SoftTarget), C.c_void_p]),
    "mal_peer_allreduce_clip_adam_soft": (C.c_int, [C.POINTER(C.c_void_p), C.c_int32, C.c_void_p, C.c_int64, C.c_void_p,
                                                    C.c_int64, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p,
                                                    C.POINTER(AdamHyper), C.c_void_p, C.c_void_p, C.c_int64,
                                                    C.POINTER(SoftTarget), C.c_void_p]),
    "mal_copy_f32": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]),
    "mal_agent_step": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_void_p,
                                 C.c_int64, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p,
                                 C.POINTER(Select), C.c_void_p]),
    "mal_rollout_step": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.POINTER(RolloutIO), C.c_void_p,
                                   C.c_void_p, C.c_void_p, C.POINTER(Select), C.c_void_p]),
    "mal_policy_schedule_bytes": (C.c_int64, [C.c_int32, C.c_int32, C.c_int32]),
    "mal_policy_schedule": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p]),
    "mal_agent_step_pool": (C.c_int, [C.c_void_p, C.c_int64, C.c_int32, C.c_void_p, C.c_int32, C.c_int32, C.c_int32,
                                      C.c_int32, C.c_int32, C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_void_p,
                                      C.c_void_p, C.c_void_p, C.POINTER(Select), C.c_void_p]),
    "mal_rollout_step_pool": (C.c_int, [C.c_void_p, C.c_int64, C.c_int32, C.c_void_p, C.c_int32, C.c_int32, C.c_int32,
                                        C.c_int32, C.POINTER(RolloutIO), C.c_void_p, C.c_void_p, C.c_void_p,
                                        C.POINTER(Select), C.c_void_p]),
    "mal_mixer_forward": (C.c_int, [C.c_int32] * 7 + [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int64,
                                                      C.c_void_p, C.c_void_p, C.c_void_p]),
    "mal_agent_step_backward_workspace": (C.c_int64, [C.c_int32] * 6),
    "mal_agent_step_backward": (C.c_int, [C.c_int32, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32,
                                          C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p,
                                          C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "mal_mixer_backward_workspace": (C.c_int64, [C.c_int32] * 7),
    "mal_mixer_backward": (C.c_int, [C.c_int32] * 7 + [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_void_p,
                                                       C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "mal_eps_greedy_select": (C.c_int, [C.c_void_p, C.c_int64, C.c_int32, C.c_int32, C.c_int32, C.POINTER(Select),
                                        C.c_void_p]),
    "mal_select_philox_advance": (C.c_int, [C.c_int32, C.c_int32, C.POINTER(C.c_uint64)]),
    "mal_record_copy": (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_int32,
                                  C.c_int64, C.c_void_p]),
    "mal_wire_layout": (C.c_int, [C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.POINTER(WireLayout)]),
    "mal_wire_pack": (C.c_int, [C.POINTER(Batch), C.c_void_p, C.POINTER(WireLayout), C.c_void_p, C.c_void_p]),
    "mal_wire_unpack": (C.c_int, [C.POINTER(Batch), C.c_void_p, C.POINTER(WireLayout), C.c_void_p]),
    "mal_per_sample_check": (C.c_int, [C.c_int64, C.c_int32, C.c_float]),
    "mal_per_sample": (C.c_int, [C.c_void_p, C.c_int64, C.c_int32, C.c_float, C.c_void_p, C.c_uint64, C.c_uint64,
                                 C.c_void_p, C.c_void_p, C.POINTER(C.c_uint64), C.c_void_p]),
    "mal_per_update_check": (C.c_int, [C.c_int32, C.c_int32, C.c_int32, C.c_float, C.c_float]),
    "mal_per_update": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_float, C.c_float,
                                 C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p]),
    "mal_max_t_filled": (C.c_int, [C.c_void_p, C.c_int64, C.c_int64, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p]),
}
EXPORTS = tuple(_PROTOS)

NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17", "--shared",
              "-Xcompiler", "-fPIC"]


def build(force: bool = False, verbose: bool = False) -> str:
    """Compile csrc/ into libmal_b200.so in-tree with nvcc for sm_100a (cross-compiles without a GPU)."""
    srcs = [os.path.join(_HERE, "csrc", f) for f in os.listdir(os.path.join(_HERE, "csrc"))]
    srcs.append(os.path.join(_HERE, "..", "include", "mal_b200.h"))
    if not force and os.path.exists(LIB_PATH) and all(os.path.getmtime(LIB_PATH) >= os.path.getmtime(s) for s in srcs):
        return LIB_PATH
    nvcc = os.environ.get("NVCC", "nvcc")
    cmd = [nvcc] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-o", LIB_PATH, SRC]
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        raise MalError("nvcc failed:\n%s\n%s" % (" ".join(cmd), res.stderr[-4000:]))
    if verbose:
        sys.stderr.write(res.stderr)
    return LIB_PATH


_lib = None


def lib():
    """The loaded shared library; raises (never falls back) when it is missing or has the wrong ABI."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise MalError("libmal_b200.so is not built (%s). Run `python -c 'import __graft_entry__ as g; "
                           "g.build()'` -- there is no CPU fallback." % LIB_PATH)
        L = C.CDLL(LIB_PATH)
        for name, (res, args) in _PROTOS.items():
            fn = getattr(L, name)
            fn.restype = res
            fn.argtypes = args
        if L.mal_version() != ABI_VERSION:
            raise MalError("libmal_b200.so ABI %d != expected %d; rebuild" % (L.mal_version(), ABI_VERSION))
        _lib = L
    return _lib


def profile_begin():
    check(lib().mal_profile_begin(), "mal_profile_begin")


def profile_end():
    """{kernel name: (launches, total_ms)} for everything launched since profile_begin()."""
    buf = C.create_string_buffer(1 << 16)
    check(lib().mal_profile_end(buf, len(buf)), "mal_profile_end")
    out = {}
    for line in buf.value.decode().splitlines():
        name, n, ms = line.rsplit(" ", 2)
        out[name] = (int(n), float(ms))
    return out


def profile_end_timeline():
    """[(kernel name, start_us, end_us)] per launch since profile_begin(), relative to the first launch."""
    buf = C.create_string_buffer(1 << 18)
    check(lib().mal_profile_end_timeline(buf, len(buf)), "mal_profile_end_timeline")
    out = []
    for line in buf.value.decode().splitlines():
        name, a, b = line.rsplit(" ", 2)
        out.append((name, float(a), float(b)))
    return out


def check(rc: int, what: str = ""):
    if rc != 0:
        raise MalError("%s failed (rc=%d): %s" % (what or "libmal_b200 call", rc, lib().mal_last_error().decode()))


# ---------------------------------------------------------------------------------------------------------
# torch <-> ABI helpers (torch is plumbing: device memory + current stream)
# ---------------------------------------------------------------------------------------------------------
def agent_input_flags(obs_last_action: bool, obs_agent_id: bool) -> int:
    """IN_* bits of the agent input [obs | one-hot(a_{t-1}) | one-hot(agent id)] (basic_controller.py:80-101)."""
    return (0 if obs_last_action else IN_NO_LAST_ACTION) | (0 if obs_agent_id else IN_NO_AGENT_ID)


def require_cuda(t, what="tensor"):
    if not t.is_cuda:
        raise MalError("%s must live on a CUDA device: the B200 path has no CPU fallback" % what)
    return t


def ptr(t):
    return C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p(0)


def current_stream(device=None):
    """Raw cudaStream_t of torch's current stream on `device` (torch is only the stream/memory plumbing)."""
    import torch
    if device is None:
        idx = torch.cuda.current_device()
    else:
        idx = device if isinstance(device, int) else torch.device(device).index
        if idx is None:
            idx = torch.cuda.current_device()
    try:
        return C.c_void_p(torch._C._cuda_getCurrentRawStream(idx))
    except AttributeError:   # older / newer torch without the private fast path
        return C.c_void_p(torch.cuda.current_stream(idx).cuda_stream)


class on_device:
    """`with on_device(dev):` -- like torch.cuda.device(dev) but free when `dev` is already current."""
    __slots__ = ("idx", "prev")

    def __init__(self, device):
        import torch
        self.idx = device if isinstance(device, int) else torch.device(device).index
        self.prev = None

    def __enter__(self):
        import torch
        cur = torch.cuda.current_device()
        if self.idx is not None and self.idx != cur:
            self.prev = cur
            torch.cuda.set_device(self.idx)

    def __exit__(self, *exc):
        if self.prev is not None:
            import torch
            torch.cuda.set_device(self.prev)
        return False


def field_of(t, inner_numel: int) -> Field:
    """Describe a [B, TT, *inner] tensor whose inner dims are contiguous (slices over B / TT are fine)."""
    if t.dim() < 2:
        raise MalError("field must have batch and time dims")
    expect = 1
    for size, stride in zip(reversed(t.shape[2:]), reversed(t.stride()[2:])):
        if size != 1 and stride != expect:
            raise MalError("inner dims of a scheme field must be contiguous")
        expect *= size
    if expect != inner_numel:
        raise MalError("scheme field has %d inner elements, expected %d" % (expect, inner_numel))
    return Field(t.data_ptr(), t.stride(0), t.stride(1))
