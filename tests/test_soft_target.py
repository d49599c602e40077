"""Soft target updates (`args.target_update_interval_or_tau`) on CPU: how QLearner resolves and validates the key, the
host-side control flow of train() in hard and soft mode (device calls stubbed), mal_learner_plan's rejection of a bad
target_tau, the C layout of the new struct and field, and the reference blend of tests/soft_target_ref.py against a
float64 evaluation."""
import ctypes as C
import math
import os
import subprocess
import tempfile

import numpy as np
import pytest
import torch as th

from tests import soft_target_ref as R
from tests.helpers import ROOT


@pytest.fixture(scope="module")
def nat():
    from ma_league_b200 import _native
    _native.build()
    return _native


def _cpu_system(**over):
    from tests.gpu_helpers import build_system
    return build_system(3, 9, 32, 48, 4, 6, "qmix", True, device="cpu", **over)


@pytest.mark.parametrize("value,want", [
    ("absent", ("hard", None, 0.0)),
    (None, ("hard", None, 0.0)),
    (200, ("hard", 200, 0.0)),
    (1.5, ("hard", 1.5, 0.0)),
    (1, ("soft", None, 1.0)),
    (0.01, ("soft", None, 0.01)),
    (np.float32(0.25), ("soft", None, 0.25)),
])
def test_key_resolution(nat, value, want):
    L = _cpu_system().learner
    if value != "absent":
        L.args.target_update_interval_or_tau = value
    assert L._target_update() == want
    assert L._cfg().target_tau == want[2]           # the cfg carries tau in double: fp32(1 - tau) is formed from it


@pytest.mark.parametrize("value", [0, 0.0, -0.1, -5, float("nan"), float("inf"), -float("inf"), True, False, "0.01",
                                   [0.01]])
def test_key_rejections(nat, value):
    L = _cpu_system().learner
    L.args.target_update_interval_or_tau = value
    with pytest.raises(nat.MalError, match="target_update_interval_or_tau"):
        L._target_update()
    with pytest.raises(nat.MalError, match="target_update_interval_or_tau"):
        L._cfg()                                    # _prepare builds the cfg before any launch


class _Stubbed:
    """train() with the device work stubbed out: what is left is the host logic that decides about target updates."""

    def __init__(self, nat, monkeypatch, **over):
        self.s = _cpu_system(**over)
        L = self.L = self.s.learner
        self.copies, self.cfgs = [], []
        n = sum(p.numel() for p in L.parameters())
        L._grad = th.zeros(n)
        L._grad_store = th.zeros(n + 8)

        def prepare(batch):
            cfg = L._cfg()
            self.cfgs.append(cfg)
            return nat.Batch(), cfg, {}
        monkeypatch.setattr(L, "_prepare", prepare)
        monkeypatch.setattr(L, "_step_graphed", lambda *a: True)
        monkeypatch.setattr(L, "_step_eager", lambda *a: None)
        monkeypatch.setattr(L, "scalars", lambda: th.zeros(64))
        monkeypatch.setattr(L, "update_targets", lambda: self.copies.append(True))

    def run(self, episodes):
        for i, ep in enumerate(episodes):
            self.L.train({"obs": th.zeros(1)}, t_env=i, episode_num=ep)


def test_train_with_only_the_new_key_in_both_modes(nat, monkeypatch):
    hard = _Stubbed(nat, monkeypatch, target_update_interval_or_tau=3)
    del hard.L.args.target_update_interval
    hard.run([0, 1, 2, 3, 4, 5, 7, 8, 10])
    assert len(hard.copies) == 3 and hard.L.last_target_update_episode == 10     # copies at 3, 7, 10
    assert all(c.target_tau == 0.0 for c in hard.cfgs)

    soft = _Stubbed(nat, monkeypatch, target_update_interval_or_tau=0.01)
    del soft.L.args.target_update_interval
    soft.run([0, 5, 500, 10 ** 6])
    assert soft.copies == [] and soft.L.last_target_update_episode == 0
    assert all(c.target_tau == 0.01 for c in soft.cfgs)


def test_legacy_key_unchanged(nat, monkeypatch):
    old = _Stubbed(nat, monkeypatch)                              # only target_update_interval = 200
    old.run([0, 100, 199, 200, 399, 400])
    assert len(old.copies) == 2 and old.L.last_target_update_episode == 400
    assert all(c.target_tau == 0.0 for c in old.cfgs)
    both = _Stubbed(nat, monkeypatch, target_update_interval_or_tau=None)
    both.run([0, 100, 199, 200, 399, 400])
    assert len(both.copies) == 2 and both.L.last_target_update_episode == 400


def test_neither_key_keeps_todays_error(nat, monkeypatch):
    st = _Stubbed(nat, monkeypatch)
    del st.L.args.target_update_interval
    with pytest.raises(AttributeError, match="target_update_interval"):
        st.run([0])
    assert len(st.cfgs) == 1 and st.L._cfg().target_tau == 0.0  # the step ran: only the interval check needs the key


def _cfg(nat, tau):
    cfg = nat.LearnerCfg(nat.MIXER_QMIX2, 1, 32, 64, 0.99, 5e-4, 0.99, 1e-5, 10.0, 0)
    cfg.target_tau = tau
    return cfg


def test_plan_rejects_bad_target_tau(nat):
    lib = nat.lib()
    b = nat.Batch(32, 201, 5, 11, 48, 80)
    plan, ref = nat.Plan(), nat.Plan()
    assert _cfg(nat, 0.0).target_tau == 0.0
    assert nat.LearnerCfg(nat.MIXER_QMIX2, 1, 32, 64, 0.99, 5e-4, 0.99, 1e-5, 10.0, 0).target_tau == 0.0   # zeroed tail
    assert lib.mal_learner_plan(C.byref(b), C.byref(_cfg(nat, 0.0)), C.byref(ref)) == 0
    for tau in (1e-6, 0.01, 0.5, 1.0):                           # no new workspace
        assert lib.mal_learner_plan(C.byref(b), C.byref(_cfg(nat, tau)), C.byref(plan)) == 0
        assert all(getattr(plan, n) == getattr(ref, n) for n in nat._PLAN_FIELDS)
    for tau in (-1e-9, -0.5, 1.0000001, 2.0, math.nan, math.inf, -math.inf):
        assert lib.mal_learner_plan(C.byref(b), C.byref(_cfg(nat, tau)), C.byref(plan)) != 0
        assert b"target_tau must be 0 (no soft target update) or a number in (0, 1]" in lib.mal_last_error()


def test_soft_entries_reject_before_any_launch(nat):
    """Host-side argument checks of the four *_soft entries: bad tau, missing targets.  Nothing is launched, so fake
    device pointers are enough."""
    lib = nat.lib()
    p = C.c_void_p(256)
    h = nat.AdamHyper(1e-3, 0.9, 0.999, 1e-8, 0.0, 10.0)
    peers = (C.c_void_p * 2)(256, 512)
    calls = {
        "mal_clip_rmsprop_soft": lambda s: lib.mal_clip_rmsprop_soft(p, 10, p, 10, p, p, 1e-3, 0.99, 1e-5, 10.0, p, p,
                                                                     None, 0, C.byref(s), None),
        "mal_clip_adam_soft": lambda s: lib.mal_clip_adam_soft(p, 10, p, 10, p, p, C.byref(h), p, p, None, 0,
                                                               C.byref(s), None),
        "mal_peer_allreduce_clip_rmsprop_soft": lambda s: lib.mal_peer_allreduce_clip_rmsprop_soft(
            peers, 2, p, 10, p, 10, p, p, 8, p, 1e-3, 0.99, 1e-5, 10.0, p, p, 0, C.byref(s), None),
        "mal_peer_allreduce_clip_adam_soft": lambda s: lib.mal_peer_allreduce_clip_adam_soft(
            peers, 2, p, 10, p, 10, p, p, 8, p, C.byref(h), p, p, 0, C.byref(s), None),
    }
    n0 = lib.mal_launch_count()
    for name, call in calls.items():
        for tau in (0.0, -0.1, 1.5, math.nan, math.inf):
            assert call(nat.SoftTarget(tau, 256, 512)) != 0
            assert (name + ": tau must be a number in (0, 1]").encode() in lib.mal_last_error()
        assert call(nat.SoftTarget(0.5, None, 512)) != 0
        assert (name + ": target buffer missing").encode() in lib.mal_last_error()
        assert call(nat.SoftTarget(0.5, 256, None)) != 0                 # n_mixer = 10 needs the target mixer
        assert (name + ": target buffer missing").encode() in lib.mal_last_error()
    assert lib.mal_clip_rmsprop_soft(p, 10, p, 10, p, p, 1e-3, 0.99, 1e-5, 10.0, p, p, None, 0, None, None) != 0
    assert lib.mal_launch_count() == n0


def test_soft_target_struct_matches_c(nat):
    prog = r'''
    #include <stdio.h>
    #include <stddef.h>
    #include "mal_b200.h"
    int main(void) { printf("%zu %zu %zu %zu %zu\n", sizeof(mal_soft_target_t), offsetof(mal_soft_target_t, target_agent),
        offsetof(mal_soft_target_t, target_mixer), offsetof(mal_learner_cfg_t, target_tau), sizeof(mal_learner_cfg_t));
        return 0; }'''
    with tempfile.TemporaryDirectory() as d:
        src = os.path.join(d, "s.c")
        open(src, "w").write(prog)
        exe = os.path.join(d, "s")
        subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), src, "-o", exe])
        got = [int(x) for x in subprocess.check_output([exe]).split()]
    assert got == [C.sizeof(nat.SoftTarget), nat.SoftTarget.target_agent.offset, nat.SoftTarget.target_mixer.offset,
                   nat.LearnerCfg.target_tau.offset, C.sizeof(nat.LearnerCfg)]


@pytest.mark.parametrize("tau", [0.005, 0.01, 0.3, 0.7, 1.0])
def test_reference_blend_against_float64(tau):
    rng = np.random.default_rng(int(tau * 1000))
    t = (rng.standard_normal(100003) * rng.choice([1e-3, 1.0, 1e3], 100003)).astype(np.float32)
    p = (t + rng.standard_normal(100003).astype(np.float32) * 0.1).astype(np.float32)
    got = R.blend_np(t, p, tau)
    tt = th.from_numpy(t.copy())
    R.blend_(tt, th.from_numpy(p), tau)
    assert np.array_equal(tt.numpy(), got)                      # torch fp32 and numpy fp32: the same three roundings
    exact = t.astype(np.float64) * (1.0 - tau) + p.astype(np.float64) * tau
    # c1, c2 and three operations each round once: |err| <= 4u (|t| (1 - tau) + |p| tau) with u = 2^-24
    bound = 4 * 2.0 ** -24 * (np.abs(t) * (1.0 - tau) + np.abs(p) * tau)
    assert np.all(np.abs(got.astype(np.float64) - exact) <= bound)
    if tau == 1.0:
        assert np.array_equal(got, p)                           # tau = 1 copies
