"""The C-ABI library loads without a GPU and exports exactly what include/mal_b200.h declares."""
import ctypes as C
import os
import re
import subprocess
import tempfile

import pytest

from tests.helpers import ROOT

HEADER = os.path.join(ROOT, "include", "mal_b200.h")


@pytest.fixture(scope="module")
def nat():
    from ma_league_b200 import _native
    _native.build()
    return _native


def declared_functions():
    src = open(HEADER).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(mal_[a-z0-9_]+)\s*\(", src)))


def test_header_functions_are_exported(nat):
    lib = nat.lib()
    names = declared_functions()
    assert len(names) >= 15
    for n in names:
        assert hasattr(lib, n), "libmal_b200.so does not export %s" % n
    assert sorted(nat.EXPORTS) == names, "ctypes prototypes and header disagree"
    assert lib.mal_version() == nat.ABI_VERSION


def test_struct_sizes_match_c(nat):
    prog = r'''
    #include <stdio.h>
    #include "mal_b200.h"
    int main(void) { printf("%zu %zu %zu %zu %zu %zu\n", sizeof(mal_field_t), sizeof(mal_batch_t),
        sizeof(mal_learner_cfg_t), sizeof(mal_plan_t), sizeof(mal_select_t), sizeof(mal_red_prob_t)); return 0; }'''
    with tempfile.TemporaryDirectory() as d:
        src = os.path.join(d, "s.c")
        open(src, "w").write(prog)
        exe = os.path.join(d, "s")
        subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), src, "-o", exe])
        sizes = [int(x) for x in subprocess.check_output([exe]).split()]
    assert sizes == [C.sizeof(nat.Field), C.sizeof(nat.Batch), C.sizeof(nat.LearnerCfg), C.sizeof(nat.Plan),
                     C.sizeof(nat.Select), C.sizeof(nat.RedProb)]


def test_param_counts_match_survey_table(nat):
    lib = nat.lib()
    # SURVEY.md section 8 config table: (N, agent params, qmix params)
    for N, n_agent, n_mixer in [(3, 28425, 17761), (5, 29835, 28065), (10, 33360, 53825), (20, 40410, 105345)]:
        A, OBS, S = 6 + N, 8 + 8 * N, 16 * N
        assert lib.mal_agent_param_count(OBS + A + N, A) == n_agent
        assert lib.mal_mixer_param_count(nat.MIXER_QMIX2, S, N, 32, 64) == n_mixer
    assert lib.mal_mixer_param_count(nat.MIXER_VDN, 80, 5, 32, 64) == 0


def test_plan_without_gpu_and_argument_errors(nat):
    lib = nat.lib()
    b = nat.Batch(32, 201, 5, 11, 48, 80)
    cfg = nat.LearnerCfg(nat.MIXER_QMIX2, 1, 32, 64, 0.99, 5e-4, 0.99, 1e-5, 10.0, 0)
    plan = nat.Plan()
    assert lib.mal_learner_plan(C.byref(b), C.byref(cfg), C.byref(plan)) == 0
    assert plan.n_agent_params == 29835 and plan.n_mixer_params == 28065
    offs = [getattr(plan, n) for n in nat._PLAN_FIELDS if n not in ("total_bytes", "n_agent_params", "n_mixer_params",
                                                                     "partials_bytes")]
    assert all(0 <= o < plan.total_bytes and o % 256 == 0 for o in offs)
    bad = nat.LearnerCfg(7, 1, 32, 64, 0.99, 5e-4, 0.99, 1e-5, 10.0, 0)
    assert lib.mal_learner_plan(C.byref(b), C.byref(bad), C.byref(plan)) != 0
    assert b"not recognised" in lib.mal_last_error()          # q_learner.py:24
    b2 = nat.Batch(32, 201, 5, 40, 48, 80)
    assert lib.mal_learner_plan(C.byref(b2), C.byref(cfg), C.byref(plan)) != 0
    # misaligned record copy is rejected before any launch
    assert lib.mal_record_copy(C.c_void_p(16), 24, None, C.c_void_p(32), 16, None, 1, 16, None) != 0


def test_missing_library_fails_loudly(nat, monkeypatch):
    monkeypatch.setattr(nat, "_lib", None)
    monkeypatch.setattr(nat, "LIB_PATH", "/nonexistent/libmal_b200.so")
    with pytest.raises(nat.MalError):
        nat.lib()
