"""Per-match policies without a device: schedule sizing, argument checks of the pooled entries, pairing ids."""
import ctypes as C

import pytest
import torch as th


@pytest.fixture(scope="module")
def nat():
    from ma_league_b200 import _native
    _native.build()
    return _native


def test_schedule_bytes(nat):
    lib = nat.lib()
    # header of 16 ints + 16 ints per CTA; CTAs <= ceil(rows / 8) + min(K, bs) - 1
    assert lib.mal_policy_schedule_bytes(32, 5, 1) == 4 * (16 + 16 * 20)
    assert lib.mal_policy_schedule_bytes(32, 5, 8) == 4 * (16 + 16 * 27)
    assert lib.mal_policy_schedule_bytes(2, 5, 8) == 4 * (16 + 16 * 3)
    assert lib.mal_policy_schedule_bytes(4, 5, nat.MAX_POLICIES) == 4 * (16 + 16 * 6)
    for bad in [(0, 5, 1), (4, 0, 1), (4, 5, 0), (4, 5, nat.MAX_POLICIES + 1)]:
        assert lib.mal_policy_schedule_bytes(*bad) == -1
        assert lib.mal_last_error()
    assert b"n_policies" in (lib.mal_policy_schedule_bytes(4, 5, nat.MAX_POLICIES + 1), lib.mal_last_error())[1]


def test_pooled_entries_reject_bad_arguments_before_any_launch(nat):
    lib = nat.lib()
    fake = C.c_void_p(256)
    assert lib.mal_policy_schedule(fake, 4, 5, nat.MAX_POLICIES + 1, fake, None, None) != 0
    assert b"n_policies" in lib.mal_last_error()
    assert lib.mal_policy_schedule(None, 4, 5, 2, fake, None, None) != 0
    assert lib.mal_policy_schedule(fake, 4, 5, 2, C.c_void_p(260), None, None) != 0     # misaligned schedule
    sel = nat.Select()
    P = lib.mal_agent_param_count(48 + 11 + 5, 11)
    args = (20, 5, 48, 11, 0, fake, 240, fake, 55, None, fake, fake, C.byref(sel), None)
    assert lib.mal_agent_step_pool(fake, P, 0, fake, *args) != 0                          # no policies
    assert lib.mal_agent_step_pool(fake, P - 1, 2, fake, *args) != 0                      # rows shorter than the agent
    assert b"table_ld" in lib.mal_last_error()
    assert lib.mal_agent_step_pool(fake, P, 2, fake, 21, *args[1:]) != 0                  # rows not a multiple of N
    assert lib.mal_agent_step_pool(fake, P, 2, None, *args) != 0
    io = nat.RolloutIO()
    assert lib.mal_rollout_step_pool(fake, P, 2, fake, 4, 5, 48, 11, C.byref(io), None, fake, fake, C.byref(sel), None) != 0
    assert b"mal_rollout_step_pool" in lib.mal_last_error()


def test_pairing_ids():
    from ma_league_b200.league.cross_play import pairing_ids
    i, j = pairing_ids(3, 2)
    assert i.tolist() == [0] * 6 + [1] * 6 + [2] * 6
    assert j.tolist() == [0, 0, 1, 1, 2, 2] * 3


def test_set_match_policies_rejects_a_host_table(nat):
    import ma_league_b200 as M
    from ma_league_b200.synthetic import make_args, make_scheme
    args = make_args(3, 9, 48, mixer="vdn", device="cpu")
    scheme, groups, pre = make_scheme(3, 9, 32, 48)
    buf_scheme = M.EpisodeBatch(scheme, groups, 1, 2, preprocess=pre, device="cpu").scheme
    mac = M.BasicMAC(buf_scheme, groups, args)
    with pytest.raises(nat.MalError):
        mac.set_match_policies(th.zeros(2, 10), [0, 1])
    mac.set_match_policies(None)
    assert mac.match_policies is None
