"""Cross-play of a population in one batched rollout: every ordered pairing (i, j) of K agents, home = agent i against
away = agent j, `reps` times, as K*K*reps lock-step matches of one two-team `BatchedEpisodeStepper` run.  Both controllers
play per-match policies from the same [K, P] table (`BasicMAC.set_match_policies`), so the run costs one launch per team
and timestep whatever K is.  This is the data the reference's JPC evaluation plays (runs/evaluation/jpc_eval_run.py,
eval/methods.py) pairing by pairing; metrics over the returned matrix stay the caller's.
"""
import torch as th


def pairing_ids(K, reps, device=None):
    """(home ids, away ids) of the K*K*reps matches: match (i*K + j)*reps + r plays agent i at home against agent j."""
    i = th.arange(K, device=device).repeat_interleave(K * reps)
    j = th.arange(K, device=device).repeat_interleave(reps).repeat(K)
    return i, j


def cross_play_returns(stepper, home_mac, away_mac, table, reps=1, test_mode=True, draws=None):
    """[K, K] mean home return of agent i (home) against agent j (away), over `reps` matches each.

    `stepper` is an initialised two-team `BatchedEpisodeStepper` whose environment runs K*K*reps matches; `home_mac` /
    `away_mac` become its controllers.  `table` is the [K, P] float32 CUDA table of flat agent buffers (e.g.
    `DeviceAgentPool.pool`).  Both controllers play their own agents again afterwards.  `draws` is passed to
    `stepper.run` (injected random draws, for tests)."""
    K = table.shape[0]
    n = K * K * reps
    if stepper.n_teams != 2:
        raise ValueError("cross-play needs a two-team environment")
    if stepper.batch_size != n:
        raise ValueError("cross-play of %d agents x %d repetitions needs %d matches, the environment runs %d"
                         % (K, reps, n, stepper.batch_size))
    home_ids, away_ids = pairing_ids(K, reps)
    stepper.home_mac, stepper.away_mac = home_mac, away_mac
    try:
        home_mac.set_match_policies(table, home_ids)
        away_mac.set_match_policies(table, away_ids)
        out = stepper.run(test_mode=test_mode, draws=draws)
    finally:
        home_mac.set_match_policies(None)
        away_mac.set_match_policies(None)
    returns = out[-1]["episode_returns"][0]
    return returns.view(K, K, reps).mean(dim=2)
