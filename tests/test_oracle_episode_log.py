"""The oracle's episode log (tests/oracle_episodes.py, the reference the device episode log is tested against): one record
per finished episode, in (step, env) order, consistent with the agent's counters."""
import numpy as np

import oracle
from oracle_episodes import EpisodeLoggingAgent


def _near_goal_agent(B=16, T=40, **kw):
    cfg = oracle.AgentConfig(map="easy", batch=B, order=2, max_options=3, seed=5, env_offset=100, epsilon=1.0,
                             max_episode_steps=7, option_timeout=5, **kw)
    ag = EpisodeLoggingAgent(cfg)
    tx, ty, _ = (float(v) for v in ag.map.target)
    rng = np.random.default_rng(1)
    S = ag.env.state.copy()
    S[: B // 2, 0] = tx + rng.uniform(-0.08, 0.0, B // 2)          # half of them next to the goal
    S[: B // 2, 1] = ty + rng.uniform(-0.04, 0.04, B // 2)
    S[: B // 2, 2:] = 0.0
    ag.env.reset(states=S)
    ag.start_xy = S[:, :2].copy()
    for _ in range(T):
        ag.step()
    return ag


def test_episode_log_matches_counters():
    B, T = 16, 40
    ag = _near_goal_agent(B, T)
    log = ag.episode_log()
    n = len(log["step"])
    assert n == int(ag.episodes.sum()) and n > B                  # every env finished several episodes (length <= 7)
    assert int(log["goal"].sum()) == int(ag.goals.sum()) > 0 and not log["goal"].all()
    assert log["step"].dtype == np.uint32 and log["env"].dtype == np.uint32
    assert log["ret"].dtype == np.float32 and log["length"].dtype == np.int32 and log["goal"].dtype == bool
    key = log["step"].astype(np.int64) * (1 << 32) + log["env"]
    assert np.all(np.diff(key) > 0)                                # (step, env) order, no duplicates
    assert log["env"].min() >= 100 and log["env"].max() < 100 + B
    assert np.all((log["length"] >= 1) & (log["length"] <= 7))
    assert np.all(log["length"][~log["goal"]] == 7)                # an episode that did not reach the goal timed out
    for b in range(B):
        mine = log["env"] == 100 + b
        assert int(mine.sum()) == int(ag.episodes[b])
        if mine.any():
            assert log["ret"][mine][-1] == np.float32(ag.last_return[b])
        # the recorded lengths plus the open episode's steps are every step this env has lived
        assert int(log["length"][mine].sum()) + int(ag.ep_steps[b]) == T
        # an episode ends at the step where its length runs out: the previous end + its length
        ends = log["step"][mine].astype(np.int64)
        starts = np.concatenate([[0], ends[:-1] + 1])
        assert np.array_equal(ends - starts + 1, log["length"][mine])


def test_episode_returns_are_exact_sums_of_step_rewards():
    ag = _near_goal_agent(8, 30)
    log = ag.episode_log()
    r = log["ret"].astype(np.float64)
    goal = log["goal"]
    # -1 per step (-5 on a collision), +10000 at the goal: integers, exact in float32
    assert np.all(r == np.round(r))
    assert np.all(r[goal] > 10000.0 - 5 * 7) and np.all(r[~goal] < 0)
    assert np.all(r[~goal] >= -5.0 * log["length"][~goal]) and np.all(r[~goal] <= -1.0 * log["length"][~goal])


def test_episode_log_empty_before_any_episode_ends():
    ag = EpisodeLoggingAgent(oracle.AgentConfig(map="easy", batch=4, order=2, max_options=2, seed=0))
    log = ag.episode_log()
    assert all(len(v) == 0 for v in log.values())
