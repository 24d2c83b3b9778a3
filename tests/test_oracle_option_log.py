"""The oracle's option log (tests/oracle_options.py, the reference the device option log is tested against): one record
per option termination, in (step, env) order, consistent with the agent's counters, its example rings and its episode
log."""
import numpy as np

import oracle
from oracle_options import OUTCOMES, OptionLoggingAgent


def _agent(B=16, T=60, manage_every=10, **kw):
    cfg = dict(map="easy", batch=B, order=2, max_options=3, seed=5, env_offset=100, epsilon=1.0,
               max_episode_steps=9, option_timeout=5, gestation_successes=3, example_capacity=1 << 12)
    cfg.update(kw)
    ag = OptionLoggingAgent(oracle.AgentConfig(**cfg))
    tx, ty, _ = (float(v) for v in ag.map.target)
    rng = np.random.default_rng(1)
    S = ag.env.state.copy()
    S[: B // 2, 0] = tx + rng.uniform(-0.08, 0.0, B // 2)          # half of them next to the goal
    S[: B // 2, 1] = ty + rng.uniform(-0.04, 0.04, B // 2)
    S[: B // 2, 2:] = 0.0
    ag.env.reset(states=S)
    ag.start_xy = S[:, :2].copy()
    counts = []
    for t in range(T):
        ag.step()
        if (t + 1) % manage_every == 0:
            ag.manage()
        counts.append((ag.n_success.copy(), ag.n_fail.copy()))
    return ag, counts


def test_option_log_matches_counters_and_example_rings():
    ag, counts = _agent()
    log = ag.option_log()
    n = len(log["step"])
    K = ag.options.K
    assert ag.n_active >= 1                                         # an option was promoted on the way
    key = log["step"].astype(np.int64) * (1 << 32) + log["env"]
    assert np.all(np.diff(key) > 0)                                 # (step, env) order, no duplicates
    assert np.all((log["env"] >= 100) & (log["env"] < 100 + 16))
    for k in range(K):
        mine = log["option"] == k
        # per option: the records are the rise of n_success + n_fail, the hit records the rise of n_success
        assert int(mine.sum()) == int(ag.n_success[k] + ag.n_fail[k])
        assert int((mine & log["hit"]).sum()) == int(ag.n_success[k])
        # and in order, their (start, label) are what the oracle appended to its example ring
        c = int(ag.ex_count[k])
        assert c == int(mine.sum()) <= ag.cfg.example_capacity
        assert np.array_equal(log["start"][mine], ag.ex_xy[k, :c])
        assert np.array_equal(log["label"][mine].astype(np.uint8), ag.ex_label[k, :c])
    # per step as well: the records of step t are the counters' rise during step t
    prev = (np.zeros(K, np.int64), np.zeros(K, np.int64))
    for t, (ns, nf) in enumerate(counts):
        at = log["step"] == t
        for k in range(K):
            assert int((at & (log["option"] == k)).sum()) == int(ns[k] - prev[0][k] + nf[k] - prev[1][k])
        prev = (ns, nf)
    assert n > 16 and log["hit"].any() and not log["hit"].all() and log["left"].any()


def test_option_log_outcomes():
    ag, _ = _agent()
    log = ag.option_log()
    cfg = ag.cfg
    dur = log["duration"]
    assert np.all((dur >= 1) & (dur <= cfg.option_timeout))
    assert np.array_equal(log["option_timeout"], dur >= cfg.option_timeout)
    assert np.array_equal(log["label"], log["hit"])                # init_horizon is unlimited here
    assert not np.any(log["env_done"] & log["episode_timeout"])
    # every record has a reason to stop, and every reason occurs
    reasons = np.stack([log[k] for k in OUTCOMES if k != "label"])
    assert reasons.any(axis=0).all()
    for k in OUTCOMES:
        assert log[k].any(), k
    # a termination of option 0 at the goal is a hit (its target is the goal)
    assert np.all(log["hit"][log["env_done"] & (log["option"] == 0)])
    # an execution starts where the previous one of the same env ended, unless the env was reset in between
    for b in range(100, 116):
        mine = np.nonzero(log["env"] == b)[0]
        for i, j in zip(mine[:-1], mine[1:]):
            if not (log["env_done"][i] or log["episode_timeout"][i]):
                assert np.array_equal(log["start"][j], log["end"][i])
                assert int(log["step"][j] - log["step"][i]) == int(log["duration"][j])


def test_label_respects_init_horizon():
    ag, _ = _agent(init_horizon=2)
    log = ag.option_log()
    assert np.array_equal(log["label"], log["hit"] & (log["duration"] <= 2))
    assert (log["hit"] & ~log["label"]).any()


def test_episode_ends_line_up_with_the_episode_log():
    ag, _ = _agent()
    log, eps = ag.option_log(), ag.episode_log()
    ended = log["env_done"] | log["episode_timeout"]
    assert np.array_equal(log["step"][ended], eps["step"]) and np.array_equal(log["env"][ended], eps["env"])
    assert np.array_equal(log["env_done"][ended], eps["goal"])
    assert np.array_equal(log["episode_timeout"][ended], ~eps["goal"])


def test_option_log_empty_before_any_termination():
    ag = OptionLoggingAgent(oracle.AgentConfig(map="easy", batch=4, order=2, max_options=2, seed=0))
    log = ag.option_log()
    assert all(len(v) == 0 for v in log.values())
