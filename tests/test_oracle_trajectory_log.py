"""The oracle's trajectory log (tests/oracle_trajectories.py, the reference the device trajectory log is tested
against): one record per (step, tracked env), consistent with the oracle's option log and episode log for those envs."""
import numpy as np

import oracle
from oracle_trajectories import FLAGS, TrajectoryLoggingAgent

TRACKED = (0, 3, 4, 9, 15)


def _agent(B=16, T=60, manage_every=10, **kw):
    cfg = dict(map="easy", batch=B, order=2, max_options=3, seed=5, env_offset=100, epsilon=1.0,
               max_episode_steps=9, option_timeout=5, gestation_successes=3, example_capacity=1 << 12, init_horizon=3)
    cfg.update(kw)
    ag = TrajectoryLoggingAgent(oracle.AgentConfig(**cfg), trajectory_envs=TRACKED)
    tx, ty, _ = (float(v) for v in ag.map.target)
    rng = np.random.default_rng(1)
    S = ag.env.state.copy()
    S[: B // 2, 0] = tx + rng.uniform(-0.08, 0.0, B // 2)          # half of them next to the goal
    S[: B // 2, 1] = ty + rng.uniform(-0.04, 0.04, B // 2)
    S[: B // 2, 2:] = 0.0
    ag.env.reset(states=S)
    ag.start_xy = S[:, :2].copy()
    for t in range(T):
        ag.step()
        if (t + 1) % manage_every == 0:
            ag.manage()
    return ag


def _for_tracked(log):
    mine = np.isin(log["env"], np.array(TRACKED, dtype=np.uint32) + 100)
    return {k: v[mine] for k, v in log.items()}


def test_layout_and_every_flag():
    ag = _agent()
    tr = ag.trajectory_log()
    T, n = 60, len(TRACKED)
    assert len(tr["step"]) == T * n
    assert np.array_equal(tr["step"], np.repeat(np.arange(T, dtype=np.uint32), n))
    assert np.array_equal(tr["env"], np.tile(np.array(TRACKED, dtype=np.uint32) + 100, T))
    for k in FLAGS:
        assert tr[k].any() and not tr[k].all(), k
    assert not np.any(tr["label"] & ~tr["term"]) and not np.any(tr["episode_end"] & ~tr["term"])
    assert not np.any(tr["goal"] & ~tr["episode_end"])
    assert np.all((tr["action"] >= 0) & (tr["action"] < 5))


def test_terminations_equal_the_option_log():
    ag = _agent()
    tr, ol = ag.trajectory_log(), _for_tracked(ag.option_log())
    term = tr["term"]
    for k in ("step", "env", "option", "label"):
        assert np.array_equal(tr[k][term], ol[k]), k


def test_episode_ends_equal_the_episode_log():
    ag = _agent()
    tr, el = ag.trajectory_log(), _for_tracked(ag.episode_log())
    end = tr["episode_end"]
    assert np.array_equal(tr["step"][end], el["step"]) and np.array_equal(tr["env"][end], el["env"])
    assert np.array_equal(tr["goal"][end], el["goal"])


def test_first_state_of_an_execution_is_its_start():
    ag = _agent()
    tr, ol = ag.trajectory_log(), _for_tracked(ag.option_log())
    for b in np.array(TRACKED, dtype=np.uint32) + 100:
        mine = tr["env"] == b
        st, term = tr["state"][mine], tr["term"][mine]
        first = np.concatenate([[0], np.nonzero(term)[0] + 1])     # records that begin an execution
        ex = ol["env"] == b
        n = int(ex.sum())                                           # executions that have ended
        assert n == int(term.sum()) and n > 2
        assert np.array_equal(st[first[:n], :2], ol["start"][ex])
        # and an execution that did not end its episode ends where the next one begins
        cont = ~(ol["env_done"][ex] | ol["episode_timeout"][ex])
        nxt = first[1:n + 1]
        ok = nxt < len(st)
        assert np.array_equal(st[nxt[ok & cont], :2], ol["end"][ex][ok & cont])


def test_option_and_action_follow_the_agent():
    """The option of record t + 1 is the one the agent held after step t (action likewise), as the device records."""
    ag = _agent(T=0)
    tr_opt, tr_act = [], []
    for _ in range(30):
        tr_opt.append(ag.option[list(TRACKED)].copy())
        tr_act.append(ag.action[list(TRACKED)].copy())
        ag.step()
    tr = ag.trajectory_log()
    assert np.array_equal(tr["option"], np.concatenate(tr_opt)) and np.array_equal(tr["action"], np.concatenate(tr_act))
