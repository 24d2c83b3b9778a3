"""Trajectory log of the CPU oracle, for the tests of the device trajectory log (AgentConfig.trajectory_envs /
trajectory_log).

TrajectoryLoggingAgent is tests/oracle_options.OptionLoggingAgent (so one run yields all three logs) with a record of
every step of the tracked envs, read off the oracle's own state around each step: before step t it copies the state
s_t, the action and option taken there, t_opt and ep_steps; after it, the step's output gives term, hit, env_done and
the TD error.  The label is hit within init_horizon steps of the option's start (t_opt + 1 <= init_horizon), the
episode ends where env_done or the episode timed out, and goal is env_done.  Within a step the tracked envs are in
ascending order, so the log is in the (step, env) order the device gathers in.
"""
import numpy as np

from oracle_options import OptionLoggingAgent

FLAGS = ("term", "label", "episode_end", "goal")


class TrajectoryLoggingAgent(OptionLoggingAgent):
    def __init__(self, cfg, pmap=None, trajectory_envs=()):
        super().__init__(cfg, pmap)
        self.trajectory_envs = np.array(sorted(int(b) for b in trajectory_envs), dtype=np.int64)
        self._traj = []

    def step(self, follow=None):
        cfg, tr = self.cfg, self.trajectory_envs
        t = self.t
        s = np.array(self.env.state, dtype=np.float32, copy=True)
        a, o = self.action.copy(), self.option.copy()
        t_opt0, ep0 = self.t_opt.copy(), self.ep_steps.copy()
        out = super().step(follow)
        done, hit = out["env_done"], out["hit"]
        ep_timeout = (ep0 + 1 >= cfg.max_episode_steps) & ~done
        flags = dict(term=out["term"], label=hit & (t_opt0 + 1 <= cfg.init_horizon), episode_end=done | ep_timeout,
                     goal=done)
        delta = np.asarray(out["delta"], dtype=np.float32)
        for b in tr:
            self._traj.append((t, cfg.env_offset + int(b), s[b].copy(), int(a[b]), int(o[b]), delta[b],
                               tuple(bool(flags[k][b]) for k in FLAGS)))
        return out

    def trajectory_log(self):
        """Every step of the tracked envs so far, in (step, env) order: dict of NumPy arrays step, env (uint32), state
        (float32 (n, 4)), action, option (int32), delta (float32), one bool array per flag (FLAGS)."""
        rec = self._traj
        out = dict(step=np.array([r[0] for r in rec], dtype=np.uint32),
                   env=np.array([r[1] for r in rec], dtype=np.uint32),
                   state=np.array([r[2] for r in rec], dtype=np.float32).reshape(-1, 4),
                   action=np.array([r[3] for r in rec], dtype=np.int32),
                   option=np.array([r[4] for r in rec], dtype=np.int32),
                   delta=np.array([r[5] for r in rec], dtype=np.float32))
        for i, k in enumerate(FLAGS):
            out[k] = np.array([r[6][i] for r in rec], dtype=bool)
        return out
