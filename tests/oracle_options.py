"""Option log of the CPU oracle, for the tests of the device option log (AgentConfig.option_log).

OptionLoggingAgent is tests/oracle_episodes.EpisodeLoggingAgent (so one run yields both logs) with a record of every
option termination, read off the oracle's own state around each step: `env.step` is wrapped to keep s' before the env
reset, and `t_opt`, `ep_steps`, `option` and `start_xy` are copied before the step.  A termination of env b during step
t then has duration t_opt + 1, starts at start_xy[b], ends at s'[b, :2], and its outcome flags follow
oracle/agent.py SkillChainAgent.step items 3 and 6.  Within a step the records are in ascending env order, so the log is
in the (step, env) order the device's ring pass appends in.
"""
import numpy as np

from oracle_episodes import EpisodeLoggingAgent

OUTCOMES = ("hit", "label", "env_done", "option_timeout", "left", "episode_timeout")


class OptionLoggingAgent(EpisodeLoggingAgent):
    def __init__(self, cfg, pmap=None):
        super().__init__(cfg, pmap)
        self._opt_log = []
        self._s2 = None
        env_step = self.env.step

        def step_keeping_s2(a):
            out = env_step(a)
            self._s2 = np.array(out[0], dtype=np.float32, copy=True)
            return out

        self.env.step = step_keeping_s2

    def step(self, follow=None):
        cfg = self.cfg
        t, o, t_opt0, ep0, start = self.t, self.option.copy(), self.t_opt.copy(), self.ep_steps.copy(), self.start_xy.copy()
        out = super().step(follow)
        s2 = self._s2
        # initiation sets of s' as the step saw them (the classifiers only change in manage())
        in_own = ((self.initiation_bits(s2) >> o.astype(np.uint32)) & np.uint32(1)) != 0
        dur = t_opt0 + 1
        term, hit, done = out["term"], out["hit"], out["env_done"]
        flags = dict(hit=hit, label=hit & (dur <= cfg.init_horizon), env_done=done,
                     option_timeout=dur >= cfg.option_timeout, left=self.active[o] & ~in_own,
                     episode_timeout=(ep0 + 1 >= cfg.max_episode_steps) & ~done)
        for b in np.nonzero(term)[0]:
            self._opt_log.append((t, cfg.env_offset + int(b), int(o[b]), int(dur[b]),
                                  tuple(bool(flags[k][b]) for k in OUTCOMES), start[b].copy(), s2[b, :2].copy()))
        return out

    def option_log(self):
        """Every option termination so far, in (step, env) order: dict of NumPy arrays step, env (uint32), option,
        duration (int32), one bool array per outcome flag (OUTCOMES), start, end (float32 (n, 2))."""
        rec = self._opt_log
        out = dict(step=np.array([r[0] for r in rec], dtype=np.uint32),
                   env=np.array([r[1] for r in rec], dtype=np.uint32),
                   option=np.array([r[2] for r in rec], dtype=np.int32),
                   duration=np.array([r[3] for r in rec], dtype=np.int32))
        for i, k in enumerate(OUTCOMES):
            out[k] = np.array([r[4][i] for r in rec], dtype=bool)
        out["start"] = np.array([r[5] for r in rec], dtype=np.float32).reshape(-1, 2)
        out["end"] = np.array([r[6] for r in rec], dtype=np.float32).reshape(-1, 2)
        return out
