"""Episode log of the CPU oracle, for the tests of the device episode log (AgentConfig.episode_log).

EpisodeLoggingAgent is oracle.SkillChainAgent with a record of every finished episode, read off the oracle's own
bookkeeping around each step: an env whose `episodes` count rose during step t finished an episode there, with return
`last_return` (the oracle's running return before the reset), length `ep_steps` before the step + 1, and goal = its
`goals` count rose too (else the episode timed out).  Within a step the records are in ascending env order, so the log
is in the (step, env) order the device's ring pass appends in.
"""
import numpy as np

import oracle


class EpisodeLoggingAgent(oracle.SkillChainAgent):
    def __init__(self, cfg, pmap=None):
        super().__init__(cfg, pmap)
        self._ep_log = []

    def step(self, follow=None):
        t, ep0, goals0, len0 = self.t, self.episodes.copy(), self.goals.copy(), self.ep_steps.copy()
        out = super().step(follow)
        for b in np.nonzero(self.episodes > ep0)[0]:
            self._ep_log.append((t, self.cfg.env_offset + int(b), self.last_return[b], int(len0[b]) + 1,
                                 bool(self.goals[b] > goals0[b])))
        return out

    def episode_log(self):
        """Every finished episode so far, in (step, env) order: dict of NumPy arrays step (uint32, the agent step at
        which it ended), env (uint32, global env id), ret (float32, task return), length (int32, steps), goal (bool,
        False: timed out)."""
        rec = self._ep_log
        return dict(step=np.array([r[0] for r in rec], dtype=np.uint32),
                    env=np.array([r[1] for r in rec], dtype=np.uint32),
                    ret=np.array([r[2] for r in rec], dtype=np.float32),
                    length=np.array([r[3] for r in rec], dtype=np.int32),
                    goal=np.array([r[4] for r in rec], dtype=bool))
