"""Occupancy grid of the CPU oracle, for the tests of the device occupancy grid (AgentConfig.occupancy_grid).

The definition, written down once here:
- Every agent step t of every local env b is counted, once.
- Step t of env b adds 1 to counts[o_t][iy][ix]: o_t is the option running during step t (the option field of the step
  record; the oracle's `option` before the step) and (ix, iy) the cell of the state s_t at which the step began (the
  record's x, y; the oracle's `env.state` before the step, the state trajectories() reports).
- The cell along x is i = min(max(int(fp32(x) * G), 0), G - 1), the conversion truncating toward zero; iy likewise
  from y.  G is a power of two in 1..128, so fp32(x) * G is exact and the device and this helper agree without any
  rounding question.
- Counts are uint64 and cumulative from the agent's construction.  Slots 0..K-1 are counted, the gestating one
  included; the top-level learner's weight slots are not options and have no grid.

OccupancyAgent is tests/oracle_trajectories.TrajectoryLoggingAgent (so one oracle run yields every log) that applies
this before every step() from its own state and option.
"""
import numpy as np

from oracle_trajectories import TrajectoryLoggingAgent


def cells(v, grid):
    """Cell index along one axis of the fp32 coordinates `v` on a `grid` x `grid` map (int64 array)."""
    i = (np.asarray(v, dtype=np.float32) * np.float32(grid)).astype(np.int64)     # truncates toward zero
    return np.clip(i, 0, grid - 1)


class OccupancyAgent(TrajectoryLoggingAgent):
    def __init__(self, cfg, pmap=None, trajectory_envs=(), grid=64):
        super().__init__(cfg, pmap, trajectory_envs)
        self.grid = int(grid)
        self.counts = np.zeros((cfg.max_options, self.grid, self.grid), dtype=np.uint64)

    def step(self, follow=None):
        s = np.asarray(self.env.state, dtype=np.float32)
        np.add.at(self.counts, (np.asarray(self.option, dtype=np.int64), cells(s[:, 1], self.grid),
                                cells(s[:, 0], self.grid)), np.uint64(1))
        return super().step(follow)
