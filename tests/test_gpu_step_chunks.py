"""The Pinball step tests several substeps per walk of a cell's candidate edges (`pinball_step`, csrc/scg_step.cuh).

Its results must stay the oracle's bit for bit.  The sample below is built so that it contains every case where the
chunked walk could part from the one-substep-at-a-time loop, and the coverage is checked on the oracle's own
trajectories (a replay of `step_batched` that records every substep), not assumed:
  * a first collision at every substep index 0-19, including a single hit on the last substep (the extra move);
  * a bounce and a goal entry within one chunk of substeps (and on the same substep);
  * a ball that changes broad-phase cell between two substeps, at every grid resolution tested;
  * a double hit (velocity reversal);
  * a ball leaving the unit square (the all-edges path).
"""
import numpy as np
import pytest

import oracle
from oracle.pinball import N_SUBSTEPS, step_batched, f32

CHUNK = 4          # kStepChunk in csrc/scg_step.cuh
GRIDS = [8, 64, 128]

# a map whose wall passes through the goal's neighbourhood, so that a bounce and a goal entry can be a few substeps
# apart (on the shipped maps the goal is 0.03 from any contact position, 20 or more substeps)
GOAL_WALL = dict(ball_r=0.02, target=(0.5, 0.5, 0.04), starts=[(0.2, 0.2)],
                 polygons=[[(0.3, 0.555), (0.7, 0.555), (0.7, 0.6), (0.3, 0.6)],
                           [(0.56, 0.3), (0.6, 0.3), (0.6, 0.45), (0.56, 0.45)]])


def _omap(name):
    if name == "goal_wall":
        return oracle.PinballMap(**GOAL_WALL)
    return oracle.PinballMap.from_name(name)


def _gmap(scg, name, grid_n):
    if name == "goal_wall":
        return scg.PinballMap(**GOAL_WALL, grid_n=grid_n)
    return scg.PinballMap.from_name(name, grid_n=grid_n)


def _sample(omap, n, seed):
    """Balls near random edges at random speeds (collisions at every substep), near the goal, and near and outside
    the border of the unit square, with random actions."""
    rng = np.random.default_rng(seed)
    parts = []
    m = n // 2          # near walls: within 2.5 radii of a random point of a random edge
    e = omap.edges[rng.integers(0, omap.n_edges, m)]
    t = rng.uniform(0, 1, m).astype(np.float32)
    off = rng.uniform(-2.5, 2.5, m).astype(np.float32) * omap.ball_r
    parts.append(np.stack([e[:, 0] + t * e[:, 2] + off * e[:, 5], e[:, 1] + t * e[:, 3] + off * e[:, 6],
                           rng.uniform(-1, 1, m), rng.uniform(-1, 1, m)], axis=1))
    m = n // 4          # around the goal, up to 0.03 outside it
    tx, ty, tr = (float(v) for v in omap.target)
    ang = rng.uniform(0, 2 * np.pi, m)
    rad = tr + rng.uniform(-0.01, 0.03, m)
    parts.append(np.stack([tx + rad * np.cos(ang), ty + rad * np.sin(ang),
                           rng.uniform(-1, 1, m), rng.uniform(-1, 1, m)], axis=1))
    m = n - len(parts[0]) - len(parts[1])      # near or beyond the border of the unit square, fast
    side = rng.integers(0, 4, m)
    u = rng.uniform(0, 1, m)
    d = rng.uniform(-0.03, 0.01, m)            # d > 0: already outside
    x = np.where(side == 0, -d, np.where(side == 1, 1 + d, u))
    y = np.where(side == 2, -d, np.where(side == 3, 1 + d, u))
    parts.append(np.stack([x, y, rng.uniform(-1, 1, m), rng.uniform(-1, 1, m)], axis=1))
    S = np.concatenate(parts).astype(np.float32)
    A = rng.integers(0, 5, len(S)).astype(np.int32)
    return S, A


def _replay(omap, S, A):
    """`step_batched`'s operations for every env and substep, recording the substep's position after the move, its
    hit count and its goal test; also returns the next states, which must be `step_batched`'s."""
    x, y, vx, vy = (S[:, i].copy() for i in range(4))
    one = f32(1.0)
    imp = f32(1.0) / f32(5.0)
    vx = np.where(A == 0, np.clip(vx + imp, -one, one), vx)
    vy = np.where(A == 1, np.clip(vy + imp, -one, one), vy)
    vx = np.where(A == 2, np.clip(vx - imp, -one, one), vx)
    vy = np.where(A == 3, np.clip(vy - imp, -one, one), vy)
    E = omap.edges
    X1, Y1, DX, DY, INV = (E[None, :, i] for i in range(5))
    tx, ty, _ = omap.target
    n = len(S)
    pos = np.zeros((n, N_SUBSTEPS, 2), np.float32)
    nhit = np.zeros((n, N_SUBSTEPS), np.int32)
    goal = np.zeros((n, N_SUBSTEPS), bool)
    live = np.ones((n, N_SUBSTEPS), bool)
    alive = np.ones(n, bool)
    for i in range(N_SUBSTEPS):
        live[:, i] = alive
        px = x + vx * omap.h
        py = y + vy * omap.h
        t = np.minimum(np.maximum(((px[:, None] - X1) * DX + (py[:, None] - Y1) * DY) * INV, f32(0)), f32(1))
        ex = (X1 + t * DX) - px[:, None]
        ey = (Y1 + t * DY) - py[:, None]
        hit = ((ex * ex + ey * ey) <= omap.r2) & ((ex * vx[:, None] + ey * vy[:, None]) > 0)
        nh = hit.sum(axis=1)
        first = hit.argmax(axis=1)
        nx, ny = E[first, 5], E[first, 6]
        k = f32(2.0) * (vx * nx + vy * ny)
        qx = np.where(nh == 1, vx - k * nx, np.where(nh >= 2, -vx, vx))
        qy = np.where(nh == 1, vy - k * ny, np.where(nh >= 2, -vy, vy))
        if i == N_SUBSTEPS - 1:
            px = np.where(nh == 1, px + qx * omap.h, px)
            py = np.where(nh == 1, py + qy * omap.h, py)
        g = ((px - tx) * (px - tx) + (py - ty) * (py - ty)) < omap.tr2
        pos[:, i, 0], pos[:, i, 1] = px, py
        nhit[:, i] = np.where(alive, nh, 0)
        goal[:, i] = alive & g
        x, y, vx, vy = (np.where(alive, a, b) for a, b in ((px, x), (py, y), (qx, vx), (qy, vy)))
        alive &= ~g
    return pos, nhit, goal, live, np.stack([x, y], axis=1)


def _coverage(omap, S, A, grids):
    pos, nhit, goal, live, xy = _replay(omap, S, A)
    ons = step_batched(omap, S, A)[0]
    done = goal.any(axis=1)
    # the replay is the oracle's trajectory: the same end positions (after the bounds clamp of the envs still running)
    for i, (lo, hi) in enumerate(((f32(0.05), f32(0.95)),) * 2):
        xy[:, i] = np.where(~done & (xy[:, i] > 1), hi, xy[:, i])
        xy[:, i] = np.where(~done & (xy[:, i] < 0), lo, xy[:, i])
    assert np.array_equal(xy.view(np.uint32), ons[:, :2].view(np.uint32))
    cov = {}
    any_hit = nhit > 0
    has = any_hit.any(axis=1)
    first = np.where(has, any_hit.argmax(axis=1), -1)
    cov["first_hit_at"] = set(first[has].tolist())
    cov["single_hit_last_substep"] = bool((nhit[:, N_SUBSTEPS - 1] == 1).any())
    cov["double_hit"] = bool((nhit >= 2).any())
    g_at = np.where(done, goal.argmax(axis=1), -1)
    same, near = False, False
    for s in range(N_SUBSTEPS):
        hs = any_hit[:, s] & done
        same |= bool((hs & (g_at == s)).any())
        near |= bool((hs & (g_at > s) & (g_at < s + CHUNK)).any())
    cov["hit_and_goal_same_substep"] = same
    cov["hit_then_goal_within_chunk"] = near
    for G in grids:
        c = np.floor(pos * G).astype(np.int64)
        moved = (c[:, 1:] != c[:, :-1]).any(axis=2) & live[:, 1:] & ~any_hit[:, :-1]
        cov[f"cell_change_G{G}"] = bool(moved.any())
    inside = ((S[:, 0] >= 0) & (S[:, 0] < 1) & (S[:, 1] >= 0) & (S[:, 1] < 1))[:, None]
    out = ((pos < 0) | (pos >= 1)).any(axis=2) & live
    cov["leaves_unit_square"] = bool((out & inside).any())
    return cov


def _check_coverage(cov, need_goal_chunk):
    assert cov["first_hit_at"] == set(range(N_SUBSTEPS)), sorted(cov["first_hit_at"])
    assert cov["single_hit_last_substep"] and cov["double_hit"] and cov["leaves_unit_square"], cov
    assert all(v for k, v in cov.items() if k.startswith("cell_change")), cov
    if need_goal_chunk:
        assert cov["hit_and_goal_same_substep"] and cov["hit_then_goal_within_chunk"], cov


N = 30000


def test_sample_covers_the_chunk_cases():
    """CPU-only: the sample the GPU tests use contains every case the chunked walk must get right."""
    for name, seed in (("easy", 1), ("hard", 2), ("goal_wall", 3)):
        omap = _omap(name)
        S, A = _sample(omap, N, seed)
        _check_coverage(_coverage(omap, S, A, GRIDS), need_goal_chunk=name == "goal_wall")


@pytest.fixture(scope="module")
def scg():
    import skill_chaining_with_graphs_b200 as m
    m.load_library()
    return m


@pytest.mark.gpu
@pytest.mark.parametrize("cull", [True, False])
@pytest.mark.parametrize("grid_n", GRIDS)
@pytest.mark.parametrize("name,seed", [("easy", 1), ("hard", 2), ("goal_wall", 3)])
def test_step_chunks_bit_exact(scg, name, seed, grid_n, cull):
    import torch
    omap = _omap(name)
    S, A = _sample(omap, N, seed)
    gmap = _gmap(scg, name, grid_n)
    env = scg.PinballEnv(gmap, len(S), cull=cull)
    env.reset(states=S)
    ns, r, done, hit = env.step(torch.as_tensor(A).cuda())
    ons, orr, ofl = step_batched(omap, S, A)
    assert np.array_equal(ns.cpu().numpy().view(np.uint32), ons.view(np.uint32))
    assert np.array_equal(r.cpu().numpy().view(np.uint32), orr.view(np.uint32))
    assert np.array_equal(env.flags.cpu().numpy(), ofl)
