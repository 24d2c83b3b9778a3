"""The device occupancy grid (AgentConfig.occupancy_grid): every env-step of every env counted by the option running
during it and the cell of the state at which it began, against the oracle's counts (tests/oracle_occupancy.py).  Counts
are integers added atomically, so every comparison here is equality."""
import ctypes as C

import numpy as np
import pytest

import oracle
from oracle_occupancy import OccupancyAgent, cells
from oracle_replay import activate

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def scg():
    import skill_chaining_with_graphs_b200 as m
    m.load_library()
    return m


@pytest.fixture(scope="module")
def torch():
    import torch as t
    return t


THETA = np.array([[-1.0, 2.0, 0.0, 0.0, 0.0, 0.0],      # option 0: x >= 0.5
                  [-0.6, 0.0, 2.0, 0.0, 0.0, 0.0]],     # option 1: y >= 0.3
                 dtype=np.float32)
GPU_ONLY = ("window", "event_history", "deterministic")


def _pair(scg, torch, B, K, seed, grid, active=2, oracle_side=True, **kw):
    """Oracle (or None) and GPU agents on the same start states (a quarter of them next to the goal) and weights, with
    the first `active` options active (fixed classifiers, chain parents); the grid is a GPU-only setting."""
    name = "easy"
    omap, gmap = oracle.PinballMap.from_name(name), scg.PinballMap.from_name(name)
    cfg = dict(map=name, batch=B, order=2, max_options=K, seed=seed, **kw)
    rng = np.random.default_rng(seed)
    S = omap.sample_free_states(rng, B)
    tx, ty, _ = omap.target
    n = B // 4
    S[:n, 0] = tx + rng.uniform(-0.1, 0.0, n)
    S[:n, 1] = ty + rng.uniform(-0.05, 0.05, n)
    S[:n, 2:] = 0.0
    gag = scg.SkillChainAgent(scg.AgentConfig(occupancy_grid=grid, **cfg), gmap, initial_states=S)
    W = (rng.standard_normal(tuple(gag.options.W.shape)) * 0.3).astype(np.float32)
    gag.options.set_weights(W)
    A = rng.integers(0, 5, B).astype(np.int32)
    theta = np.zeros((K, 6), dtype=np.float32)
    theta[:active] = THETA[:active]
    if active:
        gag.options.theta.copy_(torch.as_tensor(theta))
        gag.active_mask, gag.n_active = (1 << active) - 1, active
        for j in range(1, active + 1):
            gag.parents_host[j] = 1 << (j - 1)
        gag._push_parents()
    gag.action.copy_(torch.as_tensor(A))
    gag.invalidate()
    if not oracle_side:
        return None, gag
    oag = OccupancyAgent(oracle.AgentConfig(**{k: v for k, v in cfg.items() if k not in GPU_ONLY}), omap,
                         grid=max(grid, 1))
    oag.env.reset(states=S)
    oag.start_xy = oag.env.state[:, :2].copy()
    oag.opt_s0 = oag.env.state.copy()
    oag.options.W[:] = W
    if active:
        activate(oag, theta, active)
    oag.action = A.copy()
    return oag, gag


def _check(got, want, B, t, what):
    assert got["counts"].dtype == np.uint64 and got["counts"].shape == want.shape, what
    assert got["env_steps"] == B * t == int(want.sum()), f"{what}: {got['env_steps']} env-steps counted, expected {B * t}"
    bad = np.argwhere(got["counts"] != want)
    assert bad.size == 0, f"{what}: {len(bad)} cells differ, first [option, iy, ix] = {bad[:5].tolist()}"


CHUNKS = (5, 11, 1, 8, 24, 3, 29)


@pytest.mark.parametrize("window,top_level,B,G,K", [
    (1, False, 257, 16, 4), (8, False, 1000, 64, 4), (1, True, 1000, 128, 4), (8, True, 257, 1, 4),
    (8, False, 257, 128, 16), (1, False, 1000, 64, 16), (8, True, 1000, 16, 13)])
def test_occupancy_matches_oracle(scg, torch, window, top_level, B, G, K):
    """epsilon = 1 (and epsilon_top = 1): both agents follow identical trajectories, with two active options.  Read after
    chunks of uneven length, so most reads fall inside an open window (the read counts that window's first steps, the
    flush the rest): the device counts equal the oracle's after every chunk."""
    kw = dict(sync_interval=8, option_timeout=6, epsilon=1.0, epsilon_top=1.0, alpha=1e-3, max_episode_steps=14,
              gestation_successes=10 ** 9, window=window, event_history=16, top_level=top_level, init_horizon=3)
    oag, gag = _pair(scg, torch, B, K, 41, G, **kw)
    for i, n in enumerate(CHUNKS):
        gag.run(n)
        for _ in range(n):
            oag.step()
        if i % 2:
            gag.manage()
        got = gag.occupancy()
        assert got["grid"] == G
        _check(got, oag.counts, B, gag.t, f"chunk {i}")
    assert (oag.counts.reshape(K, -1).sum(axis=1) > 0).sum() >= 3       # the active options and the gestating one ran


def _gpu_window(gag, torch, n):
    """n free-running GPU steps in one call; the (action, option) each env held before every step and after the last."""
    wl0 = int(gag._struct.win_len)
    gag.run(n)
    torch.cuda.synchronize()
    meta = gag.win_rec[wl0:wl0 + n, :, 5].cpu().numpy().view(np.uint32)
    acts = np.concatenate([(meta & 7).astype(np.int32), gag.action.cpu().numpy()[None]])
    opts = np.concatenate([((meta >> 8) & 0xFF).astype(np.int32), gag.option.cpu().numpy()[None]])
    return acts, opts


def test_occupancy_with_learning_matches_oracle_follow(scg, torch):
    """Learning on (alpha > 0, epsilon = 0.05): the GPU agent runs free for 3 windows with its weight syncs, the oracle
    follows its choices (oracle/agent.py step(follow=)), and the counts are equal after every window."""
    B, K, G = 1000, 4, 64
    kw = dict(sync_interval=8, window=8, option_timeout=6, epsilon=0.05, alpha=5e-3, max_episode_steps=20,
              gestation_successes=10 ** 9)
    oag, gag = _pair(scg, torch, B, K, 17, G, **kw)
    W0 = gag.options.W.clone()
    for w in range(3):
        acts, opts = _gpu_window(gag, torch, 8)
        for t in range(8):
            assert np.array_equal(oag.option, opts[t]), f"window {w} step {t}: option before the step"
            oag.step(follow=dict(action=acts[t + 1], option=opts[t + 1]))
        assert np.array_equal(gag.state.cpu().numpy().view(np.uint32), oag.env.state.view(np.uint32))
        _check(gag.occupancy(), oag.counts, B, gag.t, f"window {w}")
    assert not torch.equal(gag.options.W, W0)             # it learned


def _learning_state(gag, torch):
    o = gag.options
    gag.flush()
    torch.cuda.synchronize()
    return dict(W=o.W.clone(), trace=o._trace.clone(), dW=o._dW.clone(), cnt=o._cnt.clone(), s=gag.s.clone(),
                action=gag.action.clone(), option=gag.option.clone(), ex_xy=gag.ex_xy.clone(),
                ex_label=gag.ex_label.clone(), ex_count=gag.ex_count.clone(), theta=o.theta.clone())


def test_reading_changes_nothing(scg, torch):
    """deterministic=True: the grid off, on and never read, and on and read after every chunk (mostly inside an open
    window) - W, traces, dW, the example rings, the controller and the state are bit-identical; the two grids too."""
    B, K = 2048, 3
    kw = dict(sync_interval=8, window=8, option_timeout=6, epsilon=0.1, alpha=5e-3, max_episode_steps=9,
              deterministic=True, gestation_successes=40)
    res = []
    for grid, read in ((0, False), (32, False), (32, True)):
        _, gag = _pair(scg, torch, B, K, 23, grid, active=1, oracle_side=False, **kw)
        for i, n in enumerate(CHUNKS):
            gag.run(n)
            if i % 2:
                gag.manage()
            if read:
                gag.occupancy()
        assert int(gag._struct.win_len) == sum(CHUNKS) % 8
        occ = gag.occupancy() if grid else None
        res.append((_learning_state(gag, torch), gag.controller_state(), occ))
        del gag
    (a, ca, _), (b, cb, ob), (c, cc, oc) = res
    for k in a:
        assert torch.equal(a[k], b[k]) and torch.equal(a[k], c[k]), k
    assert ca == cb == cc
    assert np.array_equal(ob["counts"], oc["counts"]) and ob["env_steps"] == B * sum(CHUNKS)


def test_host_paths_count_as_run(scg, torch):
    """run(60), 60 step() calls, 60 step_host() calls (the pipelined step over two parts of the batch) and run_host() in
    two calls: the same counts, equal to the oracle's."""
    B, K, G, T = 1024, 3, 64, 60
    kw = dict(sync_interval=4, option_timeout=6, epsilon=1.0, alpha=5e-3, max_episode_steps=9, deterministic=True)
    oag, _ = _pair(scg, torch, B, K, 7, G, active=1, **kw)
    for _ in range(T):
        oag.step()
    for mode in ("run", "step", "host", "run_host"):
        _, gag = _pair(scg, torch, B, K, 7, G, active=1, oracle_side=False, **kw)
        if mode == "run":
            gag.run(T)
        elif mode == "step":
            for _ in range(T):
                gag.step()
        elif mode == "host":
            hs, ha = gag.s.cpu().numpy().copy(), gag.action.cpu().numpy().copy()
            for _ in range(T):
                hs, r, f, ha, d = gag.step_host(hs, ha)
        else:
            hs, ha = gag.s.cpu().numpy().copy(), gag.action.cpu().numpy().copy()
            for n in (21, 39):
                hs, ha, r, f, d = gag.run_host(hs, ha, n)
        assert gag.t == T
        _check(gag.occupancy(), oag.counts, B, T, mode)
        del gag


def test_occupancy_checkpoint(scg, torch, tmp_path):
    """save() / load() carry the counts (the open window folded in); a checkpoint without a grid loads with zeros; a
    grid of another size is refused before anything is restored."""
    kw = dict(sync_interval=4, option_timeout=6, epsilon=1.0, max_episode_steps=5)
    B, K = 128, 2
    _, a = _pair(scg, torch, B, K, 4, 16, active=1, oracle_side=False, **kw)
    a.run(23)
    a.save(tmp_path / "a.npz")
    want = a.occupancy()
    assert want["env_steps"] == 23 * B
    _, b = _pair(scg, torch, B, K, 4, 16, active=1, oracle_side=False, **kw)
    b.run(2)
    b.load(tmp_path / "a.npz")
    assert np.array_equal(b.occupancy()["counts"], want["counts"])
    a.run(9)
    b.run(9)
    assert np.array_equal(b.occupancy()["counts"], a.occupancy()["counts"])
    _, c = _pair(scg, torch, B, K, 4, 0, active=1, oracle_side=False, **kw)      # no grid
    c.run(3)
    c.save(tmp_path / "c.npz")
    b.load(tmp_path / "c.npz")
    assert b.occupancy()["env_steps"] == 0 and not b.occupancy()["counts"].any()
    b.run(5)
    assert b.occupancy()["env_steps"] == 5 * B
    _, d = _pair(scg, torch, B, K, 4, 32, active=1, oracle_side=False, **kw)
    d.run(3)
    before = d.occupancy()["counts"].copy()
    with pytest.raises(ValueError):
        d.load(tmp_path / "a.npz")
    assert d.t == 3 and np.array_equal(d.occupancy()["counts"], before)


def test_two_ranks_gathered_occupancy(scg, torch):
    """Two half-batch ranks on one device (connected exchange contexts, one stream each) and the unsharded agent: the
    ranks' counts summed - what occupancy(gather=True) returns across a process group - equal the unsharded agent's."""
    import test_gpu_parity as tp
    lib = scg.load_library()
    Bh = 2048
    streams = [torch.cuda.Stream(), torch.cuda.Stream()]
    kw = dict(window=0, order=3, K=4, name="easy", max_episode_steps=5, occupancy_grid=64)
    whole, halves, xs = tp._two_rank_agents_one_device(scg, torch, Bh, streams, **kw)
    try:
        for h in halves + [whole]:
            h.cfg.sync_interval = 8
        for _ in range(3):
            for r in range(2):
                with torch.cuda.stream(streams[r]):
                    halves[r].run(8)
        with torch.cuda.stream(streams[0]):
            whole.run(24)
        torch.cuda.synchronize()
        assert torch.equal(torch.cat([halves[0].s, halves[1].s], dim=1), whole.s)
        parts = []
        for r in range(2):
            with torch.cuda.stream(streams[r]):
                p = halves[r].occupancy(gather=True)          # no process group: this rank's own counts
            assert p["per_rank"] == [24 * Bh]
            parts.append(halves[r].occupancy())
        merged = scg.merge_occupancy(parts)
        ref = whole.occupancy()
        assert merged["per_rank"] == [24 * Bh, 24 * Bh] and merged["env_steps"] == ref["env_steps"] == 24 * 2 * Bh
        assert np.array_equal(merged["counts"], ref["counts"])
        assert not np.array_equal(parts[0]["counts"], ref["counts"])
    finally:
        for h in halves:
            h._xchg = None
        for x in xs:
            lib.scg_xchg_destroy(x)


def test_occupancy_at_configs1_shape(scg, torch):
    """The configs[1] shape (easy map, 65,536 envs, order 3, 4 option slots, sync every 8 steps) for 200 steps with the
    controller running, too large for the oracle: the counts equal those built on the host from the state and option
    of every env before every step, and env_steps = 65,536 x 200."""
    B, K, G, T = 65536, 4, 64, 200
    cfg = scg.AgentConfig(map="easy", batch=B, order=3, max_options=K, sync_interval=8, seed=1, option_timeout=20,
                          max_episode_steps=100, gestation_successes=3000, example_capacity=4096, occupancy_grid=G)
    ag = scg.SkillChainAgent(cfg)
    theta = np.zeros((K, 6), dtype=np.float32)
    theta[0] = THETA[0]
    ag.options.theta.copy_(torch.as_tensor(theta))
    ag.active_mask, ag.n_active = 1, 1
    ag.parents_host[1] = 1
    ag._push_parents()
    want = np.zeros(K * G * G, dtype=np.int64)
    for t in range(T):
        s = ag.s[:2].cpu().numpy()
        o = ag.option.cpu().numpy().astype(np.int64)
        want += np.bincount((o * G + cells(s[1], G)) * G + cells(s[0], G), minlength=K * G * G)
        ag.step()
        if (t + 1) % 64 == 0:
            ag.manage()
    got = ag.occupancy()
    _check(got, want.reshape(K, G, G).astype(np.uint64), B, T, "configs[1] shape")
    assert ag.n_active >= 1 and (want.reshape(K, -1).sum(axis=1) > 0).sum() >= 2


def test_occupancy_off_by_default_and_bad_input(scg, torch):
    """occupancy() raises with the grid off; the C ABI refuses a grid that is not a power of two up to 128, counts
    without a grid and a grid without counts (SCG_EINVAL), and works again once the fields are restored."""
    cfg = dict(map="easy", batch=64, order=2, max_options=2, seed=1, max_episode_steps=5)
    off = scg.SkillChainAgent(scg.AgentConfig(**cfg))
    with pytest.raises(scg.ScgError):
        off.occupancy()
    ag = scg.SkillChainAgent(scg.AgentConfig(occupancy_grid=8, **cfg))
    lib, g = scg.load_library(), ag._struct
    saved = (g.occ_grid, g.occ_counts)
    try:
        for fields in ((3, saved[1]), (256, saved[1]), (12, saved[1]), (8, None), (0, saved[1])):
            g.occ_grid, g.occ_counts = fields
            assert lib.scg_agent_run(ag.map.handle, ag.options.ctx, C.byref(g), 1, 4, None, None) == -1, fields
            assert lib.scg_agent_occupancy(ag.options.ctx, C.byref(g), None) == -1, fields
            assert lib.scg_agent_step(ag.map.handle, ag.options.ctx, C.byref(g), None) == -1, fields
    finally:
        g.occ_grid, g.occ_counts = saved
    assert ag.t == 0
    ag.run(6)
    assert ag.occupancy()["env_steps"] == 6 * 64
