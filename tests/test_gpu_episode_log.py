"""The device episode log (AgentConfig.episode_log): every finished episode (step, env, return, length, goal), appended by
the deterministic ring pass in the oracle's (step, env) order, against the oracle's episodes (tests/oracle_episodes.py)
record for record."""
import numpy as np
import pytest

import oracle
from oracle_episodes import EpisodeLoggingAgent

pytestmark = pytest.mark.gpu

KEYS = ("step", "env", "ret", "length", "goal")


@pytest.fixture(scope="module")
def scg():
    import skill_chaining_with_graphs_b200 as m
    m.load_library()
    return m


@pytest.fixture(scope="module")
def torch():
    import torch as t
    return t


def _pair(scg, torch, B, K, seed, capacity, near_goal=4, **kw):
    """Oracle and GPU agents on the same start states (1 / near_goal of the envs next to the goal) and weights; the
    episode log is a GPU-only setting."""
    name = "easy"
    omap, gmap = oracle.PinballMap.from_name(name), scg.PinballMap.from_name(name)
    gpu_only = ("window", "event_history", "deterministic")
    cfg = dict(map=name, batch=B, order=2, max_options=K, seed=seed, **kw)
    oag = EpisodeLoggingAgent(oracle.AgentConfig(**{k: v for k, v in cfg.items() if k not in gpu_only}), omap)
    rng = np.random.default_rng(seed)
    S = omap.sample_free_states(rng, B)
    tx, ty, _ = omap.target
    n = B // near_goal
    S[:n, 0] = tx + rng.uniform(-0.1, 0.0, n)
    S[:n, 1] = ty + rng.uniform(-0.05, 0.05, n)
    S[:n, 2:] = 0.0
    oag.env.reset(states=S)
    oag.start_xy = oag.env.state[:, :2].copy()
    oag.opt_s0 = oag.env.state.copy()
    gag = scg.SkillChainAgent(scg.AgentConfig(episode_log=capacity, **cfg), gmap, initial_states=S)
    W = (rng.standard_normal(oag.options.W.shape) * 0.3).astype(np.float32)
    oag.options.W[:] = W
    gag.options.set_weights(W)
    A = rng.integers(0, 5, B).astype(np.int32)
    oag.action = A.copy()
    gag.action.copy_(torch.as_tensor(A))
    gag.invalidate()
    return oag, gag


def _same(got, want, what):
    for k in KEYS:
        assert len(got[k]) == len(want[k]), f"{what}: {len(got[k])} records, oracle {len(want[k])}"
        g, w = np.asarray(got[k]), np.asarray(want[k])
        if k == "ret":                                     # bit for bit
            g, w = g.astype(np.float32).view(np.uint32), w.astype(np.float32).view(np.uint32)
        assert np.array_equal(g, w), f"{what}: field {k} differs"


def _tail(log, n):
    return {k: v[len(v) - n:] if n else v[:0] for k, v in log.items()}


@pytest.mark.parametrize("window,top_level", [(1, False), (8, False), (1, True), (8, True)])
def test_episode_log_matches_oracle(scg, torch, window, top_level):
    """epsilon = 1: both agents follow identical trajectories.  Several chunks of steps with the ring pass run by
    manage() and, with a 16-step event history, by the flush when the history is full; polled incrementally
    (since = the previous total) and in full, the GPU log equals the oracle's record for record."""
    B, K = 512, 3
    kw = dict(sync_interval=4, option_timeout=6, epsilon=1.0, alpha=1e-3, max_episode_steps=14,
              gestation_successes=10 ** 9, window=window, event_history=16, top_level=top_level)
    oag, gag = _pair(scg, torch, B, K, 41, 1 << 16, **kw)
    polled = {k: [] for k in KEYS}
    total = 0
    for i, n in enumerate((5, 11, 8, 24, 3, 29)):
        gag.run(n)
        for _ in range(n):
            oag.step()
        if i % 2:
            gag.manage()
        got = gag.episodes(since=total)
        want = oag.episode_log()
        assert got["total"] == len(want["step"]) == int(oag.episodes.sum())
        _same(got, _tail(want, got["total"] - total), f"chunk {i}: new records")
        for k in KEYS:
            polled[k].append(got[k])
        total = got["total"]
    want = oag.episode_log()
    _same({k: np.concatenate(v) for k, v in polled.items()}, want, "incremental polls")
    _same(gag.episodes(), want, "whole log")
    assert want["goal"].any() and not want["goal"].all() and total > 2 * B
    assert np.array_equal(gag.ep_count.cpu().numpy(), oag.episodes)
    assert int(gag.stats[0]) == total and int(gag.stats[1]) == int(want["goal"].sum())


def test_episode_log_independent_of_launch_geometry(scg, torch):
    """The same run through run(60), run() in uneven chunks, 60 step() calls and 60 step_host() calls: identical logs
    (deterministic mode, so the learned weights and with them the greedy actions are identical too)."""
    B, K, T = 1024, 3, 60
    kw = dict(sync_interval=4, option_timeout=6, epsilon=0.1, alpha=5e-3, max_episode_steps=9, deterministic=True)
    logs = []
    for mode in ("run", "chunks", "step", "host"):
        _, gag = _pair(scg, torch, B, K, 7, 1 << 15, **kw)
        if mode == "run":
            gag.run(T)
        elif mode == "chunks":
            for n in (7, 13, 1, 39):
                gag.run(n)
        elif mode == "step":
            for _ in range(T):
                gag.step()
        else:
            hs, ha = gag.s.cpu().numpy().copy(), gag.action.cpu().numpy().copy()
            for _ in range(T):
                hs, r, f, ha, d = gag.step_host(hs, ha)
        assert gag.t == T
        logs.append((mode, gag.episodes()))
        del gag
    ref = logs[0][1]
    assert ref["total"] > B and ref["goal"].any()
    for mode, log in logs[1:]:
        assert log["total"] == ref["total"], mode
        _same(log, ref, mode)


@pytest.mark.parametrize("capacity", [100, 500])
def test_episode_log_overflow_keeps_the_last_records(scg, torch, capacity):
    """More episodes than the ring holds: the log holds exactly the oracle's last `capacity` records, total counts every
    one, and a poll from an index that has been overwritten returns what survives."""
    B, K = 256, 2
    kw = dict(sync_interval=4, option_timeout=6, epsilon=1.0, alpha=1e-3, max_episode_steps=7, gestation_successes=10 ** 9)
    oag, gag = _pair(scg, torch, B, K, 3, capacity, **kw)
    for n in (9, 17, 30):
        gag.run(n)
        for _ in range(n):
            oag.step()
        want = oag.episode_log()
        got = gag.episodes()
        assert got["total"] == len(want["step"])
        _same(got, _tail(want, min(capacity, got["total"])), f"after {gag.t} steps")
        part = gag.episodes(since=got["total"] - 37)
        _same(part, _tail(want, min(37, capacity)), "poll of the last 37")
        old = gag.episodes(since=1)
        _same(old, _tail(want, min(capacity, got["total"] - 1)), "poll from an overwritten index")
    assert got["total"] > 3 * capacity


def test_episode_log_off_changes_nothing(scg, torch):
    """episode_log = 0 against the same run with the log on: the event history, the example rings, the weights and the
    traces are bitwise equal, and the event bytes differ only in the log's own two bits (EPEND 0x20, GOAL 0x10)."""
    B, K = 2048, 3
    kw = dict(sync_interval=4, option_timeout=6, epsilon=0.1, alpha=5e-3, max_episode_steps=9, deterministic=True,
              gestation_successes=40, event_history=24)
    ags = []
    for cap in (0, 1 << 15):
        _, gag = _pair(scg, torch, B, K, 19, cap, **kw)
        for _ in range(5):
            gag.run(8)
            gag.manage()
        gag.run(5)            # an open window, events not yet in the rings
        torch.cuda.synchronize()
        ev = gag.ev_hist.clone()
        gag.flush()
        ags.append((gag, ev))
    (off, ev_off), (on, ev_on) = ags
    assert off.ev_ep is None and on.ev_ep is not None
    assert int((ev_off & 0x30).sum()) == 0
    log = on.episodes()
    assert int(((ev_on & 0x20) != 0).sum()) > 0 and log["goal"].any() and log["total"] == int(on.stats[0]) < 1 << 15
    assert bool(((ev_on & 0x10) == 0).logical_or((ev_on & 0x20) != 0).all())      # GOAL only on an episode end
    assert torch.equal(ev_on & 0xCF, ev_off)
    assert bool(((ev_on & 0x20) == 0).logical_or((ev_on & 0x80) != 0).all())     # an episode end is a termination
    assert torch.equal(off.ex_count, on.ex_count) and torch.equal(off.ex_xy, on.ex_xy)
    assert torch.equal(off.ex_label, on.ex_label)
    assert torch.equal(off.options.W, on.options.W) and torch.equal(off.options.trace, on.options.trace)
    assert torch.equal(off.options.theta, on.options.theta) and torch.equal(off.s, on.s)
    assert off.controller_state() == on.controller_state()
    with pytest.raises(scg.ScgError):
        off.episodes()


def test_episode_log_rejects_half_set_fields(scg, torch):
    """The C ABI takes the log's fields all set or all NULL."""
    import ctypes as C
    _, gag = _pair(scg, torch, 64, 2, 1, 128, max_episode_steps=5)
    lib, g = scg.load_library(), gag._struct
    saved = (g.ev_ep, g.ep_log, g.episode_capacity)
    try:
        for ev_ep, ep_log, cap in ((saved[0], None, 128), (None, saved[1], 128), (saved[0], saved[1], 0)):
            g.ev_ep, g.ep_log, g.episode_capacity = ev_ep, ep_log, cap
            assert lib.scg_agent_run(gag.map.handle, gag.options.ctx, C.byref(g), 1, 4, None, None) == -1
            assert lib.scg_agent_ring(gag.options.ctx, C.byref(g), None) == -1
    finally:
        g.ev_ep, g.ep_log, g.episode_capacity = saved
    gag.run(6)
    assert gag.episodes()["total"] == int(gag.ep_count.sum()) >= 64


def test_episode_log_checkpoint(scg, torch, tmp_path):
    """save() / load() carry the log and its count; a checkpoint without a log loads with an empty one."""
    kw = dict(sync_interval=4, option_timeout=6, epsilon=1.0, max_episode_steps=5)
    _, a = _pair(scg, torch, 128, 2, 4, 300, **kw)
    a.run(23)
    a.save(tmp_path / "a.npz")
    want = a.episodes()
    _, b = _pair(scg, torch, 128, 2, 4, 300, **kw)
    b.load(tmp_path / "a.npz")
    _same(b.episodes(), want, "restored log")
    assert b.episodes()["total"] == want["total"] == int(a.ep_count.sum()) >= 128 * 4
    a.run(9)
    b.run(9)
    _same(b.episodes(), a.episodes(), "after resuming")
    _, c = _pair(scg, torch, 128, 2, 4, 0, **kw)              # no log
    c.run(3)
    c.save(tmp_path / "c.npz")
    b.load(tmp_path / "c.npz")
    assert b.episodes()["total"] == 0 and len(b.episodes()["step"]) == 0


def test_two_ranks_gathered_log(scg, torch):
    """Two half-batch ranks on one device (connected exchange contexts, one stream each) and the unsharded agent: the
    per-rank logs merged by (step, env) - what episodes(gather=True) returns across a process group - equal the
    unsharded agent's log, and each rank's env ids lie in its slice."""
    from test_gpu_parity import _two_rank_agents_one_device
    lib = scg.load_library()
    Bh = 2048
    streams = [torch.cuda.Stream(), torch.cuda.Stream()]
    kw = dict(window=0, order=3, K=4, name="easy", max_episode_steps=5, episode_log=1 << 16)
    whole, halves, xs = _two_rank_agents_one_device(scg, torch, Bh, streams, **kw)
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
                p = halves[r].episodes(gather=True)                # no process group: this rank's own log
            env = p["env"].astype(np.int64)
            assert env.min() >= r * Bh and env.max() < (r + 1) * Bh
            parts.append(p)
        merged = scg.merge_episodes(parts)
        ref = whole.episodes()
        assert merged["total"] == ref["total"] == sum(p["total"] for p in parts) and merged["totals"] == [p["total"] for p in parts]
        _same(merged, ref, "merged ranks vs unsharded")
        cat = {k: np.concatenate([p[k] for p in parts]) for k in KEYS}
        order = np.lexsort((cat["env"], cat["step"]))
        _same({k: v[order] for k, v in cat.items()}, merged, "merge is the (step, env)-sorted concatenation")
        assert ref["total"] >= 2 * Bh * 4                         # every env timed out at least 4 times in 24 steps
    finally:
        for h in halves:
            h._xchg = None
        for x in xs:
            lib.scg_xchg_destroy(x)
