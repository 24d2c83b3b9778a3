"""The device option log (AgentConfig.option_log): every option termination (step, env, option, duration, outcome, start
and end), appended by the deterministic ring pass in the oracle's (step, env) order, against the oracle's executions
(tests/oracle_options.py) record for record, with positions compared bit for bit."""
import numpy as np
import pytest

import oracle
from oracle_options import OUTCOMES, OptionLoggingAgent

pytestmark = pytest.mark.gpu

KEYS = ("step", "env", "option", "duration") + OUTCOMES + ("start", "end")
EP_KEYS = ("step", "env", "ret", "length", "goal")


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


def _pair(scg, torch, B, K, seed, capacity, near_goal=4, active=0, episode_log=0, **kw):
    """Oracle and GPU agents on the same start states (1 / near_goal of the envs next to the goal) and weights, with the
    first `active` options active (fixed classifiers, chain parents); the logs are GPU-only settings."""
    name = "easy"
    omap, gmap = oracle.PinballMap.from_name(name), scg.PinballMap.from_name(name)
    gpu_only = ("window", "event_history", "deterministic")
    cfg = dict(map=name, batch=B, order=2, max_options=K, seed=seed, **kw)
    oag = OptionLoggingAgent(oracle.AgentConfig(**{k: v for k, v in cfg.items() if k not in gpu_only}), omap)
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
    gag = scg.SkillChainAgent(scg.AgentConfig(option_log=capacity, episode_log=episode_log, **cfg), gmap, initial_states=S)
    W = (rng.standard_normal(oag.options.W.shape) * 0.3).astype(np.float32)
    oag.options.W[:] = W
    gag.options.set_weights(W)
    if active:
        theta = np.zeros((K, 6), dtype=np.float32)
        theta[:active] = THETA[:active]
        oag.options.theta[:] = theta
        oag.active[:active] = True
        oag.n_active = active
        for j in range(1, active + 1):
            oag.parents[j] = 1 << (j - 1)
        gag.options.theta.copy_(torch.as_tensor(theta))
        gag.active_mask, gag.n_active = (1 << active) - 1, active
        for j in range(1, active + 1):
            gag.parents_host[j] = 1 << (j - 1)
        gag._push_parents()
    A = rng.integers(0, 5, B).astype(np.int32)
    oag.action = A.copy()
    gag.action.copy_(torch.as_tensor(A))
    gag.invalidate()
    return oag, gag


def _same(got, want, what, keys=KEYS):
    for k in keys:
        assert len(got[k]) == len(want[k]), f"{what}: {len(got[k])} records, oracle {len(want[k])}"
        g, w = np.asarray(got[k]), np.asarray(want[k])
        if g.dtype.kind == "f":                            # bit for bit
            g, w = g.astype(np.float32).view(np.uint32), w.astype(np.float32).view(np.uint32)
        assert np.array_equal(g, w), f"{what}: field {k} differs"


def _tail(log, n):
    return {k: v[len(v) - n:] if n else v[:0] for k, v in log.items()}


@pytest.mark.parametrize("window,top_level", [(1, False), (8, False), (1, True), (8, True)])
def test_option_log_matches_oracle(scg, torch, window, top_level):
    """epsilon = 1 (and epsilon_top = 1): both agents follow identical trajectories, with two active options so that
    every outcome occurs.  Several chunks of steps with the ring pass run by manage() and, with a 16-step event
    history, by the flush when the history is full; polled incrementally (since = the previous total) and in full, the
    GPU log equals the oracle's record for record."""
    B, K = 512, 4
    kw = dict(sync_interval=4, option_timeout=6, epsilon=1.0, epsilon_top=1.0, alpha=1e-3, max_episode_steps=14,
              gestation_successes=10 ** 9, window=window, event_history=16, top_level=top_level, init_horizon=3)
    oag, gag = _pair(scg, torch, B, K, 41, 1 << 16, active=2, **kw)
    polled = {k: [] for k in KEYS}
    total = 0
    for i, n in enumerate((5, 11, 8, 24, 3, 29)):
        gag.run(n)
        for _ in range(n):
            oag.step()
        if i % 2:
            gag.manage()
        got = gag.option_executions(since=total)
        want = oag.option_log()
        assert got["total"] == len(want["step"]) == int(oag.n_success.sum() + oag.n_fail.sum())
        _same(got, _tail(want, got["total"] - total), f"chunk {i}: new records")
        for k in KEYS:
            polled[k].append(got[k])
        total = got["total"]
    want = oag.option_log()
    _same({k: np.concatenate(v) for k, v in polled.items()}, want, "incremental polls")
    _same(gag.option_executions(), want, "whole log")
    for k in OUTCOMES:
        assert want[k].any() and not want[k].all(), k
    assert total > 4 * B
    assert np.array_equal(gag.n_success.cpu().numpy(), oag.n_success)
    assert np.array_equal(gag.n_fail.cpu().numpy(), oag.n_fail)


def _run_mode(gag, mode, T):
    if mode == "run":
        gag.run(T)
    elif mode == "chunks":
        for n in (7, 13, 1, 39):
            gag.run(n)
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


def test_option_log_independent_of_launch_geometry(scg, torch):
    """The same run through run(60), run() in uneven chunks, 60 step() calls, 60 step_host() calls (the pipelined step
    over two parts of the batch) and run_host(): identical logs (deterministic mode, so the learned weights and with
    them the greedy actions are identical too)."""
    B, K, T = 1024, 3, 60
    kw = dict(sync_interval=4, option_timeout=6, epsilon=0.1, alpha=5e-3, max_episode_steps=9, deterministic=True)
    logs = []
    for mode in ("run", "chunks", "step", "host", "run_host"):
        _, gag = _pair(scg, torch, B, K, 7, 1 << 15, active=1, **kw)
        _run_mode(gag, mode, T)
        assert gag.t == T
        logs.append((mode, gag.option_executions()))
        del gag
    ref = logs[0][1]
    assert ref["total"] > B and ref["hit"].any() and ref["left"].any()
    for mode, log in logs[1:]:
        assert log["total"] == ref["total"], mode
        _same(log, ref, mode)


@pytest.mark.parametrize("capacity", [100, 500])
def test_option_log_overflow_keeps_the_last_records(scg, torch, capacity):
    """More executions than the ring holds: the log holds exactly the oracle's last `capacity` records, total counts
    every one, and a poll from an index that has been overwritten returns what survives (total - since - len of them
    are lost)."""
    B, K = 256, 2
    kw = dict(sync_interval=4, option_timeout=6, epsilon=1.0, alpha=1e-3, max_episode_steps=7, gestation_successes=10 ** 9)
    oag, gag = _pair(scg, torch, B, K, 3, capacity, **kw)
    for n in (9, 17, 30):
        gag.run(n)
        for _ in range(n):
            oag.step()
        want = oag.option_log()
        got = gag.option_executions()
        assert got["total"] == len(want["step"])
        _same(got, _tail(want, min(capacity, got["total"])), f"after {gag.t} steps")
        part = gag.option_executions(since=got["total"] - 37)
        _same(part, _tail(want, min(37, capacity)), "poll of the last 37")
        old = gag.option_executions(since=1)
        _same(old, _tail(want, min(capacity, got["total"] - 1)), "poll from an overwritten index")
        assert old["total"] - 1 - len(old["step"]) == max(0, got["total"] - capacity - 1)
    assert got["total"] > 3 * capacity


def _run_for_compare(scg, torch, option_log, episode_log):
    B, K = 2048, 3
    kw = dict(sync_interval=4, option_timeout=6, epsilon=0.1, alpha=5e-3, max_episode_steps=9, deterministic=True,
              gestation_successes=40, event_history=24)
    _, gag = _pair(scg, torch, B, K, 19, option_log, active=1, episode_log=episode_log, **kw)
    for _ in range(5):
        gag.run(8)
        gag.manage()
    gag.run(5)            # an open window, events not yet in the rings
    torch.cuda.synchronize()
    ev = gag.ev_hist.clone()
    gag.flush()
    return gag, ev


def test_option_log_off_changes_nothing(scg, torch):
    """option_log = 0 against the same run with the log on, and both logs on against each alone: the event history, the
    example rings, the weights, the traces, the controller and the episode log are bitwise equal, and the option log is
    the same whether the episode log is on or not."""
    runs = {(o, e): _run_for_compare(scg, torch, o, e) for o, e in ((0, 0), (1 << 16, 0), (0, 1 << 15), (1 << 16, 1 << 15))}
    off, ev_off = runs[(0, 0)]
    assert off.ev_opt is None
    with pytest.raises(scg.ScgError):
        off.option_executions()
    for (o, e), (ag, ev) in runs.items():
        assert torch.equal(ev & 0xCF, ev_off), (o, e)          # the episode log's own bits aside
        if not e:
            assert torch.equal(ev, ev_off)
        assert torch.equal(off.ex_count, ag.ex_count) and torch.equal(off.ex_xy, ag.ex_xy)
        assert torch.equal(off.ex_label, ag.ex_label)
        assert torch.equal(off.options.W, ag.options.W) and torch.equal(off.options.trace, ag.options.trace)
        assert torch.equal(off.options.theta, ag.options.theta) and torch.equal(off.s, ag.s)
        assert off.controller_state() == ag.controller_state()
    on = runs[(1 << 16, 0)][0]
    log = on.option_executions()
    assert log["left"].any() and log["hit"].any()
    assert log["total"] == int(on.n_success.sum() + on.n_fail.sum()) == int(on.ex_count.sum()) < 1 << 16
    _same(runs[(1 << 16, 1 << 15)][0].option_executions(), log, "option log with the episode log on")
    _same(runs[(1 << 16, 1 << 15)][0].episodes(), runs[(0, 1 << 15)][0].episodes(), "episode log with the option log on",
          keys=EP_KEYS)


def test_option_log_rejects_half_set_fields(scg, torch):
    """The C ABI takes the log's fields all set or all NULL."""
    import ctypes as C
    _, gag = _pair(scg, torch, 64, 2, 1, 128, max_episode_steps=5)
    lib, g = scg.load_library(), gag._struct
    saved = (g.ev_opt, g.opt_log, g.opt_log_count, g.option_capacity)
    bad = ((saved[0], None, saved[2], 128), (None, saved[1], saved[2], 128), (saved[0], saved[1], None, 128),
           (saved[0], saved[1], saved[2], 0), (None, None, None, 128), (None, None, saved[2], 0))
    try:
        for fields in bad:
            g.ev_opt, g.opt_log, g.opt_log_count, g.option_capacity = fields
            assert lib.scg_agent_run(gag.map.handle, gag.options.ctx, C.byref(g), 1, 4, None, None) == -1
            assert lib.scg_agent_ring(gag.options.ctx, C.byref(g), None) == -1
    finally:
        g.ev_opt, g.opt_log, g.opt_log_count, g.option_capacity = saved
    gag.run(6)
    assert gag.option_executions()["total"] == int(gag.n_success.sum() + gag.n_fail.sum()) >= 64


def test_option_log_checkpoint(scg, torch, tmp_path):
    """save() / load() carry the log and its count; a checkpoint without a log loads with an empty one."""
    kw = dict(sync_interval=4, option_timeout=6, epsilon=1.0, max_episode_steps=5)
    _, a = _pair(scg, torch, 128, 2, 4, 300, **kw)
    a.run(23)
    a.save(tmp_path / "a.npz")
    want = a.option_executions()
    _, b = _pair(scg, torch, 128, 2, 4, 300, **kw)
    b.load(tmp_path / "a.npz")
    _same(b.option_executions(), want, "restored log")
    assert b.option_executions()["total"] == want["total"] == int(a.n_success.sum() + a.n_fail.sum()) >= 128 * 4
    a.run(9)
    b.run(9)
    _same(b.option_executions(), a.option_executions(), "after resuming")
    _, c = _pair(scg, torch, 128, 2, 4, 0, **kw)              # no log
    c.run(3)
    c.save(tmp_path / "c.npz")
    b.load(tmp_path / "c.npz")
    assert b.option_executions()["total"] == 0 and len(b.option_executions()["step"]) == 0


def test_two_ranks_gathered_log(scg, torch):
    """Two half-batch ranks on one device (connected exchange contexts, one stream each) and the unsharded agent: the
    per-rank logs merged by (step, env) - what option_executions(gather=True) returns across a process group - equal
    the unsharded agent's log, and each rank's env ids lie in its slice."""
    from test_gpu_parity import _two_rank_agents_one_device
    lib = scg.load_library()
    Bh = 2048
    streams = [torch.cuda.Stream(), torch.cuda.Stream()]
    kw = dict(window=0, order=3, K=4, name="easy", max_episode_steps=5, option_log=1 << 17)
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
                p = halves[r].option_executions(gather=True)       # no process group: this rank's own log
            env = p["env"].astype(np.int64)
            assert env.min() >= r * Bh and env.max() < (r + 1) * Bh
            parts.append(p)
        merged = scg.merge_episodes(parts)
        ref = whole.option_executions()
        assert merged["total"] == ref["total"] == sum(p["total"] for p in parts) and merged["totals"] == [p["total"] for p in parts]
        _same(merged, ref, "merged ranks vs unsharded")
        assert ref["total"] >= 2 * Bh * 4                         # every env timed out at least 4 times in 24 steps
    finally:
        for h in halves:
            h._xchg = None
        for x in xs:
            lib.scg_xchg_destroy(x)


def test_option_log_reproduces_example_rings_at_configs1_shape(scg, torch):
    """The configs[1] shape (easy map, 65,536 envs, order 3, 4 options, sync every 8 steps), too large for the oracle,
    with short option timeouts, option 0 active (x >= 0.5, so that its successor has a target it reaches) and the
    controller running: per option, the records are the rise of n_success + n_fail (the hits that of n_success), and
    option k's records, in order, reproduce its device example ring - the last example_capacity of them, at slot
    index % example_capacity."""
    B, K, cap = 65536, 4, 4096
    cfg = scg.AgentConfig(map="easy", batch=B, order=3, max_options=K, sync_interval=8, seed=1, option_timeout=20,
                          max_episode_steps=100, gestation_successes=3000, example_capacity=cap, option_log=1 << 24)
    ag = scg.SkillChainAgent(cfg)
    theta = np.zeros((K, 6), dtype=np.float32)
    theta[0] = THETA[0]
    ag.options.theta.copy_(torch.as_tensor(theta))
    ag.active_mask, ag.n_active = 1, 1
    ag.parents_host[1] = 1
    ag._push_parents()
    for _ in range(6):
        ag.run(32)
        ag.manage()
    ag.run(13)
    log = ag.option_executions()
    assert log["total"] == len(log["step"]) < 1 << 24     # (at most one termination per env-step)
    key = log["step"].astype(np.int64) * (1 << 32) + log["env"]
    assert np.all(np.diff(key) > 0)
    assert np.all((log["duration"] >= 1) & (log["duration"] <= 20))
    ns, nf = ag.n_success.cpu().numpy().astype(np.int64), ag.n_fail.cpu().numpy().astype(np.int64)
    ex_count, ex_xy, ex_label = ag.ex_count.cpu().numpy(), ag.ex_xy.cpu().numpy(), ag.ex_label.cpu().numpy()
    assert log["hit"].any() and not log["hit"].all() and log["left"].any() and ex_count[1] > cap
    for k in range(K):
        mine = log["option"] == k
        n = int(mine.sum())
        assert n == int(ns[k] + nf[k]) == int(ex_count[k])
        assert int((mine & log["hit"]).sum()) == int(ns[k])
        keep = min(n, cap)
        idx = np.arange(n - keep, n) % cap
        assert np.array_equal(log["start"][mine][n - keep:].view(np.uint32), ex_xy[k, idx].view(np.uint32)), k
        assert np.array_equal(log["label"][mine][n - keep:].astype(np.uint8), ex_label[k, idx]), k
    assert log["total"] > B
