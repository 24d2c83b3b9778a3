"""The device trajectory log (AgentConfig.trajectory_envs / trajectory_log): every step of chosen envs (state, action,
option, TD error, termination, label, episode end, goal), gathered from the window's step records in (step, env) order,
against the oracle's (tests/oracle_trajectories.py) record for record, with states compared bit for bit."""
import ctypes as C

import numpy as np
import pytest

import oracle
from oracle.compare import assert_close
from oracle_trajectories import FLAGS, TrajectoryLoggingAgent

pytestmark = pytest.mark.gpu

EXACT = ("step", "env", "state", "action", "option") + FLAGS
KEYS = EXACT + ("delta",)
OPT_KEYS = ("step", "env", "option", "duration", "hit", "label", "env_done", "option_timeout", "left",
            "episode_timeout", "start", "end")
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


def _pair(scg, torch, B, K, seed, capacity, envs, near_goal=4, active=0, episode_log=0, option_log=0, **kw):
    """Oracle and GPU agents on the same start states (1 / near_goal of the envs next to the goal) and weights, with the
    first `active` options active (fixed classifiers, chain parents), tracking `envs`; the logs are GPU-only settings."""
    name = "easy"
    omap, gmap = oracle.PinballMap.from_name(name), scg.PinballMap.from_name(name)
    gpu_only = ("window", "event_history", "deterministic")
    cfg = dict(map=name, batch=B, order=2, max_options=K, seed=seed, **kw)
    oag = TrajectoryLoggingAgent(oracle.AgentConfig(**{k: v for k, v in cfg.items() if k not in gpu_only}), omap,
                                 trajectory_envs=envs)
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
    log = dict(trajectory_envs=tuple(envs), trajectory_log=capacity) if capacity else {}
    gag = scg.SkillChainAgent(scg.AgentConfig(episode_log=episode_log, option_log=option_log, **log, **cfg), gmap,
                              initial_states=S)
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


def _same(got, want, what, keys=EXACT, delta=False):
    """Fields equal (floats bit for bit); with delta=True the TD error within the oracle comparison's tolerance."""
    for k in keys:
        assert len(got[k]) == len(want[k]), f"{what}: {len(got[k])} records, expected {len(want[k])}"
        g, w = np.asarray(got[k]), np.asarray(want[k])
        if g.dtype.kind == "f":
            g, w = g.astype(np.float32).view(np.uint32), w.astype(np.float32).view(np.uint32)
        assert np.array_equal(g, w), f"{what}: field {k} differs"
    if delta and len(want["delta"]):
        assert_close(np.asarray(got["delta"]), np.asarray(want["delta"]), what=f"{what}: TD error")


def _tail(log, n):
    return {k: v[len(v) - n:] if n else v[:0] for k, v in log.items()}


def _for_envs(log, envs):
    mine = np.isin(log["env"], np.asarray(envs, dtype=np.uint32))
    return {k: v[mine] for k, v in log.items() if k not in ("total", "totals")}


@pytest.mark.parametrize("window,top_level", [(1, False), (8, False), (1, True), (8, True)])
def test_trajectory_log_matches_oracle(scg, torch, window, top_level):
    """epsilon = 1 (and epsilon_top = 1): both agents follow identical trajectories, with two active options so that
    every flag occurs.  Chunks of uneven length, so most polls fall inside an open window (the log then gathers that
    window's first steps, and the flush the rest); polled incrementally (since = the previous total) and in full, the
    GPU log equals the oracle's record for record."""
    B, K = 512, 4
    envs = sorted(set(range(0, B, 5)) | {1, 2, B - 1})
    kw = dict(sync_interval=8, option_timeout=6, epsilon=1.0, epsilon_top=1.0, alpha=1e-3, max_episode_steps=14,
              gestation_successes=10 ** 9, window=window, event_history=16, top_level=top_level, init_horizon=3)
    oag, gag = _pair(scg, torch, B, K, 41, 1 << 16, envs, active=2, **kw)
    polled = {k: [] for k in KEYS}
    total = 0
    for i, n in enumerate((5, 11, 1, 8, 24, 3, 29)):
        gag.run(n)
        for _ in range(n):
            oag.step()
        if i % 2:
            gag.manage()
        got = gag.trajectories(since=total)
        want = oag.trajectory_log()
        assert got["total"] == len(want["step"]) == gag.t * len(envs)
        _same(got, _tail(want, got["total"] - total), f"chunk {i}: new records", delta=True)
        for k in KEYS:
            polled[k].append(got[k])
        total = got["total"]
    want = oag.trajectory_log()
    _same({k: np.concatenate(v) for k, v in polled.items()}, want, "incremental polls", delta=True)
    _same(gag.trajectories(), want, "whole log", delta=True)
    for k in FLAGS:
        assert want[k].any() and not want[k].all(), k
    assert len(np.unique(want["option"])) >= 3


def _run_mode(gag, mode, T):
    if mode == "run":
        gag.run(T)
    elif mode == "chunks":
        for n in (7, 13, 1, 39):
            gag.run(n)
            gag.trajectories()
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


def test_trajectory_log_independent_of_launch_geometry(scg, torch):
    """The same run through run(60), run() in uneven chunks with a read after each, 60 step() calls, 60 step_host()
    calls (the pipelined step over two parts of the batch: tracked envs in both) and run_host(): identical logs
    (deterministic mode), TD errors within the comparison tolerance (a host step re-evaluates Q_o(s, a) where a device
    loop carries it, so the last bits may differ)."""
    B, K, T = 1024, 3, 60
    envs = list(range(3, B, 37))
    kw = dict(sync_interval=4, option_timeout=6, epsilon=0.1, alpha=5e-3, max_episode_steps=9, deterministic=True)
    logs = []
    for mode in ("run", "chunks", "step", "host", "run_host"):
        _, gag = _pair(scg, torch, B, K, 7, 1 << 15, envs, active=1, **kw)
        _run_mode(gag, mode, T)
        assert gag.t == T
        logs.append((mode, gag.trajectories()))
        del gag
    ref = logs[0][1]
    assert ref["total"] == T * len(envs) and ref["term"].any() and ref["episode_end"].any()
    for mode, log in logs[1:]:
        assert log["total"] == ref["total"], mode
        _same(log, ref, mode, delta=True)


def test_polling_does_not_perturb_learning(scg, torch):
    """The same run with trajectories() read after every step and with no reads at all: weights, traces, dW, example
    rings, state and the log itself are bitwise equal, also in the middle of a window (reading gathers, it never
    flushes, so the sweeps split the windows in the same places)."""
    B, K = 2048, 3
    envs = list(range(0, B, 9))
    kw = dict(sync_interval=8, window=8, option_timeout=6, epsilon=0.1, alpha=5e-3, max_episode_steps=9,
              deterministic=True, gestation_successes=40)
    res = []
    for poll in (False, True):
        _, gag = _pair(scg, torch, B, K, 23, 1 << 16, envs, active=1, **kw)
        for t in range(45):
            gag.step()
            if (t + 1) % 16 == 0:
                gag.manage()
            if poll:
                gag.trajectories()
        torch.cuda.synchronize()
        assert int(gag._struct.win_len) == 45 % 8
        o = gag.options
        # (not ev_hist itself: the example-ring pass every read runs recycles its rows sooner, the events are the same)
        raw = dict(dW=o._dW.clone(), trace=o._trace.clone(), cnt=o._cnt.clone(), W=o.W.clone(), s=gag.s.clone(),
                   action=gag.action.clone(), win_rec=gag.win_rec.clone())
        log = gag.trajectories()
        gag.flush()
        raw.update(dW2=o._dW.clone(), trace2=o._trace.clone(), ex_xy=gag.ex_xy.clone(), ex_label=gag.ex_label.clone(),
                   ex_count=gag.ex_count.clone(), theta=o.theta.clone())
        res.append((raw, log, gag.controller_state()))
        del gag
    (a, la, ca), (b, lb, cb) = res
    for k in a:
        assert torch.equal(a[k], b[k]), k
    assert ca == cb
    _same(la, lb, "polled vs unpolled", keys=KEYS)
    assert la["total"] == 45 * len(envs)


@pytest.mark.parametrize("capacity", [100, 500])
def test_trajectory_log_overflow_keeps_the_last_records(scg, torch, capacity):
    """More records than the ring holds (capacity not a multiple of the 7 tracked envs): the log holds exactly the
    oracle's last `capacity` records, total counts every one, and a poll from an index that has been overwritten
    returns what survives (total - since - len of them are lost)."""
    B, K = 256, 2
    envs = [0, 1, 40, 41, 100, 200, 255]
    kw = dict(sync_interval=4, option_timeout=6, epsilon=1.0, alpha=1e-3, max_episode_steps=7, gestation_successes=10 ** 9)
    oag, gag = _pair(scg, torch, B, K, 3, capacity, envs, **kw)
    for n in (9, 17, 30, 70, 121):
        gag.run(n)
        for _ in range(n):
            oag.step()
        want = oag.trajectory_log()
        got = gag.trajectories()
        assert got["total"] == len(want["step"]) == gag.t * len(envs)
        _same(got, _tail(want, min(capacity, got["total"])), f"after {gag.t} steps", delta=True)
        part = gag.trajectories(since=got["total"] - 37)
        _same(part, _tail(want, min(37, capacity)), "poll of the last 37")
        old = gag.trajectories(since=1)
        _same(old, _tail(want, min(capacity, got["total"] - 1)), "poll from an overwritten index")
        assert old["total"] - 1 - len(old["step"]) == max(0, got["total"] - capacity - 1)
    assert got["total"] > 3 * capacity


def _run_for_compare(scg, torch, traj, episode_log, option_log):
    B, K = 2048, 3
    kw = dict(sync_interval=4, option_timeout=6, epsilon=0.1, alpha=5e-3, max_episode_steps=9, deterministic=True,
              gestation_successes=40, event_history=24)
    _, gag = _pair(scg, torch, B, K, 19, traj, list(range(5, B, 11)), active=1, episode_log=episode_log,
                   option_log=option_log, **kw)
    for _ in range(5):
        gag.run(8)
        gag.manage()
        if traj:
            gag.trajectories()
    gag.run(5)            # an open window, events not yet in the rings
    torch.cuda.synchronize()
    ev = gag.ev_hist.clone()
    gag.flush()
    return gag, ev


def test_trajectory_log_off_changes_nothing(scg, torch):
    """The log off against on, with and without the episode and option logs: the event history is equal but for the
    episode bits (ev & 0xCF), and fully equal when neither the episode log nor the trajectory log is on; weights, traces,
    example rings, controller, state and the other two logs are bitwise equal, and the trajectory log is the same
    whatever other log is on."""
    T, E, O = 1 << 16, 1 << 15, 1 << 16
    combos = ((0, 0, 0), (T, 0, 0), (0, E, O), (T, E, O), (T, 0, O))
    runs = {c: _run_for_compare(scg, torch, *c) for c in combos}
    off, ev_off = runs[(0, 0, 0)]
    with pytest.raises(scg.ScgError):
        off.trajectories()
    for (t, e, o), (ag, ev) in runs.items():
        assert torch.equal(ev & 0xCF, ev_off), (t, e, o)
        if not (t or e):
            assert torch.equal(ev, ev_off)
        else:
            assert not torch.equal(ev, ev_off)                  # the episode ends are marked
        assert torch.equal(off.ex_count, ag.ex_count) and torch.equal(off.ex_xy, ag.ex_xy)
        assert torch.equal(off.ex_label, ag.ex_label)
        assert torch.equal(off.options.W, ag.options.W) and torch.equal(off.options.trace, ag.options.trace)
        assert torch.equal(off.options.theta, ag.options.theta) and torch.equal(off.s, ag.s)
        assert off.controller_state() == ag.controller_state()
    ref = runs[(T, 0, 0)][0].trajectories()
    assert ref["total"] == 45 * len(range(5, 2048, 11)) and ref["episode_end"].any() and ref["goal"].any()
    for c in ((T, E, O), (T, 0, O)):
        _same(runs[c][0].trajectories(), ref, f"trajectory log with {c}", keys=KEYS)
    _same(runs[(T, E, O)][0].episodes(), runs[(0, E, O)][0].episodes(), "episode log", keys=EP_KEYS)
    for c in ((T, E, O), (T, 0, O)):
        _same(runs[c][0].option_executions(), runs[(0, E, O)][0].option_executions(), f"option log with {c}",
              keys=OPT_KEYS)


def test_trajectory_log_rejects_bad_input(scg, torch):
    """Python refuses half-set, duplicate and out-of-range settings; the C ABI refuses half-set fields and traj_n > B,
    and an out-of-range device index yields records with env 0xFFFFFFFF and a zero payload instead of a fault."""
    B = 64
    cfg = dict(map="easy", batch=B, order=2, max_options=2, seed=1, max_episode_steps=5)
    for bad in (dict(trajectory_envs=(1, 2)), dict(trajectory_log=100), dict(trajectory_envs=(3, 1, 3), trajectory_log=9),
                dict(trajectory_envs=(0, B), trajectory_log=9), dict(trajectory_envs=(-1, 2), trajectory_log=9),
                dict(trajectory_envs=(0,), trajectory_log=-1)):
        with pytest.raises(ValueError):
            scg.SkillChainAgent(scg.AgentConfig(**cfg, **bad))
    ag = scg.SkillChainAgent(scg.AgentConfig(**cfg, trajectory_envs=(5, 0, 9), trajectory_log=128))
    assert ag._traj_env.cpu().tolist() == [0, 5, 9]            # sorted
    lib, g = scg.load_library(), ag._struct
    saved = (g.traj_n, g.traj_env, g.traj_capacity, g.traj_log, g.traj_log_count)
    bad = ((3, None, 128, saved[3], saved[4]), (3, saved[1], 128, None, saved[4]), (3, saved[1], 128, saved[3], None),
           (3, saved[1], 0, saved[3], saved[4]), (0, saved[1], 128, saved[3], saved[4]),
           (B + 1, saved[1], 128, saved[3], saved[4]), (0, None, 128, None, None), (0, None, 0, None, saved[4]))
    try:
        for fields in bad:
            g.traj_n, g.traj_env, g.traj_capacity, g.traj_log, g.traj_log_count = fields
            assert lib.scg_agent_run(ag.map.handle, ag.options.ctx, C.byref(g), 1, 4, None, None) == -1
            assert lib.scg_agent_traj(ag.options.ctx, C.byref(g), None) == -1
    finally:
        g.traj_n, g.traj_env, g.traj_capacity, g.traj_log, g.traj_log_count = saved
    ag.run(6)
    assert ag.trajectories()["total"] == 18
    # out-of-range indices poked into the device list (Python never passes them): flagged records, no fault
    ag._traj_env.copy_(torch.tensor([0, B + 1000, -7], dtype=torch.int32))
    ag.run(3)
    log = ag.trajectories(since=18)
    torch.cuda.synchronize()
    assert log["total"] == 27
    assert np.array_equal(log["env"], np.tile(np.array([0, 0xFFFFFFFF, 0xFFFFFFFF], dtype=np.uint32), 3))
    assert np.array_equal(log["step"], np.repeat(np.arange(6, 9, dtype=np.uint32), 3))
    bad_rows = log["env"] == 0xFFFFFFFF
    assert not log["state"][bad_rows].view(np.uint32).any() and not log["delta"][bad_rows].view(np.uint32).any()
    assert not (log["action"][bad_rows].any() or log["option"][bad_rows].any())
    for k in FLAGS:
        assert not log[k][bad_rows].any()


def test_trajectory_log_checkpoint(scg, torch, tmp_path):
    """save() / load() carry the log and its count; a checkpoint without a log loads with an empty one."""
    kw = dict(sync_interval=4, option_timeout=6, epsilon=1.0, max_episode_steps=5)
    envs = [0, 7, 100, 127]
    _, a = _pair(scg, torch, 128, 2, 4, 300, envs, **kw)
    a.run(23)
    a.save(tmp_path / "a.npz")
    want = a.trajectories()
    _, b = _pair(scg, torch, 128, 2, 4, 300, envs, **kw)
    b.run(2)
    b.load(tmp_path / "a.npz")
    _same(b.trajectories(), want, "restored log", keys=KEYS)
    assert b.trajectories()["total"] == want["total"] == 23 * len(envs)
    a.run(9)
    b.run(9)
    _same(b.trajectories(), a.trajectories(), "after resuming", delta=True)     # (b re-evaluates Q_o(s, a) first)
    _, c = _pair(scg, torch, 128, 2, 4, 0, envs, **kw)              # no log
    c.run(3)
    c.save(tmp_path / "c.npz")
    b.load(tmp_path / "c.npz")
    assert b.trajectories()["total"] == 0 and len(b.trajectories()["step"]) == 0
    b.run(5)
    assert b.trajectories()["total"] == 5 * len(envs)


def test_two_ranks_gathered_log(scg, torch):
    """Two half-batch ranks on one device (connected exchange contexts, one stream each) each tracking the same local
    envs, and the unsharded agent tracking both copies: the per-rank logs merged by (step, env) - what
    trajectories(gather=True) returns across a process group - equal the unsharded agent's log."""
    import test_gpu_parity as tp
    lib = scg.load_library()
    Bh = 2048
    local = list(range(0, Bh, 97)) + [Bh - 1]
    streams = [torch.cuda.Stream(), torch.cuda.Stream()]
    kw = dict(window=0, order=3, K=4, name="easy", max_episode_steps=5)
    log = dict(trajectory_envs=tuple(local), trajectory_log=1 << 14)
    _, halves, xs = tp._two_rank_agents_one_device(scg, torch, Bh, streams, **kw, **log)
    saved, tp.FULL_B = tp.FULL_B, 2 * Bh
    try:
        with torch.cuda.stream(streams[0]):
            whole = tp._full_agent(scg, torch, 2 * Bh, 0, trajectory_envs=tuple(local + [b + Bh for b in local]),
                                   trajectory_log=1 << 15, **kw)
        torch.cuda.synchronize()
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
                p = halves[r].trajectories(gather=True)          # no process group: this rank's own log
            env = p["env"].astype(np.int64)
            assert env.min() >= r * Bh and env.max() < (r + 1) * Bh
            parts.append(p)
        merged = scg.merge_episodes(parts)
        ref = whole.trajectories()
        assert merged["total"] == ref["total"] == 24 * 2 * len(local) and merged["totals"] == [p["total"] for p in parts]
        _same(merged, ref, "merged ranks vs unsharded", delta=True)    # (dW summed over ranks in another order)
        assert ref["episode_end"].any() and ref["term"].any()
    finally:
        tp.FULL_B = saved
        for h in halves:
            h._xchg = None
        for x in xs:
            lib.scg_xchg_destroy(x)


def test_trajectory_log_at_configs1_shape(scg, torch):
    """The configs[1] shape (easy map, 65,536 envs, order 3, 4 options, sync every 8 steps), too large for the oracle,
    with all three logs on, every 64th env tracked and the controller running: record t of a tracked env is its state,
    action and option before step t, bit for bit; its terminations are the option log's records of those envs and its
    episode ends the episode log's."""
    B, K = 65536, 4
    envs = np.arange(0, B, 64)
    cfg = scg.AgentConfig(map="easy", batch=B, order=3, max_options=K, sync_interval=8, seed=1, option_timeout=20,
                          max_episode_steps=100, gestation_successes=3000, example_capacity=4096, option_log=1 << 22,
                          episode_log=1 << 20, trajectory_envs=tuple(int(b) for b in envs), trajectory_log=1 << 18)
    ag = scg.SkillChainAgent(cfg)
    theta = np.zeros((K, 6), dtype=np.float32)
    theta[0] = THETA[0]
    ag.options.theta.copy_(torch.as_tensor(theta))
    ag.active_mask, ag.n_active = 1, 1
    ag.parents_host[1] = 1
    ag._push_parents()
    idx = torch.as_tensor(envs).cuda()
    states, actions, options = [], [], []
    T = 200
    for t in range(T):
        states.append(ag.s[:, idx].t().cpu().numpy())
        actions.append(ag.action[idx].cpu().numpy())
        options.append(ag.option[idx].cpu().numpy())
        ag.step()
        if (t + 1) % 64 == 0:
            ag.manage()
    tr = ag.trajectories()
    n = len(envs)
    assert tr["total"] == T * n == len(tr["step"])
    assert np.array_equal(tr["step"], np.repeat(np.arange(T, dtype=np.uint32), n))
    assert np.array_equal(tr["env"], np.tile(envs.astype(np.uint32), T))
    assert np.array_equal(tr["state"].view(np.uint32), np.concatenate(states).view(np.uint32))
    assert np.array_equal(tr["action"], np.concatenate(actions)) and np.array_equal(tr["option"], np.concatenate(options))
    ol = _for_envs(ag.option_executions(), envs)
    assert ol["step"].size < (1 << 22) and tr["term"].sum() > n
    for k in ("step", "env", "option", "label"):
        assert np.array_equal(tr[k][tr["term"]], ol[k]), k
    el = _for_envs(ag.episodes(), envs)
    end = tr["episode_end"]
    assert end.sum() > n
    for k in ("step", "env", "goal"):
        assert np.array_equal(tr[k][end], el[k]), k
    assert ag.n_active >= 1 and tr["label"].any()
