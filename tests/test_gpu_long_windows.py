"""GPU parity of the multi-block window sweep (k_window with more than one table block of 8 steps, csrc/scg_sarsa.cu) at
windows of 13 to 32 steps: the third and fourth table blocks, windows that end on a block boundary, option segments that
straddle a boundary, envs with many segments, 32-step step-kernel launches, k_top over 32-step windows and the event
history at its minimum of two windows.

The bars are the suite's: states, termination flags, cnt, event bytes and example rings bit for bit; TD errors, traces,
dW and W element-wise (oracle.compare.assert_close, rtol 1e-4).  Traces and dW are held to two oracle forms: the dense
per-step agent (the normative numbers, fp32 traces) and a twin with windowed=True that follows the same choices (the
forward view with G_t and c_t in fp64).  A failure says which bar failed: one that only the dense bar sees lies in the
oracle's fp32 per-step traces, not in the kernel."""
import dataclasses

import numpy as np
import pytest

import oracle
from oracle.compare import assert_close
from oracle_replay import activate, default_theta
from test_gpu_option_capacity import _follow_windows, stripe_theta
from test_gpu_parity import (FULL_B, _check_choices, _full_agent, _full_size_vs_oracle, _gpu_run_window, _paired_agents,
                             _set_gpu_options)

pytestmark = pytest.mark.gpu

TB = 8                          # steps per table block of the sweep (SCG_WIN_TB)
OPT_TIMEOUT, MAX_EP = 40, 60    # longer than any window: terminations only where the schedule or the dynamics put them


@pytest.fixture(scope="module")
def scg():
    import skill_chaining_with_graphs_b200 as m
    m.load_library()
    return m


@pytest.fixture(scope="module")
def torch():
    import torch as t
    return t


def _windowed_twin(oag):
    """An oracle agent with Sarsa(lambda) in the fp64 forward-view form, in exactly oag's state."""
    wag = oracle.SkillChainAgent(dataclasses.replace(oag.cfg, windowed=True), oag.map)
    wag.env.reset(states=oag.env.state)
    for k in ("start_xy", "opt_s0", "active", "parents", "option", "action", "t_opt", "ep_steps"):
        setattr(wag, k, getattr(oag, k).copy())
    wag.n_active, wag.t = oag.n_active, oag.t
    for k in ("W", "theta", "trace"):
        getattr(wag.options, k)[:] = getattr(oag.options, k)
    return wag


def _check_both(got, dense, fwd, what):
    """got against the dense oracle and against the forward-view oracle, each at the suite's bar; on failure, say which."""
    fails = {}
    for name, ref in (("dense", dense), ("forward-view", fwd)):
        try:
            assert_close(got, ref, what=f"{what} against the {name} oracle")
        except AssertionError as e:
            fails[name] = str(e)
    if len(fails) == 2:
        raise AssertionError(f"{what}: fails both bars (an error of the kernel):\n" + "\n".join(fails.values()))
    if "dense" in fails:
        raise AssertionError(f"{what}: fails only the dense oracle's bar and meets the fp64 forward-view oracle's - the "
                             f"error lies in the oracle's fp32 per-step traces, not in the kernel:\n{fails['dense']}")
    if fails:
        raise AssertionError(f"{what}: fails only the fp64 forward-view oracle's bar:\n{fails['forward-view']}")


def _segments(opts, term):
    """Per env, the option segments of a window as the sweep forms them (maximal runs of steps under one option)."""
    return 1 + (opts[1:len(term)] != opts[:len(term) - 1]).sum(axis=0)


def _follow(oag, wag, pre, dl, acts, opts, term, what0=""):
    """Both oracles step through the GPU's window after it: pre-step states and termination flags bit for bit, TD errors
    element-wise, the oracle's own choices equal but for near-ties.  Returns the oracle outputs and the disagreements."""
    outs, n_dis = [], 0
    for t in range(len(term)):
        what = f"{what0}step {t}"
        assert np.array_equal(oag.env.state.view(np.uint32), pre[t].view(np.uint32)), f"{what}: pre-step state"
        assert np.array_equal(oag.action, acts[t]) and np.array_equal(oag.option, opts[t]), f"{what}: choices held"
        follow = dict(action=acts[t + 1], option=opts[t + 1])
        out, outw = oag.step(follow=follow), wag.step(follow=follow)
        assert np.array_equal(out["term"], term[t]), f"{what}: termination flags"
        assert np.array_equal(out["delta"], outw["delta"])
        assert_close(dl[t], out["delta"], what=f"{what}: TD error")
        n_dis += _check_choices(out, acts[t + 1], opts[t + 1], what)
        outs.append(out)
    return outs, n_dis


# ---- a. one window of T steps with terminations at scheduled steps ---------------------------------------------------
# (order, K, active options, T, map).  Order 3 with 2 slots in use runs the split-warp configuration (WinCfgO3Split);
# with 5 in use it no longer fits that configuration's shared-memory budget and runs WinCfg<4>.  Order 5 with 16 slots
# keeps the slots beyond the on-chip accumulator in the per-CTA slabs (the spill sweep).
_SCHED_ROWS = [(1, 2, 1, 32, "easy"), (2, 3, 1, 17, "easy"), (3, 4, 1, 16, "easy"), (3, 4, 1, 24, "easy"),
               (3, 4, 1, 32, "easy"), (3, 5, 4, 32, "easy"), (4, 2, 1, 25, "hard"), (5, 8, 3, 31, "hard"),
               (5, 16, 15, 32, "hard")]


@pytest.mark.parametrize("order,K,n_active,T,name", _SCHED_ROWS,
                         ids=[f"o{o}-k{k}-a{a}-T{t}" for o, k, a, t, _ in _SCHED_ROWS])
def test_long_window_with_scheduled_terminations(scg, torch, order, K, n_active, T, name):
    """One free-running window of exactly T steps (one step-kernel launch, then the sweep), weights frozen, the oracle
    following.  The per-env counters place the terminations: with option_timeout = 40, t_opt = 39 - j makes the option
    time out at step j, and ep_steps = 59 - j (max_episode_steps = 60) ends the episode at step j.  A quarter of the envs
    has no scheduled termination and starts in the gestating slot (pure decay unless it reaches its target), a quarter
    one option timeout, half an option timeout and an episode timeout; active options add their own terminations and
    re-selections.  The window
    starts from non-zero traces, so the carry-in and the decay over the whole window are in every env's result."""
    B = 2048 if order <= 3 else 512
    kw = dict(sync_interval=1000, option_timeout=OPT_TIMEOUT, epsilon=0.1, alpha=0.0, max_episode_steps=MAX_EP)
    oag, gag = _paired_agents(scg, torch, B, order, K, name, 17, window=T, **kw)
    theta = stripe_theta(K, n_active) if n_active > 8 else default_theta(K)
    activate(oag, theta, n_active)
    _set_gpu_options(gag, torch, theta, n_active)
    rng = np.random.default_rng(T)
    b = np.arange(B)
    j1 = (b // 4) % T                                              # option timeout at step j1
    j2 = (j1 + 1 + (b // 4) % (T - 1)) % T                         # episode timeout at step j2 != j1
    t_opt0 = np.where(b % 4 == 0, 0, OPT_TIMEOUT - 1 - j1).astype(np.int32)
    ep0 = np.where(b % 4 >= 2, MAX_EP - 1 - j2, 0).astype(np.int32)
    opt0 = np.where(b % 4 == 0, n_active, rng.integers(0, n_active + 1, B)).astype(np.int32)   # (unscheduled: gestating)
    E0 = (rng.standard_normal(oag.options.trace.shape) * 0.1).astype(np.float32)
    oag.t_opt, oag.ep_steps, oag.option = t_opt0.copy(), ep0.copy(), opt0.copy()
    oag.options.trace[:] = E0
    gag.t_opt.copy_(torch.as_tensor(t_opt0))
    gag.ep_steps.copy_(torch.as_tensor(ep0))
    gag.option.copy_(torch.as_tensor(opt0))
    gag.options._trace.copy_(torch.as_tensor(E0))
    gag.invalidate()
    wag = _windowed_twin(oag)

    pre, dl, acts, opts, term = _gpu_run_window(gag, torch, T)
    assert int(gag._struct.win_len) == 0                           # the whole window was swept
    ev_len = int(gag._struct.ev_len)
    assert ev_len == T
    ev = gag.ev_hist[:T].cpu().numpy()
    outs, n_dis = _follow(oag, wag, pre, dl, acts, opts, term)
    assert n_dis <= B * T // 200
    for t, out in enumerate(outs):                                 # event bytes: TERM | HIT | option of the step
        want = np.where(out["term"], 0x80 | np.where(out["hit"], 0x40, 0) | opts[t], 0).astype(np.uint8)
        assert np.array_equal(ev[t], want), f"event bytes of step {t}"

    # the schedule happened: terminations at every step index, segments across every block boundary, option changes
    # right at the boundaries, envs without any termination and envs with several
    n_term = term.sum(axis=0)
    for t in range(T):
        assert term[t].sum() >= 4, f"terminations at step {t}: {term[t].sum()}"
    for edge in range(TB, T, TB):
        assert (~term[edge - 1]).sum() >= 16, f"segments across the boundary of steps {edge - 1} -> {edge}"
        assert (opts[edge] != opts[edge - 1]).any(), f"option changes at the boundary {edge - 1} -> {edge}"
    assert (n_term == 0).sum() >= 8 and (n_term >= 2).sum() >= 8 and (n_term >= 3).any()
    assert _segments(opts, term).max() >= 3

    for x in (oag, wag):
        assert np.array_equal(gag.state.cpu().numpy().view(np.uint32), x.env.state.view(np.uint32))
    assert np.array_equal(gag.t_opt.cpu().numpy(), oag.t_opt) and np.array_equal(gag.ep_steps.cpu().numpy(), oag.ep_steps)
    assert np.array_equal(gag.n_success.cpu().numpy(), oag.n_success) and np.array_equal(gag.n_fail.cpu().numpy(), oag.n_fail)
    assert np.array_equal(gag.ex_count.cpu().numpy(), oag.ex_count)          # (the read runs the ring pass)
    assert np.array_equal(gag.ex_xy.cpu().numpy().view(np.uint32), oag.ex_xy.view(np.uint32))
    assert np.array_equal(gag.ex_label.cpu().numpy(), oag.ex_label)
    wag.options.flush()
    assert np.array_equal(gag.options.cnt.cpu().numpy(), oag.options.cnt)
    assert np.array_equal(wag.options.cnt, oag.options.cnt) and int(oag.options.cnt.sum()) == B * T
    _check_both(gag.options.trace.cpu().numpy(), oag.options.trace, wag.options.trace, f"T = {T}: traces")
    _check_both(gag.options.dW.cpu().numpy(), oag.options.dW, wag.options.dW, f"T = {T}: dW")


# ---- b. many segments per env -------------------------------------------------------------------------------------
def test_long_window_with_a_segment_per_step(scg, torch):
    """T = 32 with option_timeout = 1: every option ends after one step, and the top-level learner with epsilon_top = 1
    re-selects among all 8 slots (7 active options whose initiation sets hold everywhere, and the gestating one), so the
    option changes at most steps and an env's window has up to 32 segments (seg_o, mask of the sweep's control block).
    Every env-step is also a termination event of the top-level learner: k_top's update over 32 x B events."""
    order, K, n_active, B, T = 3, 8, 7, 2048, 32
    kw = dict(sync_interval=1000, option_timeout=1, epsilon=0.1, alpha=0.0, max_episode_steps=MAX_EP, top_level=True,
              alpha_top=1e-3, epsilon_top=1.0)
    oag, gag = _paired_agents(scg, torch, B, order, K, "easy", 23, window=T, **kw)
    oag.opt_s0 = oag.env.state.copy()
    theta = np.zeros((K, 6), dtype=np.float32)
    activate(oag, theta, n_active)
    _set_gpu_options(gag, torch, theta, n_active)
    opt0 = np.random.default_rng(4).integers(0, n_active + 1, B).astype(np.int32)
    oag.option = opt0.copy()
    gag.option.copy_(torch.as_tensor(opt0))
    gag.invalidate()
    wag = _windowed_twin(oag)
    pre, dl, acts, opts, term = _gpu_run_window(gag, torch, T)
    top = gag.win_top[:T].cpu().numpy()                            # (T, B, 8): s0, delta_top, option
    assert int(gag._struct.win_len) == 0
    outs, n_dis = _follow(oag, wag, pre, dl, acts, opts, term)
    assert n_dis <= B * T // 200
    assert term.all()                                              # a termination at every env-step
    for t, out in enumerate(outs):
        assert_close(top[t, :, 4], out["delta_top"], what=f"step {t}: top-level TD error")
    seg = _segments(opts, term)
    assert seg.max() >= 24, f"largest segment count {seg.max()}"
    wag.options.flush()
    assert np.array_equal(gag.options.cnt.cpu().numpy(), oag.options.cnt)
    assert int(oag.options.cnt[K:].min()) == B * T                 # every top-level slot counts every event
    gdW = gag.options.dW.cpu().numpy()
    _check_both(gdW[K:], oag.options.dW[K:], wag.options.dW[K:], "top-level rows of dW")
    _check_both(gdW[:K], oag.options.dW[:K], wag.options.dW[:K], "option rows of dW")
    _check_both(gag.options.trace.cpu().numpy(), oag.options.trace, wag.options.trace, "traces")


# ---- c. long windows across applies --------------------------------------------------------------------------------
# (window, sync_interval, run() lengths).  w32-s32: one 32-step launch and one 32-step sweep per apply.  w32-s20: the
# sync ends windows of 20 steps, and a read in the middle of an interval sweeps a partial window of 12 (then one of 8).
# w13-s40: windows of 13, 13, 13 and 1 per apply, so the trace is carried from the multi-block sweep into the
# single-block one and back.
_APPLY_ROWS = {"w32-s32": (32, 32, [32, 32, 32, 1]), "w32-s20": (32, 20, [20, 12, 8, 20, 1]),
               "w13-s40": (13, 40, [13, 13, 13, 1] * 3 + [1])}


@pytest.mark.parametrize("order,K,n_active,name,B", [(3, 4, 2, "easy", 3000), (5, 8, 3, "hard", 500)],
                         ids=["o3-k4", "o5-k8"])
@pytest.mark.parametrize("sched", list(_APPLY_ROWS))
def test_long_windows_across_applies(scg, torch, sched, order, K, n_active, name, B):
    """The fused pipeline over three applies with long windows, alpha > 0: the GPU runs free, the oracle follows; pre-step
    states bit for bit and TD errors at every step, W after every apply, and at the end (and where a read sweeps a
    partial window) cnt, traces and dW."""
    window, sync, runs = _APPLY_ROWS[sched]
    kw = dict(sync_interval=sync, option_timeout=5, epsilon=0.1, alpha=2e-3, max_episode_steps=9)
    oag, gag = _paired_agents(scg, torch, B, order, K, name, 13, window=window, **kw)
    theta = default_theta(K)
    activate(oag, theta, n_active)
    _set_gpu_options(gag, torch, theta, n_active)
    opt0 = np.random.default_rng(3).integers(0, n_active + 1, B).astype(np.int32)
    oag.option = opt0.copy()
    gag.option.copy_(torch.as_tensor(opt0))
    gag.invalidate()
    W0 = oag.options.W.copy()
    n_dis, n_term, n_apply = 0, 0, 0
    for i, n in enumerate(runs):
        d, m = _follow_windows(oag, gag, torch, [n], W0, what0=f"run {i}: ")
        n_dis, n_term = n_dis + d, n_term + m
        if int(gag._struct.window_steps) == 0:
            n_apply += 1
            assert np.abs(oag.options.W - W0).max() > 1e-3                 # the applies really moved the weights
        elif n == 12:                                                        # the read sweeps the open partial window
            assert_close(gag.options.dW.cpu().numpy(), oag.options.dW, what=f"run {i}: dW of the partial window")
            assert_close(gag.options.trace.cpu().numpy(), oag.options.trace, what=f"run {i}: traces")
            assert int(gag._struct.win_len) == 0
    assert n_apply == 3 and int(gag._struct.window_steps) == 1
    assert n_term > B and n_dis <= B * sum(runs) // 500
    assert np.array_equal(gag.options.cnt.cpu().numpy(), oag.options.cnt)
    assert_close(gag.options.trace.cpu().numpy(), oag.options.trace, what="traces")
    assert_close(gag.options.dW.cpu().numpy(), oag.options.dW, what="dW of the open window")
    assert np.array_equal(gag.t_opt.cpu().numpy(), oag.t_opt) and np.array_equal(gag.ep_steps.cpu().numpy(), oag.ep_steps)


# ---- d. full size --------------------------------------------------------------------------------------------------
def test_full_size_long_window_length_invariance(scg, torch):
    """configs[1] size (65,536 envs): the same 32 steps swept with windows of 1 (the dense per-step form), 13, 16, 24
    and 32 steps give the same states bit for bit and the same traces and dW to 1e-4 of their maximum (weights
    frozen: the forward-view sweep is exact for any window length)."""
    ref = None
    for window in (1, 13, 16, 24, 32):
        ag = _full_agent(scg, torch, FULL_B, 0, window=window)
        ag.run(32)
        tr, dW, st = ag.options.trace.clone(), ag.options.dW.clone(), ag.s.clone()
        assert int(ag._struct.win_len) == 0
        del ag
        if ref is None:
            ref = (tr, dW, st)
            continue
        assert torch.equal(st, ref[2]), f"window {window}: states"
        assert float((tr - ref[0]).abs().max()) <= 1e-4 * max(1.0, float(ref[0].abs().max())), f"window {window}: traces"
        assert float((dW - ref[1]).abs().max()) <= 1e-4 * max(1.0, float(ref[1].abs().max())), f"window {window}: dW"


def test_window32_at_scale_vs_oracle(scg, torch):
    """A 32-step window of 16,384 envs (hard map, order 5, 8 option slots, 3 active) in one launch, then the sweep and the
    apply, against the sharded oracle replay; the event history runs at its minimum of two windows (64 steps)."""
    _full_size_vs_oracle(scg, torch, "hard", 16384, 5, 8, 3, 32, 2048)


# ---- e. determinism and launch geometry at window 32 ----------------------------------------------------------------
def _det_agents(scg, torch, n, **kw):
    ags = []
    for _ in range(n):
        _, gag = _paired_agents(scg, torch, 2048, 3, 4, "easy", 5, **kw)
        _set_gpu_options(gag, torch, default_theta(4), 2)
        gag.invalidate()
        ags.append(gag)
    return ags


def test_window32_run_equals_step_loop_deterministic(scg, torch):
    """deterministic=True, window 32, a sync every 32 steps: run(64) (two 32-step launches), 64 step() calls and a second
    run(64) give the same states, actions, W and traces bit for bit."""
    a, b, c = _det_agents(scg, torch, 3, sync_interval=32, window=32, epsilon=0.05, option_timeout=6, alpha=5e-3,
                          deterministic=True)
    W0 = a.options.W.clone()
    a.run(64)
    for _ in range(64):
        b.step()
    c.run(64)
    torch.cuda.synchronize()
    assert a.t == b.t == c.t == 64
    for x, what in ((b, "step loop"), (c, "second run")):
        assert torch.equal(a.s, x.s) and torch.equal(a.action, x.action), what
        assert torch.equal(a.options.W, x.options.W) and torch.equal(a.options.trace, x.options.trace), what
    assert float((a.options.W - W0).abs().max()) > 1e-4


def test_window32_run_host_equals_run(scg, torch):
    """run_host with 32-step calls == the device-resident run at window 32: states and actions bit for bit, W to 1e-5
    (run_host re-evaluates Q_o(s, a) at the start of every call instead of carrying it)."""
    a, b = _det_agents(scg, torch, 2, sync_interval=32, window=32, epsilon=0.05, option_timeout=6, alpha=5e-3)
    hs, ha = b.s.cpu().numpy().copy(), b.action.cpu().numpy().copy()
    for _ in range(2):
        a.run(32)
        hs, ha, r, f, d = b.run_host(hs, ha, 32)
    assert np.array_equal(hs, a.s.cpu().numpy()) and np.array_equal(ha, a.action.cpu().numpy())
    assert float((a.options.W - b.options.W).abs().max()) <= 1e-5 * max(1.0, float(a.options.W.abs().max()))


# ---- f. the device logs at window 32 --------------------------------------------------------------------------------
def test_logs_at_window32_match_oracle(scg, torch):
    """One 64-step run at window 32 (two 32-step launches and sweeps, the event history at its minimum of 64 steps) with
    the episode, option and trajectory logs on: each log equals the oracle's record for record."""
    from test_gpu_trajectory_log import EP_KEYS, OPT_KEYS, _pair, _same
    B, K = 512, 4
    envs = sorted(set(range(0, B, 5)) | {1, 2, B - 1})
    kw = dict(sync_interval=32, option_timeout=6, epsilon=1.0, alpha=1e-3, max_episode_steps=14,
              gestation_successes=10 ** 9, window=32, init_horizon=3)
    oag, gag = _pair(scg, torch, B, K, 41, 1 << 16, envs, active=2, episode_log=1 << 16, option_log=1 << 16, **kw)
    assert gag.win_cap == 32 and gag.ev_cap == 64
    gag.run(64)
    for _ in range(64):
        oag.step()
    traj, opt, ep = oag.trajectory_log(), oag.option_log(), oag.episode_log()
    _same(gag.trajectories(), traj, "trajectory log", delta=True)
    _same(gag.option_executions(), opt, "option log", keys=OPT_KEYS)
    _same(gag.episodes(), ep, "episode log", keys=EP_KEYS)
    assert len(traj["step"]) == 64 * len(envs)
    for log in (opt, ep):                                          # records from both windows
        assert (log["step"] < 32).any() and (log["step"] >= 32).any()
    for k in ("term", "label", "episode_end", "goal"):
        assert traj[k].any() and not traj[k].all(), k
