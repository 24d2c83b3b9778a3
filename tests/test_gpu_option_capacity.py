"""Option capacity: every option-slot count the interface accepts trains, at every Fourier order and batch size.

At order 5 one option slot's dW accumulator takes 25,920 bytes, so a CTA's shared memory holds eight of them; the window
sweep accumulates the slots beyond in its own global slab.  The top-level learner's update walks each CTA's chunk of the
event bytes in bounded rounds, so its shared memory does not grow with B * win_len.  Each test here runs a shape that
needs one of the two, against the CPU oracle.
"""
import numpy as np
import pytest

import oracle
from oracle.compare import assert_close

from test_gpu_parity import _check_choices, _gpu_run_window, _paired_agents, _set_gpu_options, _states
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


def stripe_theta(K, n):
    """Initiation classifiers of n options (n <= 15): disjoint stripes a_k <= x <= b_k across the map, written as the
    quadratic -(x - a)(x - b) >= 0, scaled so that the logit is 4 at a stripe's centre."""
    theta = np.zeros((K, 6), dtype=np.float32)
    edges = np.linspace(0.05, 0.95, n + 1)
    for k in range(n):
        a, b = edges[k], edges[k + 1]
        s = 4.0 / ((b - a) / 2) ** 2
        theta[k] = [-s * a * b, s * (a + b), 0.0, -s, 0.0, 0.0]
    return theta


def _uniform_options(oag, gag, torch, n_used, B, seed=3):
    opt0 = np.random.default_rng(seed).integers(0, n_used, B).astype(np.int32)
    if oag is not None:
        oag.option = opt0.copy()
    gag.option.copy_(torch.as_tensor(opt0))


# ---- window sweep: slots beyond the shared accumulator --------------------------------------------------------------
@pytest.mark.parametrize("K,window,n_active", [(9, 8, 8), (12, 8, 11), (16, 12, 15)],
                         ids=["k9-T8", "k12-T8", "k16-T12-multi"])
def test_spilled_window_sweep_equals_oracle_dense_traces(scg, torch, K, window, n_active):
    """One window of fused steps with frozen weights at order 5 with k_used = n_active + 1 > 8 option slots: the
    slots 8 .. k_used-1 accumulate in global memory.  Traces and dW element-wise, cnt bit for bit, and every slot in use
    (the spilled ones included) has steps."""
    order, name, B = 5, "hard", 700
    kw = dict(sync_interval=1000, option_timeout=5, epsilon=0.5, alpha=0.0, max_episode_steps=11)
    oag, gag = _paired_agents(scg, torch, B, order, K, name, 7, window=window, **kw)
    theta = stripe_theta(K, n_active)
    activate(oag, theta, n_active)
    _set_gpu_options(gag, torch, theta, n_active)
    _uniform_options(oag, gag, torch, n_active + 1, B)
    gag.invalidate()
    out = None
    for t in range(window):
        out = oag.step()
        gag.step()
        # with eps = 0.5 most actions are exploratory (identical draws); follow the oracle's choices exactly
        gag.action.copy_(torch.as_tensor(out["action"]))
        gag.option.copy_(torch.as_tensor(out["option"]))
        gag.invalidate()
        assert np.array_equal(gag.state.cpu().numpy().view(np.uint32), out["state"].view(np.uint32))
        assert_close(gag.delta.cpu().numpy(), out["delta"], what=f"TD error, step {t}")
    assert int(gag._struct.win_len) == 0                                    # the full window was swept
    assert np.array_equal(gag.options.cnt.cpu().numpy(), oag.options.cnt)
    assert (oag.options.cnt[:n_active + 1] > 0).all()                       # every slot in use has steps
    assert_close(gag.options.trace.cpu().numpy(), oag.options.trace, what="traces")
    assert_close(gag.options.dW.cpu().numpy(), oag.options.dW, what="dW")
    assert np.abs(oag.options.dW[8:n_active + 1]).max() > 0                 # the spilled slots carry weight deltas
    assert oag.n_fail.sum() + oag.n_success.sum() > B // 4


# ---- the dense operator over all K slots ----------------------------------------------------------------------------
@pytest.mark.parametrize("K,top_slots", [(12, 0), (16, 0), (8, 2)])
def test_dense_update_with_spilled_slots_matches_oracle(scg, torch, K, top_slots):
    """OptionSet.update at order 5 sweeps all K_all slots: more than fit a CTA's shared accumulator.  Several updates
    with a sync every 2: TD errors, traces, cnt, dW and W as in test_sarsa_updates_match_oracle."""
    order, B = 5, 257
    omap = oracle.PinballMap.from_name("easy")
    rng = np.random.default_rng(200 + K)
    hp = dict(gamma=0.95, lam=0.8, alpha=0.05, seed=1, top_slots=top_slots)
    oset = oracle.OptionSet(K, order, B, **hp)
    gset = scg.OptionSet(K, order, B, **hp)
    assert gset.K_all == K + top_slots > 8
    W = (rng.standard_normal(oset.W.shape) * 0.05).astype(np.float32)
    oset.W[:] = W
    gset.set_weights(W)
    for it in range(6):
        S, A = _states(omap, B, seed=20 + it)
        S2, A2 = _states(omap, B, seed=40 + it)
        opt = rng.integers(0, K, B).astype(np.int32)
        r = rng.standard_normal(B).astype(np.float32)
        done = rng.random(B) < 0.15
        mask = None if it % 2 == 0 else (rng.random(B) < 0.8)
        od = oset.update(S, A, r, S2, A2, done, opt, mask=mask)
        gd = gset.update(S, A, r, S2, A2, done, opt, mask=mask).cpu().numpy()
        oset.tick(); gset.tick()
        assert_close(gd, od, what=f"TD error, update {it}")
        assert_close(gset.trace.cpu().numpy(), oset.trace, what=f"trace, update {it}")
        assert np.array_equal(gset.cnt.cpu().numpy(), oset.cnt), f"cnt, update {it}"
        assert_close(gset.dW.cpu().numpy(), oset.dW, what=f"dW, update {it}")
        if it % 2 == 1:
            oset.apply(); gset.apply()
            assert_close(gset.W.cpu().numpy(), oset.W, what=f"W after apply, update {it}")
            assert float(gset.dW.abs().max()) == 0.0 and int(gset.cnt.sum()) == 0
    S, _ = _states(omap, B, seed=99)
    opt = rng.integers(0, K, B).astype(np.int32)
    assert_close(gset.q(S, opt).cpu().numpy(), oset.q(S, opt))


# ---- the fused pipeline across applies ------------------------------------------------------------------------------
def _follow_windows(oag, gag, torch, windows, W0, what0=""):
    """Run the GPU agent free for the given window lengths (one launch each, the syncs inside scg_agent_run) and let the
    oracle follow its choices: pre-step states bit for bit, TD errors, W after every apply.  Returns the near-tie
    action disagreements and the terminations."""
    n_dis, n_term = 0, 0
    for w, n in enumerate(windows):
        pre, dl, acts, opts, term = _gpu_run_window(gag, torch, n)
        for t in range(n):
            what = f"{what0}window {w} step {t}"
            assert np.array_equal(oag.env.state.view(np.uint32), pre[t].view(np.uint32)), f"{what}: pre-step state"
            assert np.array_equal(oag.action, acts[t]) and np.array_equal(oag.option, opts[t])
            out = oag.step(follow=dict(action=acts[t + 1], option=opts[t + 1]))
            assert np.array_equal(out["term"], term[t]), f"{what}: termination flags"
            assert_close(dl[t], out["delta"], what=f"{what}: TD error")
            n_dis += _check_choices(out, acts[t + 1], opts[t + 1], what)
            n_term += int(out["term"].sum())
        assert np.array_equal(gag.state.cpu().numpy().view(np.uint32), oag.env.state.view(np.uint32))
        if int(gag._struct.window_steps) == 0:                              # this window ended with an apply
            assert_close(gag.options.W.cpu().numpy(), oag.options.W, what=f"{what0}W after window {w}")
            assert_close(gag.options.W.cpu().numpy() - W0, oag.options.W - W0, what=f"{what0}W - W0 after window {w}")
    return n_dis, n_term


@pytest.mark.parametrize("deterministic", [False, True], ids=["fast", "deterministic"])
def test_fused_pipeline_with_spilled_slots_across_applies(scg, torch, deterministic):
    """Order 5, 12 option slots, 10 active (11 in use): k_agent_step -> spill sweep -> k_reduce -> k_apply, 13 steps
    with a sync every 4, the oracle following.  deterministic: a second agent runs the same windows and must give the
    same bits in W and the traces."""
    order, K, n_active, name, B = 5, 12, 10, "hard", 500
    kw = dict(sync_interval=4, option_timeout=5, epsilon=0.1, alpha=5e-3, max_episode_steps=9,
              deterministic=deterministic)
    oag, gag = _paired_agents(scg, torch, B, order, K, name, 13, window=4, **kw)
    theta = stripe_theta(K, n_active)
    activate(oag, theta, n_active)
    _set_gpu_options(gag, torch, theta, n_active)
    _uniform_options(oag, gag, torch, n_active + 1, B)
    gag.invalidate()
    W0 = oag.options.W.copy()
    windows = [4, 4, 4, 1]
    n_dis, n_term = _follow_windows(oag, gag, torch, windows, W0)
    assert np.abs(oag.options.W - W0)[8:n_active + 1].max() > 1e-4         # the spilled slots really learned
    assert n_term > B // 2 and n_dis <= B // 50
    assert np.array_equal(gag.options.cnt.cpu().numpy(), oag.options.cnt)
    assert_close(gag.options.trace.cpu().numpy(), oag.options.trace, what="traces")
    assert_close(gag.options.dW.cpu().numpy(), oag.options.dW, what="dW of the open window")
    if deterministic:
        _, twin = _paired_agents(scg, torch, B, order, K, name, 13, window=4, **kw)
        _set_gpu_options(twin, torch, theta, n_active)
        _uniform_options(None, twin, torch, n_active + 1, B)
        twin.invalidate()
        for n in windows:
            twin.run(n)
        torch.cuda.synchronize()
        assert torch.equal(twin.options.W, gag.options.W)
        assert torch.equal(twin.options.trace, gag.options.trace)


# ---- a promotion past the eighth option on the device ---------------------------------------------------------------
def test_device_promotes_the_ninth_option_and_keeps_training(scg, torch):
    """Order 5, 12 slots, 8 active options set from the host: the gestating slot 8 is given enough successes and
    examples, and scg_agent_manage promotes it on the device.  The next windows use 10 option slots (9 active and the
    new gestating slot), more than the shared accumulator holds: flush and apply must run, and the windows must match
    the oracle replayed in follow mode with the device-fitted classifiers."""
    order, K, n_active, name, B = 5, 12, 8, "hard", 500
    kw = dict(sync_interval=4, option_timeout=5, epsilon=0.1, alpha=5e-3, max_episode_steps=9, gestation_successes=10,
              clf_steps=100, clf_lr=2.0)
    oag, gag = _paired_agents(scg, torch, B, order, K, name, 31, window=4, **kw)
    theta = stripe_theta(K, n_active)
    _set_gpu_options(gag, torch, theta, n_active)
    rng = np.random.default_rng(8)
    n = 2000
    X = rng.random((n, 2)).astype(np.float32)
    y = ((X[:, 0] > 0.4) & (X[:, 0] < 0.6)).astype(np.uint8)
    gag._ex_xy[n_active, :n].copy_(torch.as_tensor(X))
    gag._ex_label[n_active, :n].copy_(torch.as_tensor(y))
    gag._ex_count[n_active] = n
    gag.n_success[n_active] = 1000
    assert gag.manage(wait=True) is True
    c = gag.controller_state()
    assert c["n_active"] == gag.n_active == n_active + 1 == 9
    dev_theta = gag.options.theta.cpu().numpy()
    assert np.abs(dev_theta[n_active]).max() > 0                            # the promoted option was fitted
    activate(oag, dev_theta, n_active + 1)
    assert c["parents"] == [int(v) for v in oag.parents]
    _uniform_options(oag, gag, torch, n_active + 2, B)
    gag.invalidate()
    W0 = oag.options.W.copy()
    n_dis, n_term = _follow_windows(oag, gag, torch, [4, 4], W0)
    assert int(gag._struct.window_steps) == 0
    assert np.abs(oag.options.W - W0)[8:n_active + 2].max() > 1e-4
    assert n_term > B // 4 and n_dis <= B // 50


# ---- the top-level learner ------------------------------------------------------------------------------------------
def test_top_level_learner_with_many_slots_matches_oracle(scg, torch):
    """Order 5, 12 option slots (3 top-level slots, K_all = 15), 10 active: option and top-level TD errors per step,
    and every weight slot after every apply, against the oracle following the GPU's choices."""
    order, K, n_active, name, B = 5, 12, 10, "hard", 500
    kw = dict(sync_interval=4, option_timeout=4, epsilon=0.1, alpha=5e-3, max_episode_steps=9,
              top_level=True, alpha_top=1e-3, epsilon_top=0.15)
    oag, gag = _paired_agents(scg, torch, B, order, K, name, 29, window=4, **kw)
    assert gag.options.K_all == oag.options.K_all == 15
    # top-level weights of 5e-3 instead of 0.5: a window's step there is ~1e-4, and at 0.5 one float32 ulp of W (6e-8)
    # is already 4x the bar on W - W0, so any rounding of the event sum would flip it
    W = oag.options.W.copy()
    W[K:] *= 0.01
    oag.options.W[:] = W
    gag.options.set_weights(W)
    oag.opt_s0 = oag.env.state.copy()
    theta = stripe_theta(K, n_active)
    activate(oag, theta, n_active)
    _set_gpu_options(gag, torch, theta, n_active)
    _uniform_options(oag, gag, torch, n_active + 1, B)
    W0 = oag.options.W.copy()
    n_term, n_dis_o = 0, 0
    for w in range(4):
        n = 4 if w < 3 else 1
        wl0 = int(gag._struct.win_len)
        pre, dl, acts, opts, term = _gpu_run_window(gag, torch, n)
        top = gag.win_top[wl0:wl0 + n].cpu().numpy()                        # (n, B, 8): s0, delta_top, option
        for t in range(n):
            what = f"window {w} step {t}"
            assert np.array_equal(oag.env.state.view(np.uint32), pre[t].view(np.uint32)), f"{what}: pre-step state"
            s0_before, o_before = oag.opt_s0.copy(), oag.option.copy()
            out = oag.step(follow=dict(action=acts[t + 1], option=opts[t + 1]))
            assert np.array_equal(out["term"], term[t]), f"{what}: termination flags"
            assert_close(dl[t], out["delta"], what=f"{what}: TD error")
            tm = out["term"]
            if tm.any():
                assert np.array_equal(top[t, tm, :4].view(np.uint32), s0_before[tm].view(np.uint32)), f"{what}: s0"
                assert np.array_equal(top[t, tm, 5].copy().view(np.int32), o_before[tm])
                assert_close(top[t, tm, 4], out["delta_top"][tm], what=f"{what}: top-level TD error")
                dis = out["own_option"] != opts[t + 1]
                if dis.any():                                              # only at a near-tie of the oracle's Q_top row
                    Q = out["Qtop"][dis].astype(np.float64)
                    gap = Q.max(axis=1) - Q[np.arange(len(Q)), opts[t + 1][dis]]
                    fin = np.isfinite(out["Qtop"])
                    assert gap.max() <= 1e-4 * max(1e-30, float(np.abs(out["Qtop"][fin]).mean())), f"{what}: option choice"
                n_dis_o += int(dis.sum())
            _check_choices(dict(out, own_option=opts[t + 1]), acts[t + 1], opts[t + 1], what)
            n_term += int(tm.sum())
        assert np.array_equal(gag.state.cpu().numpy().view(np.uint32), oag.env.state.view(np.uint32))
        if w < 3:
            gW = gag.options.W.cpu().numpy()
            assert_close(gW[:K], oag.options.W[:K], what=f"option weights after apply {w}")
            assert_close(gW[K:] - W0[K:], oag.options.W[K:] - W0[K:], what=f"top-level weights after apply {w}")
            assert np.abs(oag.options.W[K:] - W0[K:]).max() > 1e-4
    assert n_term > B // 2 and n_dis_o <= B // 100
    assert np.array_equal(gag.options.cnt.cpu().numpy(), oag.options.cnt)


def test_top_level_update_beyond_one_event_list(scg, torch):
    """Order 3, 4 option slots with the top-level learner, 1,048,576 envs and an 8-step window: 8.4 M event bytes,
    several list rounds per CTA (and past the event list the update used to reserve in full).  One window without an
    apply; the top-level rows of dW are rebuilt from the recorded win_top rows and the window's event bytes,
    delta_top * phi(s0) summed per option in float64, and cnt[K:] is the number of events."""
    order, K, n_active, name, B, T = 3, 4, 2, "easy", 1 << 20, 8
    gmap = scg.PinballMap.from_name(name)
    cfg = scg.AgentConfig(map=name, batch=B, order=order, max_options=K, seed=5, window=T, sync_interval=1000,
                          option_timeout=4, epsilon=0.1, alpha=5e-3, top_level=True, alpha_top=1e-3, epsilon_top=0.15)
    gag = scg.SkillChainAgent(cfg, gmap)
    dev = gag.options.W.device
    gen = torch.Generator(device=dev).manual_seed(0)
    gag.options.set_weights(torch.randn(gag.options.W.shape, generator=gen, device=dev) * 0.5)
    _set_gpu_options(gag, torch, stripe_theta(K, n_active), n_active)
    _uniform_options(None, gag, torch, n_active + 1, B)
    gag.invalidate()
    assert int(gag._struct.ev_len) == 0 and int(gag._struct.win_len) == 0
    gag.run(T)                                                              # the full window is swept: k_top, k_window
    torch.cuda.synchronize()
    assert int(gag._struct.win_len) == 0 and int(gag._struct.window_steps) == T
    ev = gag.ev_hist[:T, :B]
    term = (ev & 0x80) != 0                                                 # SCG_EV_TERM
    n_ev = int(term.sum())
    assert n_ev > B                                                         # events in every list round
    top_slots = (K + 4) // 5
    C = torch.as_tensor(oracle.FourierBasis(order).C, device=dev).to(torch.float64)   # (F, 4)
    F = C.shape[0]
    want = torch.zeros((K, F), dtype=torch.float64, device=dev)
    rows = gag.win_top[:T, :B][term]                                        # (n_ev, 8): s0, delta_top, option
    for i in range(0, n_ev, 1 << 18):
        r = rows[i:i + (1 << 18)]
        s = r[:, :4].clone()
        s[:, 2:] = (s[:, 2:] + 2.0) * 0.25                                  # as the oracle: fp32, then widened
        phi = torch.cos(torch.pi * (s.to(torch.float64) @ C.T))
        o = r[:, 5].contiguous().view(torch.int32).long().clamp(0, K - 1)
        want.index_add_(0, o, r[:, 4].to(torch.float64)[:, None] * phi)
    got = gag.options.dW[K:].reshape(top_slots * 5, F)[:K]                  # row j = option j
    assert_close(got.cpu().numpy(), want.cpu().numpy(), what="top-level dW")
    assert gag.options.cnt[K:].tolist() == [n_ev] * top_slots
