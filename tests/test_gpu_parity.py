"""GPU parity: the CUDA path (through the C ABI) against the CPU oracle on the same seeded inputs.

Bars (BASELINE.json north_star): single-step transitions bit-identical in collision
(obstacle, edge) indices and terminal flags, next state within 1e-5 relative (we get bit-exact);
Q values, TD errors and classifier probabilities within 1e-4 relative after a fixed number of
updates on the same seeded transition batch.
"""
import numpy as np
import pytest

import oracle
from oracle.pinball import step_batched

pytestmark = pytest.mark.gpu

RTOL = 1e-4


from oracle.compare import assert_close  # noqa: E402  element-wise |a-b| <= rtol*|b| + rtol*typical(b)


@pytest.fixture(scope="module")
def scg():
    import skill_chaining_with_graphs_b200 as m
    m.load_library()
    return m


@pytest.fixture(scope="module")
def torch():
    import torch as t
    return t


def _states(omap, n, seed, near_walls=False):
    rng = np.random.default_rng(seed)
    S = omap.sample_free_states(rng, n)
    if near_walls:
        # concentrate positions within ~1.5 ball radii of a random edge so most steps collide
        e = omap.edges[rng.integers(0, omap.n_edges, n)]
        t = rng.uniform(0, 1, n).astype(np.float32)
        off = rng.uniform(-1.5, 1.5, n).astype(np.float32) * omap.ball_r
        S[:, 0] = e[:, 0] + t * e[:, 2] + off * e[:, 5]
        S[:, 1] = e[:, 1] + t * e[:, 3] + off * e[:, 6]
    A = rng.integers(0, 5, n).astype(np.int32)
    return S, A


# ---- K1 ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["easy", "hard"])
def test_edge_table_matches_oracle(scg, name):
    omap = oracle.PinballMap.from_name(name)
    gmap = scg.PinballMap.from_name(name)
    edges, obst, local = gmap.edge_table()
    assert np.array_equal(edges.view(np.uint32), omap.edges.view(np.uint32))
    assert np.array_equal(obst, omap.edge_obstacle)
    assert np.array_equal(local, omap.edge_local)


@pytest.mark.parametrize("name,near", [("easy", False), ("easy", True), ("hard", False), ("hard", True)])
@pytest.mark.parametrize("cull", [True, False])
def test_step_bit_exact(scg, torch, name, near, cull):
    omap = oracle.PinballMap.from_name(name)
    gmap = scg.PinballMap.from_name(name)
    B = 20000
    S, A = _states(omap, B, seed=11 + near, near_walls=near)
    env = scg.PinballEnv(gmap, B, cull=cull)
    env.reset(states=S)
    ns, r, done, hit = env.step(torch.as_tensor(A).cuda())
    ons, orr, ofl = step_batched(omap, S, A)
    odone, okind, oobst, oedge = oracle.unpack_flags(ofl)
    assert np.array_equal(env.flags.cpu().numpy(), ofl)
    assert np.array_equal(done.cpu().numpy(), odone)
    assert np.array_equal(hit.cpu().numpy(), np.stack([okind, oobst, oedge], axis=1))
    assert np.array_equal(ns.cpu().numpy().view(np.uint32), ons.view(np.uint32))
    assert np.array_equal(r.cpu().numpy(), orr)
    if near:
        assert (okind != 0).mean() > 0.2      # the case really exercises collisions


@pytest.mark.parametrize("grid_n", [8, 32, 128])
def test_step_bit_exact_at_other_grid_resolutions(scg, torch, grid_n):
    """The broad-phase grid only prunes: every resolution gives the oracle's bits (collisions, flags, next states)."""
    omap = oracle.PinballMap.from_name("hard")
    gmap = scg.PinballMap.from_name("hard", grid_n=grid_n)
    assert gmap.grid()[0] == grid_n
    B = 20000
    S, A = _states(omap, B, seed=5, near_walls=True)
    env = scg.PinballEnv(gmap, B, cull=True)
    env.reset(states=S)
    ns, r, done, hit = env.step(torch.as_tensor(A).cuda())
    ons, orr, ofl = step_batched(omap, S, A)
    assert np.array_equal(env.flags.cpu().numpy(), ofl)
    assert np.array_equal(ns.cpu().numpy().view(np.uint32), ons.view(np.uint32))
    assert np.array_equal(r.cpu().numpy(), orr)


def test_step_goal_and_bounds_cases(scg, torch):
    omap = oracle.PinballMap.from_name("easy")
    gmap = scg.PinballMap.from_name("easy")
    tx, ty, tr = (float(v) for v in omap.target)
    S = np.array([
        [tx - 0.05, ty, 1.0, 0.0],       # flies into the goal
        [tx, ty, 0.0, 0.0],              # starts inside the goal
        [1.5, 0.5, 0.0, 0.0],            # outside the unit square: clamp, brute-force edge path
        [-0.2, -0.3, 0.0, 0.0],
        [0.5, 0.5, 0.0, 0.0],            # at rest in open space
        [0.2, 0.9, 1.0, 1.0],            # start position, fast
    ], dtype=np.float32)
    for a in range(5):
        A = np.full(len(S), a, dtype=np.int32)
        env = scg.PinballEnv(gmap, len(S))
        env.reset(states=S)
        ns, r, done, hit = env.step(torch.as_tensor(A).cuda())
        ons, orr, ofl = step_batched(omap, S, A)
        assert np.array_equal(ns.cpu().numpy().view(np.uint32), ons.view(np.uint32))
        assert np.array_equal(env.flags.cpu().numpy(), ofl)
        assert np.array_equal(r.cpu().numpy(), orr)


def test_step_empty_and_bad_actions(scg, torch):
    gmap = scg.PinballMap.from_name("easy")
    env = scg.PinballEnv(gmap, 0)
    ns, r, done, hit = env.step(torch.zeros(0, dtype=torch.int32).cuda())
    assert ns.shape == (0, 4)
    env = scg.PinballEnv(gmap, 4)
    with pytest.raises(ValueError):
        env.step(torch.tensor([0, 1, 5, 2], dtype=torch.int32).cuda())
    with pytest.raises(ValueError):
        env.step(torch.tensor([0, 1], dtype=torch.int32).cuda())


def test_step_host_path_matches_device_path(scg, torch):
    omap = oracle.PinballMap.from_name("hard")
    gmap = scg.PinballMap.from_name("hard")
    B = 5000
    S, A = _states(omap, B, seed=5)
    env = scg.PinballEnv(gmap, B)
    env.reset(states=S)
    ns, r, done, hit = env.step(A)          # NumPy in -> host path
    ons, orr, ofl = step_batched(omap, S, A)
    assert isinstance(ns, np.ndarray)
    assert np.array_equal(ns.view(np.uint32), ons.view(np.uint32))
    assert np.array_equal(r, orr)


def test_step_trajectory_roundtrip_many_steps(scg, torch):
    """50 consecutive steps: GPU and oracle stay bit-identical because each step is."""
    omap = oracle.PinballMap.from_name("easy")
    gmap = scg.PinballMap.from_name("easy")
    B = 2000
    S, _ = _states(omap, B, seed=9)
    rng = np.random.default_rng(1)
    env = scg.PinballEnv(gmap, B)
    env.reset(states=S)
    cur = S.copy()
    for t in range(50):
        A = rng.integers(0, 5, B).astype(np.int32)
        ns, r, done, hit = env.step(torch.as_tensor(A).cuda())
        cur, orr, ofl = step_batched(omap, cur, A)
        assert np.array_equal(ns.cpu().numpy().view(np.uint32), cur.view(np.uint32)), f"diverged at step {t}"


def test_reset_matches_oracle(scg, torch):
    omap = oracle.PinballMap(0.02, (0.9, 0.2, 0.04), [(0.2, 0.9), (0.5, 0.5), (0.1, 0.3)],
                             [p.tolist() for p in oracle.PinballMap.from_name("easy").polygons])
    gmap = scg.PinballMap(0.02, (0.9, 0.2, 0.04), [(0.2, 0.9), (0.5, 0.5), (0.1, 0.3)],
                          [p.tolist() for p in omap.polygons])
    B = 1000
    oenv = oracle.PinballEnv(omap, B, seed=42, env_offset=7)
    genv = scg.PinballEnv(gmap, B, seed=42, env_offset=7)
    mask = np.random.default_rng(0).random(B) < 0.5
    o = oenv.reset(mask=mask, step=5)
    g = genv.reset(mask=mask, step=5)
    assert np.array_equal(g.cpu().numpy(), o)
    assert len(np.unique(o[:, 0])) == 3


# ---- K2 ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("order", [1, 2, 3, 4, 5])
def test_features_match_oracle(scg, torch, order):
    omap = oracle.PinballMap.from_name("easy")
    S, _ = _states(omap, 512, seed=order)
    S[:, 2:] *= 1.4                                          # exercise the sqrt(2) velocity range
    phi = scg.FourierBasis(order).features(S).cpu().numpy()
    ophi = oracle.FourierBasis(order).features(S)
    assert phi.shape == ophi.shape
    assert np.abs(phi - ophi).max() < 2e-5


@pytest.mark.parametrize("order", [1, 2, 3, 4, 5])
def test_packed_weights_follow_the_documented_layout(scg, torch, order):
    """include/scg_b200.h: a slot holds its features in pairs over the last multi-index digit, 12 floats per pair
    (w0a w1a w2a w3a | w0b w1b w2b w3b | w4a w4b 0 0); an odd N1 pairs its last feature with a phantom of weight 0.
    apply keeps the packed copy current in the same layout."""
    K, B = 3, 64
    n1 = order + 1
    F, NP = n1 ** 4, (n1 + 1) // 2
    rng = np.random.default_rng(order)
    gset = scg.OptionSet(K, order, B, gamma=0.97, seed=5)
    W = rng.standard_normal((K, 5, F)).astype(np.float32)

    def packed(W):
        slot = gset.lib.scg_packed_slot_floats(order)
        out = np.zeros((K, slot), np.float32)
        for f in range(F):
            row, c3 = divmod(f, n1)
            p, h = row * NP + c3 // 2, c3 & 1
            out[:, p * 12 + h * 4: p * 12 + h * 4 + 4] = W[:, :4, f]
            out[:, p * 12 + 8 + h] = W[:, 4, f]
        return out

    gset.set_weights(W)
    assert np.array_equal(gset.Wt.cpu().numpy(), packed(W))
    # an apply with a known delta: W changes and the packed copy follows
    gset._dW.copy_(torch.as_tensor(rng.standard_normal((K, 5, F)).astype(np.float32)).cuda())
    gset._cnt.fill_(4)
    gset.window_steps = 4
    gset.apply()
    assert not np.array_equal(gset.W.cpu().numpy(), W)
    assert np.array_equal(gset.Wt.cpu().numpy(), packed(gset.W.cpu().numpy()))


@pytest.mark.parametrize("order,K", [(3, 1), (3, 4), (5, 8), (2, 3)])
def test_q_select_td_match_oracle(scg, torch, order, K):
    omap = oracle.PinballMap.from_name("easy")
    B = 3000
    rng = np.random.default_rng(order * 10 + K)
    S, A = _states(omap, B, seed=3)
    S2, A2 = _states(omap, B, seed=4)
    opt = rng.integers(0, K, B).astype(np.int32)
    oset = oracle.OptionSet(K, order, B, gamma=0.97, seed=5, env_offset=100, epsilon=0.3)
    gset = scg.OptionSet(K, order, B, gamma=0.97, seed=5, env_offset=100, epsilon=0.3)
    W = (rng.standard_normal(oset.W.shape) * 0.05).astype(np.float32)
    oset.W[:] = W
    gset.set_weights(W)
    oQ = oset.q(S, opt)
    gQ = gset.q(S, opt).cpu().numpy()
    assert_close(gQ, oQ)
    # selection: identical uniforms; feed the ORACLE's Q so argmax cannot flip on rounding
    oa = oracle.option.epsilon_greedy(oQ, oset.epsilon, 5, oset.env_ids, 17, 0)
    ga = gset.select(torch.as_tensor(oQ).cuda(), 17, 0).cpu().numpy()
    assert np.array_equal(ga, oa)
    r = rng.standard_normal(B).astype(np.float32)
    done = rng.random(B) < 0.2
    od = oset.td_error(S, A, r, S2, A2, done, opt)
    gd = gset.td_error(S, A, r, S2, A2, done, opt).cpu().numpy()
    assert_close(gd, od)


# ---- K3 ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("order,K", [(3, 4), (3, 8), (1, 2), (2, 2), (4, 2), (5, 8)])
def test_sarsa_updates_match_oracle(scg, torch, order, K):
    """N updates on a fixed seeded transition batch with a sync every 2 steps: Q values, TD errors,
    traces, dW and weights all within 1e-4 relative of the oracle."""
    omap = oracle.PinballMap.from_name("easy")
    B = 257 if order >= 4 else 1500
    rng = np.random.default_rng(100 + order)
    hp = dict(gamma=0.95, lam=0.8, alpha=0.05, seed=1)
    oset = oracle.OptionSet(K, order, B, **hp)
    gset = scg.OptionSet(K, order, B, **hp)
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


def test_sarsa_b1_classical(scg, torch):
    """B = 1, sync every step: the classical Sarsa(lambda) rule."""
    omap = oracle.PinballMap.from_name("easy")
    hp = dict(gamma=0.9, lam=0.7, alpha=0.1, seed=1)
    oset = oracle.OptionSet(1, 3, 1, **hp)
    gset = scg.OptionSet(1, 3, 1, **hp)
    gset.pack()
    for it in range(5):
        S, A = _states(omap, 1, seed=it)
        S2, A2 = _states(omap, 1, seed=50 + it)
        r = np.array([-1.0 - it], dtype=np.float32)
        done = np.array([it == 4])
        o = np.zeros(1, dtype=np.int32)
        od = oset.update(S, A, r, S2, A2, done, o)
        gd = gset.update(S, A, r, S2, A2, done, o).cpu().numpy()
        oset.tick(); gset.tick(); oset.apply(); gset.apply()
        assert_close(gd, od)
        assert_close(gset.W.cpu().numpy(), oset.W)
    assert float(gset.trace.abs().max()) == 0.0      # done on the last update zeroed the trace


# ---- K4 ------------------------------------------------------------------------------------------
def test_classifier_eval_grad_fit_match_oracle(scg, torch):
    rng = np.random.default_rng(8)
    K, B = 4, 4000
    oset = oracle.OptionSet(K, 1, 1)
    gset = scg.OptionSet(K, 1, 1)
    theta = rng.standard_normal((K, 6)).astype(np.float32) * 2
    oset.theta[:] = theta
    gset.theta.copy_(torch.as_tensor(theta))
    S = rng.random((B, 4)).astype(np.float32)
    assert_close(gset.initiation_prob(S).cpu().numpy(), oset.initiation_prob(S))
    X = rng.random((1000, 2)).astype(np.float32)
    y = ((X[:, 0] - 0.6) ** 2 + (X[:, 1] - 0.4) ** 2 < 0.08).astype(np.uint8)
    assert_close(gset.clf_grad(2, X, y).cpu().numpy(), oset.clf_grad(2, X, y))
    oset.theta[1] = 0
    gset.theta[1].zero_()
    ot = oset.fit_initiation(1, X, y, steps=150, lr=2.0)
    gt = gset.fit_initiation(1, X, y, steps=150, lr=2.0).cpu().numpy()
    assert_close(gt, ot)
    op = oset.initiation_prob(np.concatenate([X, np.zeros_like(X)], axis=1))[:, 1]
    gp = gset.initiation_prob(np.concatenate([X, np.zeros_like(X)], axis=1))[:, 1].cpu().numpy()
    assert_close(gp, op)


def test_initiation_decisions_bit_identical_including_boundary_states(scg, torch):
    """I_k(s) is decided on the fp32 logit with the oracle's operation order: identical decisions for random states,
    for states exactly on a classifier's edge (x = 0.2 with theta = (2, -10, ...): the easy map's start position) and
    for states one ulp either side of it."""
    from oracle_replay import default_theta
    K = 8
    theta = default_theta(K)
    rng = np.random.default_rng(12)
    theta[6:] = rng.standard_normal((2, 6)).astype(np.float32) * 3
    oset, gset = oracle.OptionSet(K, 1, 1), scg.OptionSet(K, 1, 1)
    oset.theta[:] = theta
    gset.theta.copy_(torch.as_tensor(theta))
    S = rng.random((200000, 4)).astype(np.float32)
    edge = np.float32(0.2)
    S[:3000, 0] = np.nextafter(edge, np.float32(rng.choice([0, 1])), dtype=np.float32)
    S[3000:6000, 0] = edge
    S[6000:9000, 1] = np.float32(0.45)                       # theta[1] = (4.5, 0, -10): y <= 0.45
    S[9000:12000, 0] = np.float32(0.6)                       # theta[0] = (-6, 10): x >= 0.6
    # points on the disc's boundary (quadratic terms) by bisection of the oracle's own logit along rays
    for i in range(12000, 13000):
        lo, hi = np.float32(0.5), np.float32(1.0)
        for _ in range(40):
            mid = np.float32((lo + hi) / 2)
            inside = oset.initiation_logit(np.array([[mid, 0.5, 0, 0]], dtype=np.float32))[0, 5] >= 0
            lo, hi = (mid, hi) if inside else (lo, mid)
        S[i, 0], S[i, 1] = (lo if i % 2 else hi), 0.5
    want = oset.initiation(S)
    got = gset.initiation(S).cpu().numpy()
    assert np.array_equal(got, want)
    z = oset.initiation_logit(S)
    assert (np.abs(z) < 1e-6).sum() > 3000                   # the set really contains boundary cases


# ---- fused agent step ------------------------------------------------------------------------------
def _paired_agents(scg, torch, B, order, K, name, seed, **kw):
    omap = oracle.PinballMap.from_name(name)
    gmap = scg.PinballMap.from_name(name)
    cfg = dict(map=name, batch=B, order=order, max_options=K, seed=seed, **kw)
    S, A = _states(omap, B, seed=seed)
    gpu_only = ("deterministic", "window", "cull", "sync_backend", "event_history", "sync_timeout_s")
    oag = oracle.SkillChainAgent(oracle.AgentConfig(**{k: v for k, v in cfg.items() if k not in gpu_only}), omap)
    oag.env.reset(states=S)
    oag.start_xy = oag.env.state[:, :2].copy()
    gag = scg.SkillChainAgent(scg.AgentConfig(**cfg), gmap, initial_states=S)
    rng = np.random.default_rng(seed)
    W = (rng.standard_normal(oag.options.W.shape) * 0.5).astype(np.float32)
    oag.options.W[:] = W
    gag.options.set_weights(W)
    oag.action = A.copy()
    gag.action.copy_(torch.as_tensor(A))
    return oag, gag


@pytest.mark.parametrize("cull", [True, False])
def test_agent_step_matches_oracle_one_step(scg, torch, cull):
    """One fused step from identical state and weights, with two active options so termination,
    option reward, example recording, reset and re-selection all fire.  cull: broad-phase grid or every edge - both
    must give the oracle's bits."""
    B, K = 6000, 4
    oag, gag = _paired_agents(scg, torch, B, 3, K, "easy", 2, sync_interval=3, option_timeout=3, epsilon=0.2, cull=cull)
    theta = np.zeros((K, 6), dtype=np.float32)
    theta[0] = [-1.0, 2.0, 0.0, 0.0, 0.0, 0.0]       # x >= 0.5
    theta[1] = [-0.6, 0.0, 2.0, 0.0, 0.0, 0.0]       # y >= 0.3
    for ag_active in (oag,):
        ag_active.options.theta[:] = theta
        ag_active.active[:2] = True
        ag_active.n_active = 2
        ag_active.parents[1] = 1
        ag_active.parents[2] = 2
    gag.options.theta.copy_(torch.as_tensor(theta))
    gag.active_mask, gag.n_active = 3, 2
    gag.parents_host[1], gag.parents_host[2] = 1, 2
    gag._push_parents()
    rng = np.random.default_rng(0)
    opt = rng.integers(0, 3, B).astype(np.int32)
    oag.option = opt.copy()
    gag.option.copy_(torch.as_tensor(opt))
    tq = rng.integers(0, 3, B).astype(np.int32)      # some envs are at the option timeout
    oag.t_opt = tq.copy()
    gag.t_opt.copy_(torch.as_tensor(tq))
    out = oag.step()
    gag.step()
    torch.cuda.synchronize()
    assert_close(gag.delta.cpu().numpy(), out["delta"])
    assert np.array_equal(gag.state.cpu().numpy().view(np.uint32), out["state"].view(np.uint32))
    assert np.array_equal(gag.option.cpu().numpy(), out["option"])
    # actions come from an argmax over Q: compare where the oracle's top-2 gap is not a rounding tie
    Q = oag.options.q(out["state"], out["option"])
    top2 = np.sort(Q, axis=1)[:, -2:]
    clear = (top2[:, 1] - top2[:, 0]) > 1e-3 * np.abs(Q).max()
    ga = gag.action.cpu().numpy()
    assert clear.mean() > 0.9
    assert np.array_equal(ga[clear], out["action"][clear])
    assert np.array_equal(gag.t_opt.cpu().numpy(), oag.t_opt)
    assert np.array_equal(gag.ep_steps.cpu().numpy(), oag.ep_steps)
    assert np.array_equal(gag.n_success.cpu().numpy(), oag.n_success)
    assert np.array_equal(gag.n_fail.cpu().numpy(), oag.n_fail)
    assert np.array_equal(gag.ex_count.cpu().numpy(), oag.ex_count)
    assert np.array_equal(gag.options.cnt.cpu().numpy(), oag.options.cnt)
    assert_close(gag.options.dW.cpu().numpy(), oag.options.dW)
    assert_close(gag.options.trace.cpu().numpy(), oag.options.trace)
    assert out["term"].sum() > 100 and out["hit"].sum() > 10
    for k in range(K):                                # same examples in the same ring slots (the oracle's append order)
        n = int(oag.ex_count[k])
        assert np.array_equal(gag.ex_xy[k, :n].cpu().numpy(), oag.ex_xy[k, :n])
        assert np.array_equal(gag.ex_label[k, :n].cpu().numpy(), oag.ex_label[k, :n])


def _set_gpu_options(gag, torch, theta, n_active, graph=False):
    """GPU twin of oracle_replay.activate."""
    gag.options.theta.copy_(torch.as_tensor(theta))
    gag.n_active = n_active
    gag.active_mask = (1 << n_active) - 1
    gag.parents_host[:] = 0
    gag.parents_host[0] = 1 << 31
    for n in range(1, min(n_active + 1, gag.options.K)):
        gag.parents_host[n] = (((1 << n) - 1) | (1 << 31)) if graph else (1 << (n - 1))
    gag._push_parents()


def _gpu_run_window(gag, torch, n):
    """n free-running GPU steps in ONE call (one multi-step launch when the window allows); returns what the step
    kernel recorded: pre-step states (n, B, 4), TD errors (n, B), and the (action, option) each env held before every
    step plus after the last one (n + 1, B)."""
    wl0 = int(gag._struct.win_len)
    assert wl0 + n <= gag.win_cap
    gag.run(n)
    torch.cuda.synchronize()
    rec = gag.win_rec[wl0:wl0 + n].cpu().numpy()                      # (n, B, 8)
    meta = rec[:, :, 5].copy().view(np.uint32)
    acts = np.concatenate([(meta & 7).astype(np.int32), gag.action.cpu().numpy()[None]], axis=0)
    opts = np.concatenate([((meta >> 8) & 0xFF).astype(np.int32), gag.option.cpu().numpy()[None]], axis=0)
    return rec[:, :, :4].copy(), rec[:, :, 4].copy(), acts, opts, ((meta >> 16) & 1).astype(bool)


def _check_choices(out, action, option, what):
    """The oracle's own choices against the followed (GPU) ones: options must agree, actions may differ only at a
    near-tie of the oracle's Q row (the two sides sum F products in different orders)."""
    assert np.array_equal(out["own_option"], option), f"{what}: option choice differs"
    dis = out["own_action"] != action
    if dis.any():
        Q = out["Qsel"][dis].astype(np.float64)
        gap = Q.max(axis=1) - Q[np.arange(len(Q)), action[dis]]
        assert gap.max() <= 1e-4 * max(1e-30, float(np.abs(out["Qsel"]).mean())), f"{what}: action differs without a Q tie"
    return int(dis.sum())


@pytest.mark.parametrize("order,K,n_active,name,B,launch", [
    (3, 4, 2, "easy", 3000, "window"),        # weights staged in shared memory (bulk copy), one launch per window
    (3, 4, 2, "easy", 3000, "step"),          # one launch per step: carried Q across launches
    (3, 6, 3, "hard", 2000, "window"),        # staged, gathered (k_stage < K)
    (5, 8, 2, "hard", 500, "window"),         # order 5: one 512-thread CTA per SM, weights staged
    (5, 8, 6, "hard", 500, "window"),         # order 5 with 7 options in use: weights through the global read-only path
    (5, 8, 6, "hard", 500, "step"),
])
def test_fused_pipeline_multi_window_tight(scg, torch, order, K, n_active, name, B, launch):
    """The whole fused pipeline across weight applies, at the stated bar: k_agent_step -> k_window -> k_reduce ->
    k_apply -> next window's Q from the refreshed packed weights.  13 steps, alpha > 0, a sync every 4 steps.  The GPU
    runs free; the oracle follows its choices.  Per step: pre-step states bit-identical, TD errors element-wise 1e-4.
    launch == "window": one multi-step launch per window and the sync inside scg_agent_run (the bench path): W
    element-wise after every apply.  launch == "step": one launch per step (Q carried across launches), syncs driven by
    hand so that dW, cnt and the traces are also compared before every apply."""
    from oracle_replay import activate, default_theta
    manual = launch == "step"
    kw = dict(sync_interval=1000 if manual else 4, option_timeout=5, epsilon=0.1, alpha=5e-3, max_episode_steps=9)
    oag, gag = _paired_agents(scg, torch, B, order, K, name, 13, window=4, **kw)
    theta = default_theta(K)
    activate(oag, theta, n_active)
    _set_gpu_options(gag, torch, theta, n_active)
    opt0 = np.random.default_rng(3).integers(0, n_active + 1, B).astype(np.int32)
    oag.option = opt0.copy()
    gag.option.copy_(torch.as_tensor(opt0))
    W0 = oag.options.W.copy()
    n_dis, n_term = 0, 0
    for w in range(4):
        n = 4 if w < 3 else 1
        if not manual:
            pre, dl, acts, opts, term = _gpu_run_window(gag, torch, n)
        else:
            parts = [_gpu_run_window(gag, torch, 1) for _ in range(n)]
            pre = np.concatenate([p[0] for p in parts]); dl = np.concatenate([p[1] for p in parts])
            acts = np.concatenate([p[2][:1] for p in parts] + [parts[-1][2][1:]])
            opts = np.concatenate([p[3][:1] for p in parts] + [parts[-1][3][1:]])
            term = np.concatenate([p[4] for p in parts])
        for t in range(n):
            what = f"window {w} step {t}"
            assert np.array_equal(oag.env.state.view(np.uint32), pre[t].view(np.uint32)), f"{what}: pre-step state"
            assert np.array_equal(oag.action, acts[t]) and np.array_equal(oag.option, opts[t])
            out = oag.step(follow=dict(action=acts[t + 1], option=opts[t + 1]))
            assert np.array_equal(out["term"], term[t]), f"{what}: termination flags"
            assert_close(dl[t], out["delta"], what=f"{what}: TD error")
            n_dis += _check_choices(out, acts[t + 1], opts[t + 1], what)
            n_term += int(out["term"].sum())
        assert np.array_equal(gag.state.cpu().numpy().view(np.uint32), oag.env.state.view(np.uint32))
        if w < 3:
            if manual:
                assert np.array_equal(gag.options.cnt.cpu().numpy(), oag.options.cnt)
                assert_close(gag.options.dW.cpu().numpy(), oag.options.dW, what=f"dW of window {w}")
                assert_close(gag.options.trace.cpu().numpy(), oag.options.trace, what=f"traces after window {w}")
                gag.sync()
                oag.options.apply()
            assert_close(gag.options.W.cpu().numpy(), oag.options.W, what=f"W after apply {w}")
            assert_close(gag.options.W.cpu().numpy() - W0, oag.options.W - W0, what=f"W - W0 after apply {w}")
            assert np.abs(oag.options.W - W0).max() > 1e-3       # the applies really moved the weights
    assert n_term > B // 2 and n_dis <= B // 50
    assert np.array_equal(gag.options.cnt.cpu().numpy(), oag.options.cnt)
    assert_close(gag.options.trace.cpu().numpy(), oag.options.trace, what="traces")
    assert_close(gag.options.dW.cpu().numpy(), oag.options.dW, what="dW of the open window")
    assert np.array_equal(gag.t_opt.cpu().numpy(), oag.t_opt) and np.array_equal(gag.ep_steps.cpu().numpy(), oag.ep_steps)
    assert np.array_equal(gag.n_success.cpu().numpy(), oag.n_success) and np.array_equal(gag.n_fail.cpu().numpy(), oag.n_fail)


def test_agent_run_and_manage_promotes_option(scg, torch):
    """The controller promotes the gestating option after enough successes and wires parents."""
    B = 4096
    gmap = scg.PinballMap.from_name("easy")
    cfg = scg.AgentConfig(map="easy", batch=B, order=3, max_options=3, gestation_successes=8, option_timeout=40,
                          sync_interval=4, epsilon=0.3)
    rng = np.random.default_rng(0)
    tx, ty, tr = gmap.target
    S = np.zeros((B, 4), dtype=np.float32)                 # start next to the goal so hits happen
    S[:, 0] = tx + rng.uniform(-0.12, 0.02, B)
    S[:, 1] = ty + rng.uniform(-0.1, 0.1, B)
    ag = scg.SkillChainAgent(cfg, gmap, initial_states=S)
    for _ in range(48):
        ag.step()
    c = ag.counters()
    assert c["n_success"][0] >= 8 and c["goals"] >= 8
    assert ag.manage(wait=True) is True
    assert ag.n_active == 1 and ag.active_mask == 1 and int(ag.parents_host[1]) == 1
    for _ in range(8):
        ag.step()
    torch.cuda.synchronize()
    assert int((ag.option == 1).sum()) > 0                 # the new gestating option is being executed


def test_run_episode_matches_oracle(scg, torch):
    """SkillChainAgent.run_episode against the oracle's: same stopping rule (every env has finished one more episode),
    same step count, finished / goal counts and mean return of the last finished episodes.  epsilon = 1 makes every
    action exploratory (identical Philox draws on both sides), so the two free-running agents follow identical
    trajectories; check_every=1 evaluates the stopping rule after every step, as the oracle does."""
    B, K = 512, 3
    kw = dict(sync_interval=4, option_timeout=6, epsilon=1.0, alpha=1e-3, max_episode_steps=14, gestation_successes=10 ** 9)
    oag, gag = _paired_agents(scg, torch, B, 2, K, "easy", 41, **kw)
    tx, ty, tr = oag.map.target
    rng = np.random.default_rng(2)
    S = oag.env.state.copy()
    S[: B // 4, 0] = tx + rng.uniform(-0.1, 0.0, B // 4)          # a quarter starts next to the goal: some episodes end there
    S[: B // 4, 1] = ty + rng.uniform(-0.05, 0.05, B // 4)
    oag.env.reset(states=S)
    oag.start_xy = oag.env.state[:, :2].copy()
    gag.s.copy_(torch.as_tensor(S.T.copy()))
    gag.start_xy.copy_(torch.as_tensor(S[:, :2].copy()))
    gag.invalidate()
    for rounds in range(2):                                        # two consecutive calls: the base is per call
        o = oag.run_episode(max_steps=40, manage_every=8)
        g = gag.run_episode(max_steps=40, manage_every=8, check_every=1)
        assert g["steps"] == o["steps"] and g["finished"] == o["finished"] == B and g["goals"] == o["goals"]
        assert g["env_steps"] == o["env_steps"] and g["n_active"] == o["n_active"]
        assert abs(g["mean_return"] - o["mean_return"]) <= 1e-6 * abs(o["mean_return"])
        assert np.array_equal(gag.state.cpu().numpy().view(np.uint32), oag.env.state.view(np.uint32))
        assert np.array_equal(gag.ep_count.cpu().numpy(), oag.episodes)
    assert o["goals"] > 0 and o["steps"] <= 14
    # the default (check every manage_every steps) stops at the next multiple of 8
    g2 = gag.run_episode(max_steps=40, manage_every=8)
    assert g2["steps"] % 8 == 0 and g2["finished"] == B


# ---- top-level SMDP learner over the options (SURVEY.md section 8 f-3) ------------------------------------------
@pytest.mark.parametrize("order,K,n_active,name,B,launch", [
    (3, 4, 2, "easy", 3000, "window"),
    (3, 4, 3, "hard", 3000, "step"),
    (2, 7, 5, "easy", 2000, "window"),        # 7 option slots -> two top-level slots
    (5, 8, 3, "hard", 500, "window"),
    (5, 8, 6, "hard", 500, "step"),           # weights through the global path
])
def test_top_level_learner_matches_oracle(scg, torch, order, K, n_active, name, B, launch):
    """Option choice by the learned SMDP value function Q_top (oracle/agent.py top_level=True): per step the TD errors
    of the options AND of the top-level learner (delta_top at every option termination), the chosen options (equal to
    the oracle's own eps_top-greedy choice except at Q_top near-ties), and after every apply all weight slots -
    the options' and the top-level learner's - element-wise within 1e-4."""
    from oracle_replay import activate, default_theta
    manual = launch == "step"
    kw = dict(sync_interval=1000 if manual else 4, option_timeout=4, epsilon=0.1, alpha=5e-3, max_episode_steps=9,
              top_level=True, alpha_top=1e-3, epsilon_top=0.15)
    oag, gag = _paired_agents(scg, torch, B, order, K, name, 29, window=4, **kw)
    assert gag.options.K_all == oag.options.K_all == K + (K + 4) // 5
    oag.opt_s0 = oag.env.state.copy()
    theta = default_theta(K)
    activate(oag, theta, n_active)
    _set_gpu_options(gag, torch, theta, n_active)
    opt0 = np.random.default_rng(3).integers(0, n_active + 1, B).astype(np.int32)
    oag.option = opt0.copy()
    gag.option.copy_(torch.as_tensor(opt0))
    W0 = oag.options.W.copy()
    n_term, n_dis_o, spread = 0, 0, 0
    for w in range(4):
        n = 4 if w < 3 else 1
        wl0 = int(gag._struct.win_len)
        if not manual:
            pre, dl, acts, opts, term = _gpu_run_window(gag, torch, n)
        else:
            parts = [_gpu_run_window(gag, torch, 1) for _ in range(n)]
            pre = np.concatenate([p[0] for p in parts]); dl = np.concatenate([p[1] for p in parts])
            acts = np.concatenate([p[2][:1] for p in parts] + [parts[-1][2][1:]])
            opts = np.concatenate([p[3][:1] for p in parts] + [parts[-1][3][1:]])
            term = np.concatenate([p[4] for p in parts])
        top = gag.win_top[wl0:wl0 + n].cpu().numpy()                    # (n, B, 8): s0, delta_top, option
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
                if dis.any():                                          # only at a near-tie of the oracle's Q_top row
                    Q = out["Qtop"][dis].astype(np.float64)
                    gap = Q.max(axis=1) - Q[np.arange(len(Q)), opts[t + 1][dis]]
                    fin = np.isfinite(out["Qtop"])
                    assert gap.max() <= 1e-4 * max(1e-30, float(np.abs(out["Qtop"][fin]).mean())), f"{what}: option choice"
                n_dis_o += int(dis.sum())
            _check_choices(dict(out, own_option=opts[t + 1]), acts[t + 1], opts[t + 1], what)
            n_term += int(tm.sum())
            spread = max(spread, len(np.unique(oag.option)))
        assert np.array_equal(gag.state.cpu().numpy().view(np.uint32), oag.env.state.view(np.uint32))
        if w < 3:
            if manual:
                assert np.array_equal(gag.options.cnt.cpu().numpy(), oag.options.cnt)
                assert_close(gag.options.dW.cpu().numpy()[K:], oag.options.dW[K:], what=f"top-level dW of window {w}")
                assert_close(gag.options.dW.cpu().numpy()[:K], oag.options.dW[:K], what=f"dW of window {w}")
                gag.sync()
                oag.options.apply()
            gW = gag.options.W.cpu().numpy()
            assert_close(gW[:K], oag.options.W[:K], what=f"option weights after apply {w}")
            assert_close(gW[K:] - W0[K:], oag.options.W[K:] - W0[K:], what=f"top-level weights after apply {w}")
            assert np.abs(oag.options.W[K:] - W0[K:]).max() > 1e-4
    assert n_term > B // 2 and n_dis_o <= B // 100
    assert spread >= min(3, n_active + 1)                             # the learner really spreads over several options
    assert np.array_equal(gag.options.cnt.cpu().numpy(), oag.options.cnt)
    for got, want in ((gag.start_vxy, oag.opt_s0[:, 2:]), (gag.opt_ret, oag.opt_R), (gag.opt_disc, oag.opt_disc)):
        assert np.array_equal(got.cpu().numpy().view(np.uint32), np.ascontiguousarray(want).view(np.uint32))


# ---- controller on the device: example rings and promote-and-fit -------------------------------------------
@pytest.mark.parametrize("B,cap,launch,hist,horizon", [(3000, 64, "window", 64, 1 << 30), (3000, 64, "step", 8, 1), (777, 4096, "window", 8, 2),
                                                       (40000, 1000, "window", 64, 1 << 30), (5000, 300, "window", 12, 1 << 30),
                                                       (70000, 1000, "window", 64, 1 << 30)])
def test_example_rings_match_oracle_past_capacity(scg, torch, B, cap, launch, hist, horizon):
    """The rings hold the oracle's examples in the oracle's slots - steps in order, envs in order within a step - also
    when a ring wraps several times inside one launch (cap 64, thousands of terminations per window), and when a pass
    spans more than one tile per CTA (B = 70000: the 8-step pass of windows 1 and 2 is 137 tiles of 4 KB)."""
    from oracle_replay import activate, default_theta
    K, n_active = 4, 2
    # hist: steps of event history on the device (8 = two windows: a ring pass at every flush; 64: only when somebody
    # looks); horizon: a hit only counts as a positive example within that many steps of the option's start
    kw = dict(sync_interval=1000, option_timeout=2, epsilon=0.3, alpha=0.0, max_episode_steps=7, example_capacity=cap,
              init_horizon=horizon)
    oag, gag = _paired_agents(scg, torch, B, 2, K, "easy", 31, window=4, event_history=hist, **kw)
    theta = default_theta(K)
    activate(oag, theta, n_active)
    _set_gpu_options(gag, torch, theta, n_active)
    for w in range(3):
        if launch == "window":
            pre, dl, acts, opts, term = _gpu_run_window(gag, torch, 4)
        else:
            parts = [_gpu_run_window(gag, torch, 1) for _ in range(4)]
            acts = np.concatenate([p[2][:1] for p in parts] + [parts[-1][2][1:]])
            opts = np.concatenate([p[3][:1] for p in parts] + [parts[-1][3][1:]])
        for t in range(4):
            oag.step(follow=dict(action=acts[t + 1], option=opts[t + 1]))
        if w != 1:                                          # (window 1 is left in the history: two windows in one ring pass)
            assert np.array_equal(gag.ex_count.cpu().numpy(), oag.ex_count), f"window {w}"
            assert np.array_equal(gag.ex_xy.cpu().numpy().view(np.uint32), oag.ex_xy.view(np.uint32)), f"window {w}"
            assert np.array_equal(gag.ex_label.cpu().numpy(), oag.ex_label), f"window {w}"
    assert oag.ex_count.max() > (3 * cap if cap < 1000 else 1000)
    # one more step, read mid-window: the property appends the open window's events first
    pre, dl, acts, opts, term = _gpu_run_window(gag, torch, 1)
    oag.step(follow=dict(action=acts[1], option=opts[1]))
    assert np.array_equal(gag.ex_count.cpu().numpy(), oag.ex_count)
    assert np.array_equal(gag.ex_xy.cpu().numpy().view(np.uint32), oag.ex_xy.view(np.uint32))
    gag.run(3)                                              # and the rest of that window is appended exactly once
    for t in range(3):
        oag.step()
    assert int(gag.ex_count.sum()) == int(gag.n_success.sum() + gag.n_fail.sum())


@pytest.mark.parametrize("graph,merge_overlap", [(False, 0.0), (True, 0.0), (True, 0.25)])
def test_manage_on_device_matches_oracle(scg, torch, graph, merge_overlap):
    """scg_agent_manage (decision + classifier fit + promotion in ONE kernel, no host round trip) against
    oracle.manage(): same decision at the same call, theta within 1e-4, same parents / masks; below the threshold and at
    the last slot nothing happens."""
    from oracle_replay import activate, default_theta
    B, K = 4096, 4
    kw = dict(sync_interval=4, option_timeout=6, epsilon=0.3, alpha=1e-3, gestation_successes=40, clf_steps=120, clf_lr=2.0,
              graph=graph, merge_overlap=merge_overlap)
    oag, gag = _paired_agents(scg, torch, B, 2, K, "easy", 19, **kw)
    tx, ty, tr = oag.map.target
    rng = np.random.default_rng(0)
    S = np.zeros((B, 4), dtype=np.float32)                 # start next to the goal so option 0 collects successes
    S[:, 0] = tx + rng.uniform(-0.15, 0.03, B)
    S[:, 1] = ty + rng.uniform(-0.12, 0.12, B)
    oag.env.reset(states=S)
    oag.start_xy = oag.env.state[:, :2].copy()
    gag.s.copy_(torch.as_tensor(S.T.copy()))
    gag.start_xy.copy_(torch.as_tensor(S[:, :2].copy()))
    gag.invalidate()
    promoted = []
    for w in range(10):
        pre, dl, acts, opts, term = _gpu_run_window(gag, torch, 4)
        for t in range(4):
            out = oag.step(follow=dict(action=acts[t + 1], option=opts[t + 1]))
            assert np.array_equal(out["state"].view(np.uint32), (pre[t + 1] if t < 3 else gag.state.cpu().numpy()).view(np.uint32))
        op = oag.manage()
        gp = gag.manage(wait=True)
        assert op == gp, f"window {w}: oracle promoted={op}, device promoted={gp} (n_success {oag.n_success})"
        if op:
            promoted.append(w)
            g = oag.n_active - 1
            assert_close(gag.options.theta[g].cpu().numpy(), oag.options.theta[g], what=f"theta of option {g}")
            # the controller's fit is the stand-alone fit: the same ring from theta = 0 gives the same bits
            X, y = gag.examples(g)
            refit = scg.OptionSet(1, 1, 1).fit_initiation(0, X, y, steps=kw["clf_steps"], lr=kw["clf_lr"])
            assert torch.equal(refit, gag.options.theta[g]), f"theta of option {g}: {refit} refit, {gag.options.theta[g]} device"
        c = gag.controller_state()
        assert c["n_active"] == oag.n_active and c["active_mask"] == int(sum(1 << k for k in range(K) if oag.active[k]))
        assert c["parents"] == [int(v) for v in oag.parents]
        assert c["n_promotions"] == len(promoted)
    assert len(promoted) >= 1, promoted
    assert np.array_equal(gag.option.cpu().numpy(), oag.option) and np.array_equal(gag.n_success.cpu().numpy(), oag.n_success)
    # the last slot is never promoted
    full = scg.SkillChainAgent(scg.AgentConfig(map="easy", batch=64, order=1, max_options=2, gestation_successes=0))
    full.n_active, full.active_mask = 1, 1
    assert full.manage(wait=True) is False and full.controller_state()["n_active"] == 1


def test_merge_detection_wires_the_meeting_chains(scg, torch):
    """Option graph with merge detection: the option being promoted (2) has its positive examples inside I_0 (x >= 0.6)
    but outside I_1 (y <= 0.45), so the next slot's targets must be {2, 0} and not 1; the goal joins iff it lies inside
    the freshly fit I_2.  Same rings injected on both sides; device controller against oracle.manage()."""
    from oracle_replay import activate, default_theta
    B, K = 256, 5
    kw = dict(sync_interval=4, graph=True, merge_overlap=0.5, gestation_successes=10, clf_steps=150, clf_lr=2.0)
    oag, gag = _paired_agents(scg, torch, B, 2, K, "easy", 53, **kw)
    theta = default_theta(K)
    activate(oag, theta, 2, graph=True)
    _set_gpu_options(gag, torch, theta, 2, graph=True)
    rng = np.random.default_rng(8)
    n = 3000
    X = rng.random((n, 2)).astype(np.float32)
    y = ((X[:, 0] > 0.7) & (X[:, 1] > 0.6)).astype(np.uint8)          # positives: upper right corner -> inside I_0 only
    oag.ex_xy[2, :n], oag.ex_label[2, :n], oag.ex_count[2], oag.n_success[2] = X, y, n, 1000
    gag._ex_xy[2, :n].copy_(torch.as_tensor(X)); gag._ex_label[2, :n].copy_(torch.as_tensor(y))
    gag._ex_count[2] = n
    gag.n_success[2] = 1000
    assert oag.manage() is True and gag.manage(wait=True) is True
    c = gag.controller_state()
    assert c["n_active"] == oag.n_active == 3 and c["parents"] == [int(v) for v in oag.parents]
    pm = c["parents"][3]
    assert pm & 0b100 and pm & 0b001 and not pm & 0b010
    assert_close(gag.options.theta[2].cpu().numpy(), oag.options.theta[2], what="theta of the promoted option")
    # merge_overlap = 0 wires every older option and the goal (the plain graph mode)
    oag2, gag2 = _paired_agents(scg, torch, B, 2, K, "easy", 53, **dict(kw, merge_overlap=0.0))
    activate(oag2, theta, 2, graph=True)
    _set_gpu_options(gag2, torch, theta, 2, graph=True)
    oag2.ex_xy[2, :n], oag2.ex_label[2, :n], oag2.ex_count[2], oag2.n_success[2] = X, y, n, 1000
    gag2._ex_xy[2, :n].copy_(torch.as_tensor(X)); gag2._ex_label[2, :n].copy_(torch.as_tensor(y))
    gag2._ex_count[2] = n
    gag2.n_success[2] = 1000
    assert oag2.manage() and gag2.manage(wait=True)
    assert gag2.controller_state()["parents"][3] == int(oag2.parents[3]) == (0b111 | (1 << 31))


def test_promotion_the_host_has_not_seen_yet_is_still_correct(scg, torch):
    """The host sizes the on-chip weight staging and the sweep's accumulator with its LOWER BOUND of n_active; options
    the device promoted since are handled by the kernels' global-memory paths.  A twin launched with a stale bound
    (n_active = 0 in the struct, a context without mirror) must reproduce the run that knows: states, actions, rings
    bit for bit; dW / W to rounding (different summation order)."""
    import ctypes as C
    from skill_chaining_with_graphs_b200._lib import check, current_stream
    from oracle_replay import default_theta
    lib = scg.load_library()
    for order, K, n_active in ((3, 4, 2), (5, 8, 3)):
        B = 1500 if order == 3 else 400
        kw = dict(sync_interval=4, option_timeout=4, epsilon=0.2, alpha=5e-3, max_episode_steps=9)
        (_, a), (_, b) = (_paired_agents(scg, torch, B, order, K, "hard", 23, **kw) for _ in range(2))
        theta = default_theta(K)
        for g in (a, b):
            _set_gpu_options(g, torch, theta, n_active)
        a.run(12)
        blind = scg.OptionSet(K, order, 1)                   # a second context: no mirror to learn from
        st = b._struct
        st.n_active = 0                                     # stale lower bound: only option 0 is staged / accumulated
        check(lib.scg_agent_run(b.map.handle, blind.ctx, C.byref(st), 12, 4, None, current_stream()))
        torch.cuda.synchronize()
        assert int(st.n_active) == 0
        assert torch.equal(a.s, b.s) and torch.equal(a.action, b.action) and torch.equal(a.option, b.option)
        assert torch.equal(a.n_success, b.n_success) and torch.equal(a.t_opt, b.t_opt)
        assert_close(b.options.W.cpu().numpy(), a.options.W.cpu().numpy(), rtol=1e-5, what=f"order {order}: W")
        assert_close(b.options._trace.cpu().numpy(), a.options._trace.cpu().numpy(), rtol=1e-5, what=f"order {order}: traces")


def test_poll_returns_consistent_snapshots_while_the_device_promotes(scg, torch):
    """scg_agent_poll from a second host thread while the main thread queues steps and promotions (chain mode, every
    manage() promotes until the last slot): every snapshot is one state the controller was in - mask, count, promotions
    and the new slot's parents agree - and manage_calls never goes back."""
    import ctypes as C
    import threading
    from skill_chaining_with_graphs_b200._lib import CtlStruct, check
    lib = scg.load_library()
    K = 12
    gag = scg.SkillChainAgent(scg.AgentConfig(map="easy", batch=4096, order=1, max_options=K, gestation_successes=0,
                                              clf_steps=4, sync_interval=4))
    bad, n_polls, stop = [], [0], threading.Event()

    def poll():
        m, last_calls = CtlStruct(), 0
        while not stop.is_set():
            check(lib.scg_agent_poll(gag.options.ctx, C.byref(m)))
            n, calls = int(m.n_active), int(m.manage_calls)
            ok = (n >= 1 and m.active_mask == (1 << n) - 1 and m.n_promotions == n - 1 and m.parents[n] == 1 << (n - 1)
                  and calls >= last_calls)
            if not ok and len(bad) < 5:
                bad.append(dict(n_active=n, active_mask=int(m.active_mask), n_promotions=int(m.n_promotions),
                                parents=[int(v) for v in m.parents[:K]], manage_calls=(last_calls, calls)))
            last_calls = calls
            n_polls[0] += 1

    def reset():            # option 0 active, slot 1 gestating, no promotions: through scg_agent_set_ctl
        gag.controller_state(sync=True)
        c = gag._ctl
        c.n_active, c.active_mask, c.n_promotions = 1, 1, 0
        for k in range(K):
            c.parents[k] = 0
        c.parents[0], c.parents[1] = 1 << 31, 1
        gag._push_ctl()

    reset()
    th = threading.Thread(target=poll)
    th.start()
    try:
        for _ in range(10):
            for _ in range(K - 1):
                gag.run(4)
                gag.manage()
            assert gag.controller_state()["n_active"] == K - 1
            reset()
    finally:
        stop.set()
        th.join()
    assert not bad, bad
    assert n_polls[0] > 100


def _two_rank_agents_one_device(scg, torch, Bh, streams, **kw):
    """Two half-batch agents on cuda:0 whose exchange contexts are connected through plain device pointers: the code
    path of one process per GPU (k_sync, k_manage's peer exchange) on a single GPU, one stream per rank."""
    import ctypes as C
    from skill_chaining_with_graphs_b200._lib import check
    lib = scg.load_library()
    global FULL_B
    saved, FULL_B = FULL_B, 2 * Bh
    try:
        halves, xs = [], []
        for r in range(2):
            with torch.cuda.stream(streams[r]):
                h = _full_agent(scg, torch, Bh, r * Bh, **kw)
            x = C.c_void_p()
            check(lib.scg_xchg_create(h.options.ctx, r, 2, C.byref(x)))
            halves.append(h); xs.append(x)
        torch.cuda.synchronize()
        _connect_ranks_one_process(lib, xs)
        for r in range(2):
            halves[r]._xchg = xs[r]
        with torch.cuda.stream(streams[0]):
            whole = _full_agent(scg, torch, 2 * Bh, 0, **kw)
        torch.cuda.synchronize()
        return whole, halves, xs
    finally:
        FULL_B = saved


def test_two_rank_agents_on_one_device_equal_single_agent_and_union_fit(scg, torch):
    """Row (e) and the multi-rank controller on the driver's single GPU: two ranks (streams) exchange weight deltas
    through k_sync every sync interval and reproduce the unsharded agent; then both promote the gestating option at the
    same manage() call with a classifier fit on the UNION of their example rings (gradient sums over peer memory):
    theta bit-identical on both ranks and within 1e-4 of the oracle's fit on the concatenated examples."""
    lib = scg.load_library()
    Bh = 4096
    streams = [torch.cuda.Stream(), torch.cuda.Stream()]
    # (rings large enough not to wrap: the unsharded agent's one ring then holds the same example set as the two
    # ranks' rings together, and more than the 8192 examples the fit kernel keeps in registers)
    kw = dict(window=0, order=3, K=4, name="hard", gestation_successes=50, clf_steps=80, clf_lr=2.0, example_capacity=32768)
    whole, halves, xs = _two_rank_agents_one_device(scg, torch, Bh, streams, **kw)
    try:
        for h in halves + [whole]:
            h.cfg.sync_interval = 8
        for it in range(3):                      # three sync intervals queued back to back on both streams
            for r in range(2):
                with torch.cuda.stream(streams[r]):
                    halves[r].run(8)
        with torch.cuda.stream(streams[0]):
            whole.run(24)
        torch.cuda.synchronize()
        st = torch.cat([halves[0].s, halves[1].s], dim=1)
        assert torch.equal(st, whole.s)
        assert torch.equal(halves[0].options.W, halves[1].options.W) and torch.equal(halves[0].options.Wt, halves[1].options.Wt)
        assert not halves[0].peer_sync_timed_out() and not halves[1].peer_sync_timed_out()
        assert_close(halves[0].options.W.cpu().numpy(), whole.options.W.cpu().numpy(), rtol=1e-5, what="W: 2 ranks vs 1")
        assert torch.equal(halves[0].n_success_global, halves[1].n_success_global)
        assert torch.equal(halves[0].n_success_global, halves[0].n_success + halves[1].n_success)
        # the controller: gestating option 2 (options 0, 1 are active in _full_agent) qualifies on the summed count
        g = 2
        assert int(halves[0].n_success_global[g]) >= 50 > 0
        ex = [h.examples(g) for h in halves]
        assert min(len(e[0]) for e in ex) > 0 and sum(len(e[0]) for e in ex) == len(whole.examples(g)[0]) < 32768
        for r in range(2):
            with torch.cuda.stream(streams[r]):
                halves[r].manage()
        with torch.cuda.stream(streams[0]):
            whole.manage()
        torch.cuda.synchronize()
        c0, c1, cw = (h.controller_state() for h in (halves[0], halves[1], whole))
        assert c0 == c1 and c0["n_active"] == 3 and c0["parents"][3] == 1 << 2
        assert cw["n_active"] == 3
        th0, th1 = halves[0].options.theta[g].cpu().numpy(), halves[1].options.theta[g].cpu().numpy()
        assert np.array_equal(th0.view(np.uint32), th1.view(np.uint32))          # bit-identical replicas
        X = np.concatenate([e[0].cpu().numpy() for e in ex])
        y = np.concatenate([e[1].cpu().numpy() for e in ex])
        ora = oracle.OptionSet(4, 1, 1)
        ora.fit_initiation(g, X, y, steps=80, lr=2.0)
        assert_close(th0, ora.theta[g], what="theta: union fit over two ranks vs the oracle on the concatenated examples")
        # (the unsharded agent has the same examples in one ring, in a different order: same fit to rounding)
        assert_close(whole.options.theta[g].cpu().numpy(), ora.theta[g], what="theta: single agent")
        # and the ranks keep running in step after the promotion (the new option is staged on both)
        for r in range(2):
            with torch.cuda.stream(streams[r]):
                halves[r].run(16)
        with torch.cuda.stream(streams[0]):
            whole.run(16)
        torch.cuda.synchronize()
        assert torch.equal(torch.cat([halves[0].s, halves[1].s], dim=1), whole.s)
        assert torch.equal(halves[0].options.W, halves[1].options.W)
    finally:
        for h in halves:
            h._xchg = None
        for x in xs:
            lib.scg_xchg_destroy(x)


# ---- windowed pipeline -------------------------------------------------------------------------------
# (order, K, window, map, active options).  Windows longer than 8 steps run the multi-block sweep.  At order 3, five
# option slots in use (four active options and the gestating slot) no longer fit the eight CTAs of the split sweep, so
# the last row runs its fallback.
_WINDOW_ROWS = [(3, 4, 8, "easy", 1), (2, 3, 5, "easy", 1), (5, 8, 8, "hard", 1), (1, 2, 3, "easy", 1),
                (4, 2, 4, "hard", 1), (3, 4, 20, "easy", 1), (1, 2, 12, "easy", 1), (2, 3, 9, "easy", 1),
                (4, 2, 16, "hard", 1), (5, 8, 12, "hard", 1), (3, 5, 12, "easy", 4)]
# initiation sets of the active options, in chain order: x >= 0.5, y >= 0.7, x <= 0.3, y <= 0.3 (the gestating slot
# takes the rest)
_WINDOW_THETA = [[-1.0, 2.0, 0.0, 0.0, 0.0, 0.0], [-1.4, 0.0, 2.0, 0.0, 0.0, 0.0], [0.6, -2.0, 0.0, 0.0, 0.0, 0.0],
                 [0.6, 0.0, -2.0, 0.0, 0.0, 0.0]]


@pytest.mark.parametrize("order,K,window,name,n_active", _WINDOW_ROWS,
                         ids=["-".join(map(str, r if r[4] > 1 else r[:4])) for r in _WINDOW_ROWS])
def test_windowed_sweep_equals_oracle_dense_traces(scg, torch, order, K, window, name, n_active):
    """One window of fused steps with frozen weights: the GPU's forward-view sweep must reproduce the
    oracle's DENSE per-step traces and dW (the parity target is the dense form's numbers)."""
    B = 700 if order >= 4 else 2500
    kw = dict(sync_interval=1000, option_timeout=5, epsilon=0.5, alpha=0.0, max_episode_steps=11)
    oag, gag = _paired_agents(scg, torch, B, order, K, name, 7, **kw)
    gag2 = None
    theta = np.zeros((K, 6), dtype=np.float32)
    theta[:n_active] = _WINDOW_THETA[:n_active]
    oag.options.theta[:] = theta
    oag.active[:n_active] = True
    oag.n_active = n_active
    gag.options.theta.copy_(torch.as_tensor(theta))
    gag.active_mask, gag.n_active = (1 << n_active) - 1, n_active
    for k in range(1, n_active + 1):            # chain mode: option k reaches for option k-1's initiation set
        oag.parents[k] = gag.parents_host[k] = 1 << (k - 1)
    gag._push_parents()
    gag.win_cap = window
    # rebuild the window buffer for the requested window length
    gag.win_rec = torch.zeros((window, B, 8), dtype=torch.float32, device="cuda")
    gag._struct.win_rec = gag.win_rec.data_ptr()
    gag._struct.win_cap = window
    n_steps = window
    for t in range(n_steps):
        out = oag.step()
        gag.step()
        # with eps = 0.5 most actions are exploratory (identical draws); follow the oracle's choices exactly
        # so that the recorded transitions are the same on both sides
        gag.action.copy_(torch.as_tensor(out["action"]))
        gag.option.copy_(torch.as_tensor(out["option"]))
        gag.invalidate()
        assert np.array_equal(gag.state.cpu().numpy().view(np.uint32), out["state"].view(np.uint32))
        assert_close(gag.delta.cpu().numpy(), out["delta"])
    assert out is not None and int(gag._struct.win_len) == (n_steps % window)
    assert np.array_equal(gag.options.cnt.cpu().numpy(), oag.options.cnt)
    assert (oag.options.cnt[:n_active + 1] > 0).all()                     # every option slot in use has steps
    assert_close(gag.options.trace.cpu().numpy(), oag.options.trace)      # property flushes the window
    assert_close(gag.options.dW.cpu().numpy(), oag.options.dW)
    assert int(gag._struct.win_len) == 0
    assert oag.n_fail.sum() + oag.n_success.sum() > B // 4                          # terminations inside the window


def test_carried_q_equals_recomputed_q(scg, torch):
    """Q_o(s, a) carried from the previous step == the value recomputed from scratch every step."""
    B = 4096
    ags = []
    for _ in range(2):
        _, gag = _paired_agents(scg, torch, B, 3, 4, "easy", 3, sync_interval=4, epsilon=0.1, option_timeout=6)
        ags.append(gag)
    a, b = ags
    for t in range(10):
        a.step()
        b.invalidate()
        b.step()
        assert torch.equal(a.s, b.s) and torch.equal(a.action, b.action) and torch.equal(a.option, b.option)
        assert float((a.delta - b.delta).abs().max()) <= 1e-5 * max(1.0, float(b.delta.abs().max()))
    assert float((a.options.W - b.options.W).abs().max()) <= 1e-6 * max(1.0, float(b.options.W.abs().max()))


def test_run_equals_step_loop_and_host_step(scg, torch):
    B = 2048
    (_, a), (_, b), (_, c) = (_paired_agents(scg, torch, B, 3, 3, "easy", 5, sync_interval=3, epsilon=0.05,
                                             deterministic=True) for _ in range(3))
    a.run(10)
    for _ in range(10):
        b.step()
    hs, ha = c.s.cpu().numpy().copy(), c.action.cpu().numpy().copy()
    for _ in range(10):
        hs, r, f, ha, d = c.step_host(hs, ha)
    torch.cuda.synchronize()
    assert a.t == b.t == c.t == 10
    # deterministic=True (fixed sweep order, fixed-order slab reduction without floating-point atomics): bit for bit
    assert torch.equal(a.s, b.s) and torch.equal(a.action, b.action)
    assert torch.equal(a.options.W, b.options.W) and torch.equal(a.options.trace, b.options.trace)
    assert np.array_equal(hs, a.s.cpu().numpy()) and np.array_equal(ha, a.action.cpu().numpy())
    assert float((c.options.W - a.options.W).abs().max()) <= 1e-6 * max(1.0, float(a.options.W.abs().max()))
    assert np.array_equal(d, c.delta.cpu().numpy())


# ---- golden fixtures (tests/golden, made by tools/make_golden.py from the oracle) ----------------------
import os  # noqa: E402

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


@pytest.mark.parametrize("name", ["easy", "hard"])
def test_golden_step(scg, torch, name):
    g = np.load(os.path.join(GOLD, f"step_{name}.npz"))
    gmap = scg.PinballMap.from_name(name)
    env = scg.PinballEnv(gmap, len(g["state"]))
    env.reset(states=g["state"])
    ns, r, done, hit = env.step(torch.as_tensor(g["action"]).cuda())
    assert np.array_equal(ns.cpu().numpy().view(np.uint32), g["next_state"].view(np.uint32))
    assert np.array_equal(env.flags.cpu().numpy(), g["flags"]) and np.array_equal(r.cpu().numpy(), g["reward"])


@pytest.mark.parametrize("order", [3, 5])
def test_golden_features_q(scg, torch, order):
    g = np.load(os.path.join(GOLD, f"features_q_o{order}.npz"))
    assert np.abs(scg.FourierBasis(order).features(g["state"]).cpu().numpy() - g["phi"]).max() < 2e-5
    s = scg.OptionSet(g["W"].shape[0], order, len(g["state"]))
    s.set_weights(g["W"])
    assert_close(s.q(g["state"], g["option"]).cpu().numpy(), g["Q"])


def test_golden_sarsa_and_classifier(scg, torch):
    g = np.load(os.path.join(GOLD, "sarsa_o3.npz"))
    gamma, lam, alpha = (float(v) for v in g["hp"])
    s = scg.OptionSet(g["W0"].shape[0], 3, g["S"].shape[1], gamma=gamma, lam=lam, alpha=alpha, seed=1)
    s.set_weights(g["W0"])
    for it in range(6):
        d = s.update(g["S"][it], g["A"][it], g["r"][it], g["S2"][it], g["A2"][it], g["done"][it], g["option"][it])
        s.tick()
        assert_close(d.cpu().numpy(), g["delta"][it])
        if it == 2:
            assert_close(s.dW.cpu().numpy(), g["dW3"])
            assert np.array_equal(s.cnt.cpu().numpy(), g["cnt3"])
            assert_close(s.trace.double().sum(dim=2).cpu().numpy(), g["trace3_sum"])
            s.apply()
            assert_close(s.W.cpu().numpy(), g["W3"])
    assert_close(s.dW.cpu().numpy(), g["dW_end"])
    assert_close(s.trace.double().sum(dim=2).cpu().numpy(), g["trace_end_sum"])
    c = np.load(os.path.join(GOLD, "classifier.npz"))
    k = scg.OptionSet(2, 1, 1)
    k.theta[0].copy_(torch.as_tensor(c["theta0"]))
    assert_close(k.clf_grad(0, c["X"], c["y"]).cpu().numpy(), c["grad0"])
    assert_close(k.fit_initiation(1, c["X"], c["y"], steps=100, lr=2.0).cpu().numpy(), c["theta1_fit"])
    S4 = np.concatenate([c["X"], np.zeros_like(c["X"])], axis=1)
    assert_close(k.initiation_prob(S4).cpu().numpy(), c["prob"])


def test_golden_agent_step(scg, torch):
    g = np.load(os.path.join(GOLD, "agent_step.npz"))
    B, K = len(g["state"]), g["theta"].shape[0]
    gmap = scg.PinballMap.from_name("easy")
    cfg = scg.AgentConfig(map="easy", batch=B, order=3, max_options=K, seed=2, sync_interval=3, option_timeout=3,
                          epsilon=0.2)
    ag = scg.SkillChainAgent(cfg, gmap, initial_states=g["state"])
    ag.options.set_weights(g["W"])
    ag.options.theta.copy_(torch.as_tensor(g["theta"]))
    ag.active_mask, ag.n_active = 3, 2
    ag.parents_host[1], ag.parents_host[2] = 1, 2
    ag._push_parents()
    ag.option.copy_(torch.as_tensor(g["option"]))
    ag.t_opt.copy_(torch.as_tensor(g["t_opt"]))
    ag.action.copy_(torch.as_tensor(g["action"]))
    ag.step()
    torch.cuda.synchronize()
    assert np.array_equal(ag.state.cpu().numpy().view(np.uint32), g["next_state"].view(np.uint32))
    assert_close(ag.delta.cpu().numpy(), g["delta"])
    assert np.array_equal(ag.option.cpu().numpy(), g["next_option"])
    assert np.array_equal(ag.t_opt.cpu().numpy(), g["t_opt_after"])
    assert np.array_equal(ag.n_success.cpu().numpy(), g["n_success"]) and np.array_equal(ag.n_fail.cpu().numpy(), g["n_fail"])
    assert np.array_equal(ag.options.cnt.cpu().numpy(), g["cnt"])
    assert_close(ag.options.dW.cpu().numpy(), g["dW"])
    assert_close(ag.options.trace.double().sum(dim=2).cpu().numpy(), g["trace_sum"])


# ---- cross-GPU exchange kernel --------------------------------------------------------------------------
def test_xchg_single_rank_equals_apply(scg, torch):
    """world = 1: the exchange kernel degenerates to the apply kernel (same arithmetic, dW and cnt zeroed)."""
    import ctypes as C
    from skill_chaining_with_graphs_b200._lib import check, ptr, current_stream
    rng = np.random.default_rng(3)
    K, order = 3, 3
    a, b = scg.OptionSet(K, order, 4, alpha=0.07), scg.OptionSet(K, order, 4, alpha=0.07)
    W = (rng.standard_normal(tuple(a.W.shape)) * 0.1).astype(np.float32)
    dW = rng.standard_normal(tuple(a.W.shape)).astype(np.float32)
    cnt = np.array([5, 0, 17], dtype=np.int32)
    for o in (a, b):
        o.set_weights(W)
        o._dW.copy_(torch.as_tensor(dW))
        o.cnt.copy_(torch.as_tensor(cnt))
        o.window_steps = 4
    a.apply()
    lib = scg.load_library()
    x = C.c_void_p()
    check(lib.scg_xchg_create(b.ctx, 0, 1, C.byref(x)))
    check(lib.scg_xchg_sync(x, K, ptr(b.W), ptr(b.Wt), ptr(b._dW), ptr(b.cnt), 0.07, 0.0, 4, None, None, current_stream()))
    torch.cuda.synchronize()
    assert torch.equal(a.W, b.W) and torch.equal(a.Wt, b.Wt)
    assert float(b._dW.abs().max()) == 0.0 and int(b.cnt.sum()) == 0
    t = C.c_int(7)
    check(lib.scg_xchg_status(x, C.byref(t)))
    assert t.value == 0
    lib.scg_xchg_destroy(x)


def test_xchg_two_devices_sum_and_identical_replicas(scg, torch):
    """Two ranks on two devices of one process (peer access, plain pointers): both apply the same summed delta."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    import ctypes as C
    from skill_chaining_with_graphs_b200._lib import check, ptr
    lib = scg.load_library()
    rng = np.random.default_rng(4)
    K, order = 4, 3
    W = (rng.standard_normal((K, 5, 256)) * 0.1).astype(np.float32)
    dWs = [rng.standard_normal((K, 5, 256)).astype(np.float32) for _ in range(2)]
    cnts = [np.array([3, 0, 9, 1], dtype=np.int32), np.array([4, 0, 2, 0], dtype=np.int32)]
    sets, xs = [], []
    for r in range(2):
        with torch.cuda.device(r):
            o = scg.OptionSet(K, order, 4, alpha=0.05)
            o.set_weights(W)
            o._dW.copy_(torch.as_tensor(dWs[r]))
            o.cnt.copy_(torch.as_tensor(cnts[r]))
            x = C.c_void_p()
            check(lib.scg_xchg_create(o.ctx, r, 2, C.byref(x)))
            sets.append(o); xs.append(x)
    for r in range(2):                       # peer access both ways
        with torch.cuda.device(r):
            torch.zeros(1, device=f"cuda:{1 - r}").to(f"cuda:{r}")      # makes torch enable peer access
    ptrs = (C.c_void_p * 2)()
    for r in range(2):
        p = C.c_void_p()
        check(lib.scg_xchg_local_ptr(xs[r], C.byref(p)))
        ptrs[r] = p
    for r in range(2):
        check(lib.scg_xchg_connect_ptrs(xs[r], ptrs))
    nloc = [torch.tensor([5, 0, 7, 1], dtype=torch.int32, device=f"cuda:{r}") * (r + 1) for r in range(2)]
    nglob = [torch.zeros(4, dtype=torch.int32, device=f"cuda:{r}") for r in range(2)]
    for it in range(3):                      # three syncs: exercises the double buffering and the sequence flags
        for r in range(2):
            with torch.cuda.device(r):
                o = sets[r]
                check(lib.scg_xchg_sync(xs[r], K, ptr(o.W), ptr(o.Wt), ptr(o._dW), ptr(o.cnt), 0.05, 0.0, 8,
                                        ptr(nloc[r]), ptr(nglob[r]), C.c_void_p(torch.cuda.current_stream().cuda_stream)))
        for r in range(2):
            torch.cuda.synchronize(r)
        ref = scg.OptionSet if False else None
        w0, w1 = sets[0].W.cpu(), sets[1].W.cpu()
        assert torch.equal(w0, w1)                                           # replicas bit-identical
        assert nglob[0].cpu().tolist() == nglob[1].cpu().tolist() == [15, 0, 21, 3]   # success counters summed over ranks
        if it == 0:
            ora = oracle.OptionSet(K, order, 4, alpha=0.05)
            ora.W[:] = W
            ora.window_steps = 8
            ora.apply((dWs[0].astype(np.float64) + dWs[1]), cnts[0] + cnts[1])
            assert_close(w0.numpy(), ora.W, rtol=1e-6)
        for r in range(2):                   # next round: new deltas
            with torch.cuda.device(r):
                assert float(sets[r]._dW.abs().max()) == 0.0 and int(sets[r].cnt.sum()) == 0
                sets[r]._dW.copy_(torch.as_tensor(dWs[r] * (it + 2)))
                sets[r].cnt.copy_(torch.as_tensor(cnts[r]))
    for r in range(2):
        t = C.c_int()
        check(lib.scg_xchg_status(xs[r], C.byref(t)))
        assert t.value == 0
        lib.scg_xchg_destroy(xs[r])


def _connect_ranks_one_process(lib, xs):
    import ctypes as C
    from skill_chaining_with_graphs_b200._lib import check
    ptrs = (C.c_void_p * len(xs))()
    for r, x in enumerate(xs):
        p = C.c_void_p()
        check(lib.scg_xchg_local_ptr(x, C.byref(p)))
        ptrs[r] = p
    for x in xs:
        check(lib.scg_xchg_connect_ptrs(x, ptrs))


@pytest.mark.parametrize("world,order,K", [(2, 3, 4), (4, 5, 8), (3, 2, 3)])
def test_xchg_ranks_on_one_device_sum_and_identical_replicas(scg, torch, world, order, K):
    """The multi-rank exchange kernel on ONE GPU: `world` exchange contexts on cuda:0, one stream per rank, plain
    device pointers as peer mappings.  Same code path as one process per GPU (publish, per-slice flags, rank-ordered
    sum, apply); runs on the driver's single-GPU box."""
    import ctypes as C
    from skill_chaining_with_graphs_b200._lib import check, ptr
    lib = scg.load_library()
    rng = np.random.default_rng(40 + world)
    F = (order + 1) ** 4
    W = (rng.standard_normal((K, 5, F)) * 0.1).astype(np.float32)
    dWs = [rng.standard_normal((K, 5, F)).astype(np.float32) for _ in range(world)]
    cnts = [rng.integers(0, 9, K).astype(np.int32) for _ in range(world)]
    cnts[0][K - 1] = 0
    for c in cnts[1:]:
        c[K - 1] = 0                                         # an option nobody executed: its weights must not move
    sets, xs, streams = [], [], [torch.cuda.Stream() for _ in range(world)]
    for r in range(world):
        o = scg.OptionSet(K, order, 4, alpha=0.05)
        o.set_weights(W)
        o._dW.copy_(torch.as_tensor(dWs[r]))
        o.cnt.copy_(torch.as_tensor(cnts[r]))
        x = C.c_void_p()
        check(lib.scg_xchg_create(o.ctx, r, world, C.byref(x)))
        sets.append(o); xs.append(x)
    _connect_ranks_one_process(lib, xs)
    nloc = [torch.arange(K, dtype=torch.int32, device="cuda") * (r + 1) for r in range(world)]
    nglob = [torch.zeros(K, dtype=torch.int32, device="cuda") for _ in range(world)]
    torch.cuda.synchronize()
    try:
        for it in range(3):                                  # three syncs: double buffering and sequence flags
            for r in range(world):
                o = sets[r]
                check(lib.scg_xchg_sync(xs[r], K, ptr(o.W), ptr(o.Wt), ptr(o._dW), ptr(o.cnt), 0.05, 0.0, 8,
                                        ptr(nloc[r]), ptr(nglob[r]), C.c_void_p(streams[r].cuda_stream)))
            torch.cuda.synchronize()
            for r in range(1, world):
                assert torch.equal(sets[r].W, sets[0].W) and torch.equal(sets[r].Wt, sets[0].Wt)   # bit-identical replicas
                assert torch.equal(nglob[r], nglob[0])
            assert nglob[0].cpu().tolist() == [k * world * (world + 1) // 2 for k in range(K)]
            if it == 0:
                ora = oracle.OptionSet(K, order, 4, alpha=0.05)
                ora.W[:] = W
                ora.window_steps = 8
                ora.apply(sum(d.astype(np.float64) for d in dWs), sum(cnts))
                assert_close(sets[0].W.cpu().numpy() - W, ora.W - W, what="summed update")
                assert np.array_equal(sets[0].W.cpu().numpy()[K - 1], W[K - 1])
            for r in range(world):
                assert float(sets[r]._dW.abs().max()) == 0.0 and int(sets[r].cnt.sum()) == 0
                sets[r]._dW.copy_(torch.as_tensor(dWs[r] * (it + 2)))
                sets[r].cnt.copy_(torch.as_tensor(cnts[r]))
            torch.cuda.synchronize()
        for x in xs:
            t = C.c_int(7)
            check(lib.scg_xchg_status(x, C.byref(t)))
            assert t.value == 0
    finally:
        for x in xs:
            lib.scg_xchg_destroy(x)


def test_xchg_missing_peer_is_fatal_not_silent(scg, torch):
    """A rank whose peer never arrives gives up after the timeout WITHOUT applying or zeroing anything, and every later
    exchange on that handle fails with SCG_EPEER (a silent partial apply would de-synchronise the replicas)."""
    import ctypes as C
    from skill_chaining_with_graphs_b200._lib import check, ptr, current_stream
    lib = scg.load_library()
    K, order = 2, 2
    sets, xs = [], []
    for r in range(2):
        o = scg.OptionSet(K, order, 4, alpha=0.05)
        o.set_weights(np.full((K, 5, 81), 0.25, dtype=np.float32))
        o._dW.fill_(1.0)
        o.cnt.fill_(3)
        x = C.c_void_p()
        check(lib.scg_xchg_create(o.ctx, r, 2, C.byref(x)))
        sets.append(o); xs.append(x)
    _connect_ranks_one_process(lib, xs)
    try:
        check(lib.scg_xchg_set_timeout(xs[0], 0.05))
        o = sets[0]
        check(lib.scg_xchg_sync(xs[0], K, ptr(o.W), ptr(o.Wt), ptr(o._dW), ptr(o.cnt), 0.05, 0.0, 8, None, None,
                                current_stream()))          # rank 1 never calls
        torch.cuda.synchronize()
        t = C.c_int(0)
        check(lib.scg_xchg_status(xs[0], C.byref(t)))
        assert t.value == 1
        assert float((o.W - 0.25).abs().max()) == 0.0 and float((o._dW - 1.0).abs().max()) == 0.0   # nothing applied
        rc = lib.scg_xchg_sync(xs[0], K, ptr(o.W), ptr(o.Wt), ptr(o._dW), ptr(o.cnt), 0.05, 0.0, 8, None, None,
                               current_stream())
        assert rc == -4 and b"peer" in lib.scg_error_string(rc)
    finally:
        for x in xs:
            lib.scg_xchg_destroy(x)


# ---- BASELINE.json full sizes: size-independent properties ----------------------------------------------
FULL_B = 65536          # configs[1]: 65,536 envs on one B200


def _full_agent(scg, torch, B, lo, seed=11, window=0, order=3, K=4, name="easy", **kw):
    gmap = scg.PinballMap.from_name(name)
    rng = np.random.default_rng(99)
    S = gmap.sample_free_states(rng, FULL_B)[lo:lo + B]
    cfg = scg.AgentConfig(map=name, batch=B, order=order, max_options=K, seed=seed, env_offset=lo, sync_interval=1000,
                          epsilon=0.1, option_timeout=6, alpha=1e-3, window=window, **kw)
    ag = scg.SkillChainAgent(cfg, gmap, initial_states=S)
    W = (np.random.default_rng(5).standard_normal(tuple(ag.options.W.shape)) * 0.1).astype(np.float32)
    ag.options.set_weights(W)
    theta = np.zeros((K, 6), dtype=np.float32)
    theta[0, :3] = [-6.0, 10.0, 0.0]
    theta[1, :3] = [4.5, 0.0, -10.0]
    ag.options.theta.copy_(torch.as_tensor(theta))
    ag.active_mask, ag.n_active = 3, 2
    ag.parents_host[1], ag.parents_host[2] = 1, 2
    ag._push_parents()
    return ag


def test_full_size_sharding_invariance(scg, torch):
    """65,536 envs as one batch == the same envs as 4 shards of 16,384 (global env ids key the RNG): states and
    actions bit-identical, summed dW / cnt equal to the unsharded ones (SURVEY.md section 8e)."""
    n = 8
    whole = _full_agent(scg, torch, FULL_B, 0)
    whole.run(n)
    dW, cnt = whole.options.dW.double().cpu(), whole.options.cnt.cpu()
    sdW, scnt, states, actions = torch.zeros_like(dW), torch.zeros_like(cnt), [], []
    for i in range(4):
        sh = _full_agent(scg, torch, FULL_B // 4, i * FULL_B // 4)
        sh.run(n)
        sdW += sh.options.dW.double().cpu()
        scnt += sh.options.cnt.cpu()
        states.append(sh.s.cpu()); actions.append(sh.action.cpu())
        del sh
    assert torch.equal(torch.cat(states, dim=1), whole.s.cpu())
    assert torch.equal(torch.cat(actions), whole.action.cpu())
    assert torch.equal(scnt, cnt) and int(cnt.sum()) == n * FULL_B
    assert float((sdW - dW).abs().max()) <= 1e-4 * max(1.0, float(dW.abs().max()))


def test_full_size_window_length_invariance(scg, torch):
    """The same 12 steps swept with windows of 1 (the dense per-step form), 4 and 8 steps give the same traces and
    dW: the forward-view sweep is exact for any window length (weights frozen)."""
    ref = None
    for window in (1, 4, 8):
        ag = _full_agent(scg, torch, FULL_B, 0, window=window)
        ag.run(12)
        tr, dW = ag.options.trace.clone(), ag.options.dW.clone()
        st = ag.s.clone()
        del ag
        if ref is None:
            ref = (tr, dW, st)
            continue
        assert torch.equal(st, ref[2])
        assert float((tr - ref[0]).abs().max()) <= 1e-4 * max(1.0, float(ref[0].abs().max()))
        assert float((dW - ref[1]).abs().max()) <= 1e-4 * max(1.0, float(ref[1].abs().max()))


def test_full_size_step_properties(scg, torch):
    """One step of 65,536 envs on the hard map: rewards are in the reward set, flags decode to valid (obstacle, edge)
    pairs of the map, positions stay in the unit square, speed never grows except by the thrust impulse."""
    gmap = scg.PinballMap.from_name("hard")
    rng = np.random.default_rng(1)
    S = gmap.sample_free_states(rng, FULL_B)
    A = rng.integers(0, 5, FULL_B).astype(np.int32)
    env = scg.PinballEnv(gmap, FULL_B)
    env.reset(states=S)
    ns, r, done, hit = env.step(torch.as_tensor(A).cuda())
    ns, r, done, hit = ns.cpu().numpy(), r.cpu().numpy(), done.cpu().numpy(), hit.cpu().numpy()
    assert set(np.unique(r).tolist()) <= {-1.0, -5.0, 10000.0}
    assert np.array_equal(r == 10000.0, done)
    assert ns[:, :2].min() >= 0.0 and ns[:, :2].max() <= 1.0
    edges, obst, local = gmap.edge_table()
    n_local = np.bincount(obst)
    k = hit[:, 0] != 0
    assert k.mean() > 0.02 and hit[~k, 1].max() == -1
    assert hit[k, 1].min() >= 0 and hit[k, 1].max() < len(n_local)
    assert np.all(hit[k, 2] < n_local[hit[k, 1]])
    sp0 = np.hypot(S[:, 2], S[:, 3]) + 0.2 + 1e-6
    assert np.all(np.hypot(ns[:, 2], ns[:, 3]) <= sp0)
    # a sample of it against the oracle, bit for bit
    idx = rng.choice(FULL_B, 4000, replace=False)
    ons, orr, ofl = step_batched(oracle.PinballMap.from_name("hard"), S[idx], A[idx])
    assert np.array_equal(ns[idx].view(np.uint32), ons.view(np.uint32)) and np.array_equal(r[idx], orr)


def _full_size_vs_oracle(scg, torch, name, B, order, K, n_active, T, shard, graph=False):
    """One T-step window of the free-running GPU agent at a BASELINE.json batch size, one multi-step launch, then the
    sweep and the apply - against the oracle replaying the same steps in follow mode, sharded over host processes."""
    import os
    from oracle_replay import default_theta, replay_sharded
    omap = oracle.PinballMap.from_name(name)
    gmap = scg.PinballMap.from_name(name)
    S = omap.sample_free_states(np.random.default_rng(77), B)
    hp = dict(map=name, order=order, max_options=K, seed=21, sync_interval=1000, epsilon=0.05, alpha=1e-3,
              option_timeout=6, max_episode_steps=2000, graph=graph)
    gag = scg.SkillChainAgent(scg.AgentConfig(batch=B, window=T, **hp), gmap, initial_states=S)
    W = (np.random.default_rng(5).standard_normal(tuple(gag.options.W.shape)) * 0.1).astype(np.float32)
    gag.options.set_weights(W)
    theta = default_theta(K)
    _set_gpu_options(gag, torch, theta, n_active, graph)
    opt0 = (np.arange(B) % (n_active + 1)).astype(np.int32)
    gag.option.copy_(torch.as_tensor(opt0))
    A0 = gag.action.cpu().numpy().copy()
    pre, dl, acts, opts, term = _gpu_run_window(gag, torch, T)
    assert int(gag._struct.win_len) == 0                           # the full window was swept
    g_dW = gag.options.dW.double().cpu().numpy()
    g_cnt = gag.options.cnt.cpu().numpy().astype(np.int64)
    g_rows = gag.options._trace.double().sum(dim=2).cpu().numpy()
    probe = np.random.default_rng(1).choice(B, 256, replace=False)   # a few envs' traces in full
    g_probe = gag.options._trace[torch.as_tensor(probe).cuda()].cpu().numpy()
    gag.cfg.sync_interval = T
    gag.sync()
    g_W = gag.options.W.cpu().numpy()
    jobs = []
    for lo in range(0, B, shard):
        hi = min(B, lo + shard)
        jobs.append(dict(cfg=dict(batch=hi - lo, env_offset=lo, **hp), S0=S[lo:hi], W=W, theta=theta, n_active=n_active,
                         graph=graph, actions=acts[:, lo:hi], options=opts[:, lo:hi], want_trace=False,
                         probe=sorted(int(i - lo) for i in probe if lo <= i < hi)))
    assert np.array_equal(acts[0], A0) and np.array_equal(opts[0], opt0)
    res = replay_sharded(jobs, procs=min(32, len(os.sched_getaffinity(0))))
    o_pre = np.concatenate([r["pre_state"] for r in res], axis=1)
    assert np.array_equal(o_pre.view(np.uint32), pre.view(np.uint32)), "pre-step states of the window"
    assert np.array_equal(np.concatenate([r["state"] for r in res]).view(np.uint32),
                          gag.state.cpu().numpy().view(np.uint32))
    o_dl = np.concatenate([r["delta"] for r in res], axis=1)
    for t in range(T):
        assert_close(dl[t], o_dl[t], what=f"TD errors of step {t}")
    assert sum(r["n_dis_option"] for r in res) == 0
    n_dis = sum(r["n_dis_action"] for r in res)
    assert n_dis <= B * T // 200 and max(r["worst_gap"] for r in res) <= 1e-4, (n_dis, max(r["worst_gap"] for r in res))
    o_cnt = sum(r["cnt"] for r in res)
    o_dW = sum(r["dW"] for r in res)
    assert np.array_equal(g_cnt, o_cnt) and int(o_cnt.sum()) == B * T
    assert_close(g_dW, o_dW, what="dW of the window")
    # every env's trace through its 5 row sums (a sum of F elements, each held to the element-wise bar: the sums get
    # the typical element magnitude x sqrt(F) as their scale), and a sample of envs' traces in full further down
    o_probe = np.concatenate([r["trace_probe"] for r in res])
    from oracle.compare import robust_scale
    assert_close(g_rows, np.concatenate([r["trace_rowsum"] for r in res]), what="per-env trace row sums",
                 scale=robust_scale(o_probe) * float(np.sqrt(o_probe.shape[2])))
    ora = oracle.OptionSet(K, order, 1, alpha=hp["alpha"])
    ora.W[:] = W
    ora.window_steps = T
    ora.apply(o_dW, o_cnt)
    assert_close(g_W - W, ora.W - W, what="weight update of the apply")
    assert_close(g_W, ora.W, what="W after the apply")
    for k in ("n_success", "n_fail", "ex_count"):
        assert np.array_equal(getattr(gag, k).cpu().numpy().astype(np.int64), sum(r[k] for r in res)), k
    assert term.sum() > B // 4
    # the probed envs' full traces (shards return them in ascending env order)
    assert_close(g_probe[np.argsort(probe)], o_probe, what="probed traces")


def test_full_size_configs1_window_vs_oracle(scg, torch):
    """BASELINE.json configs[1] at full size (easy, 65,536 envs, order 3, 4 option slots, 2 active classifiers): one
    8-step window in one launch + sweep + apply against the oracle (16 shards on the host cores)."""
    _full_size_vs_oracle(scg, torch, "easy", 65536, 3, 4, 2, 8, 4096)


def test_full_size_configs2_window_vs_oracle(scg, torch):
    """BASELINE.json configs[2] per-GPU shape (hard, 131,072 envs, order 5, 8 option slots, 3 active): one 4-step
    window against the oracle (64 shards on the host cores)."""
    _full_size_vs_oracle(scg, torch, "hard", 131072, 5, 8, 3, 4, 2048)


def test_full_size_configs4_graph_window_vs_oracle(scg, torch):
    """configs[4] (option-graph variant) at a quarter of the per-GPU size: parents = all earlier options + goal."""
    _full_size_vs_oracle(scg, torch, "hard", 32768, 5, 8, 3, 4, 2048, graph=True)


def test_graph_mode_parents_match_oracle(scg, torch):
    """Option-graph variant: an option whose parents are several initiation sets and the goal terminates on any of
    them (oracle/agent.py, graph=True); one fused step against the oracle."""
    B, K = 4000, 4
    oag, gag = _paired_agents(scg, torch, B, 3, K, "hard", 12, sync_interval=5, option_timeout=50, epsilon=0.2, graph=True)
    theta = np.zeros((K, 6), dtype=np.float32)
    theta[0] = [-1.2, 2.0, 0.0, 0.0, 0.0, 0.0]
    theta[1] = [-0.8, 0.0, 2.0, 0.0, 0.0, 0.0]
    oag.options.theta[:] = theta
    oag.active[:2] = True
    oag.n_active = 2
    oag.parents[1] = np.uint32(1) | np.uint32(1 << 31)
    oag.parents[2] = np.uint32(3) | np.uint32(1 << 31)
    gag.options.theta.copy_(torch.as_tensor(theta))
    gag.active_mask, gag.n_active = 3, 2
    gag.parents_host[1], gag.parents_host[2] = 1 | (1 << 31), 3 | (1 << 31)
    gag._push_parents()
    opt = np.full(B, 2, dtype=np.int32)
    oag.option = opt.copy()
    gag.option.copy_(torch.as_tensor(opt))
    out = oag.step()
    gag.step()
    torch.cuda.synchronize()
    assert out["hit"].sum() > 20
    assert np.array_equal(gag.state.cpu().numpy().view(np.uint32), out["state"].view(np.uint32))
    assert np.array_equal(gag.option.cpu().numpy(), out["option"])
    assert_close(gag.delta.cpu().numpy(), out["delta"])
    assert np.array_equal(gag.n_success.cpu().numpy(), oag.n_success) and np.array_equal(gag.n_fail.cpu().numpy(), oag.n_fail)


def test_map_validation(scg):
    for name in ("easy", "hard"):
        assert scg.PinballMap.from_name(name).validate() == []
    walls = [p.tolist() for p in oracle.PinballMap.from_name("easy").polygons[:4]]
    bad = scg.PinballMap(0.02, (0.5, 0.5, 0.04), [(0.5, 0.5), (0.2, 0.2)], walls + [[(0.4, 0.4), (0.6, 0.4), (0.6, 0.6), (0.4, 0.6)]])
    probs = bad.validate()
    assert any("target" in p for p in probs) and any("start 0" in p for p in probs) and not any("start 1" in p for p in probs)
    open_map = scg.PinballMap(0.02, (0.9, 0.2, 0.04), [(0.2, 0.9)], [[(0.4, 0.4), (0.6, 0.4), (0.5, 0.6)]])
    assert any("no wall" in p for p in open_map.validate())


def test_agent_on_second_device(scg, torch):
    """Kernel shared-memory opt-ins are per device: an agent on cuda:1 after one on cuda:0 in the same process."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    res = []
    for dev in (0, 1):
        with torch.cuda.device(dev):
            _, gag = _paired_agents(scg, torch, 2048, 3, 4, "hard", 21, sync_interval=4)
            gag.run(8)
            torch.cuda.synchronize(dev)
            res.append((gag.s.cpu(), gag.options.W.cpu()))
    assert torch.equal(res[0][0], res[1][0])
    assert float((res[0][1] - res[1][1]).abs().max()) <= 1e-6 * max(1.0, float(res[0][1].abs().max()))


@pytest.mark.parametrize("B,order,K,name", [(1, 3, 1, "easy"), (33, 1, 2, "hard"), (95, 2, 3, "easy"), (257, 4, 2, "hard"),
                                            (64, 5, 8, "easy"), (31, 3, 16, "hard")])
def test_agent_odd_shapes_match_oracle(scg, torch, B, order, K, name):
    """Ragged batches (not a multiple of the warp size), every order, K = 1 and K = 16: three fused steps in one
    launch and a sweep, against the oracle stepping the same transitions."""
    oag, gag = _paired_agents(scg, torch, B, order, K, name, 30 + B, sync_interval=50, option_timeout=2, epsilon=0.3)
    outs = []
    for t in range(3):
        out = oag.step()
        gag.step()
        gag.action.copy_(torch.as_tensor(out["action"]))
        gag.invalidate()
        assert np.array_equal(gag.state.cpu().numpy().view(np.uint32), out["state"].view(np.uint32))
        assert_close(gag.delta.cpu().numpy(), out["delta"])
        assert np.array_equal(gag.option.cpu().numpy(), out["option"])
    assert np.array_equal(gag.options.cnt.cpu().numpy(), oag.options.cnt)
    assert_close(gag.options.trace.cpu().numpy(), oag.options.trace)
    assert_close(gag.options.dW.cpu().numpy(), oag.options.dW)
    # and the multi-step launch path: run(5) == 5 x step() on a twin (epsilon-greedy draws are keyed by env and step)
    _, a = _paired_agents(scg, torch, B, order, K, name, 30 + B, sync_interval=4, option_timeout=2, epsilon=0.3)
    _, b = _paired_agents(scg, torch, B, order, K, name, 30 + B, sync_interval=4, option_timeout=2, epsilon=0.3)
    a.run(5)
    for _ in range(5):
        b.step()
    assert torch.equal(a.s, b.s) and torch.equal(a.action, b.action) and torch.equal(a.option, b.option)
    assert float((a.options.trace - b.options.trace).abs().max()) <= 1e-5 * max(1.0, float(b.options.trace.abs().max()))
    assert float((a.options.W - b.options.W).abs().max()) <= 1e-5 * max(1.0, float(b.options.W.abs().max()))


def test_empty_batch_and_bad_arguments(scg, torch):
    import ctypes as C
    ag = scg.SkillChainAgent(scg.AgentConfig(map="easy", batch=0, order=3, max_options=2))
    ag.run(3)                                                   # no envs: nothing to do, no error
    assert ag.t == 0 or ag.t == 3
    with pytest.raises(ValueError):
        scg.SkillChainAgent(scg.AgentConfig(map="easy", batch=4, window=99))
    with pytest.raises(ValueError):
        scg.OptionSet(17, 3, 4)
    with pytest.raises(ValueError):
        scg.OptionSet(2, 6, 4)
    lib = scg.load_library()
    assert lib.scg_agent_run(None, None, None, 1, 1, None, None) == -1
    o = scg.OptionSet(2, 3, 4)
    assert lib.scg_xchg_create(o.ctx, 3, 2, C.byref(C.c_void_p())) == -1


@pytest.mark.parametrize("B,K,order,top,window,hist", [(1, 1, 1, True, 1, 1), (33, 1, 2, False, 3, 4), (70, 2, 3, True, 8, 16),
                                                       (257, 13, 2, True, 5, 64), (64, 16, 1, False, 2, 64), (5, 3, 4, True, 7, 14)])
def test_controller_and_top_level_edge_shapes_match_oracle(scg, torch, B, K, order, top, window, hist):
    """Edge shapes of the round-2 machinery against the oracle: one env, one option slot (nothing can ever be promoted),
    the largest slot counts (13 options + 3 top-level slots = 16; 16 options without), windows of one step, an event
    history of the minimum size, more manage() calls than promotions.  Ten followed steps + controller calls; states and
    counters bit for bit, TD errors / weights / classifiers element-wise."""
    from oracle_replay import activate, default_theta
    kw = dict(sync_interval=window, option_timeout=3, epsilon=0.4, alpha=2e-3, max_episode_steps=6, gestation_successes=1,
              clf_steps=20, clf_lr=1.0, top_level=top, alpha_top=1e-3, epsilon_top=0.3, example_capacity=16)
    oag, gag = _paired_agents(scg, torch, B, order, K, "easy", 61, window=window, event_history=hist, **kw)
    if top:
        oag.opt_s0 = oag.env.state.copy()
    tx, ty, tr = oag.map.target
    S = oag.env.state.copy()
    S[::2, 0], S[::2, 1], S[::2, 2], S[::2, 3] = tx - 0.03, ty, 1.0, 0.0        # every other env flies into the goal
    oag.env.reset(states=S)
    oag.start_xy = oag.env.state[:, :2].copy()
    oag.opt_s0 = oag.env.state.copy()
    gag.s.copy_(torch.as_tensor(S.T.copy()))
    gag.start_xy.copy_(torch.as_tensor(S[:, :2].copy()))
    gag.start_vxy.copy_(torch.as_tensor(S[:, 2:].copy()))
    gag.invalidate()
    n_prom = 0
    for t in range(10):
        pre, dl, acts, opts, term = _gpu_run_window(gag, torch, 1)
        assert np.array_equal(oag.env.state.view(np.uint32), pre[0].view(np.uint32)), f"step {t}: pre-step state"
        out = oag.step(follow=dict(action=acts[1], option=opts[1]))
        assert np.array_equal(out["term"], term[0]), f"step {t}: termination flags"
        assert_close(dl[0], out["delta"], what=f"step {t}: TD error")
        if t % 3 == 2:
            op, gp = oag.manage(), gag.manage(wait=True)
            assert op == gp, f"step {t}: promotion decision"
            n_prom += int(op)
            c = gag.controller_state()
            assert c["n_active"] == oag.n_active and c["parents"] == [int(v) for v in oag.parents]
            assert_close(gag.options.theta.cpu().numpy(), oag.options.theta, what=f"step {t}: classifiers")
    assert np.array_equal(gag.state.cpu().numpy().view(np.uint32), oag.env.state.view(np.uint32))
    assert np.array_equal(gag.ex_count.cpu().numpy(), oag.ex_count)
    assert np.array_equal(gag.ex_xy.cpu().numpy().view(np.uint32), oag.ex_xy.view(np.uint32))
    assert np.array_equal(gag.n_success.cpu().numpy(), oag.n_success) and np.array_equal(gag.ep_count.cpu().numpy(), oag.episodes)
    assert_close(gag.options.W.cpu().numpy(), oag.options.W, what="weights (all slots)")
    assert_close(gag.options.trace.cpu().numpy(), oag.options.trace, what="traces")
    assert (n_prom == 0) if K == 1 else (n_prom >= 1 or B < 8)


def test_full_size_order5_hard_window_and_sharding(scg, torch):
    """configs[2] per-GPU shape (hard map, 131,072 envs, order 5, 8 option slots): 8 steps as one window == as two
    windows of 4, and the two half-batches reproduce the whole batch (states bit-identical, dW to rounding)."""
    global FULL_B
    saved, FULL_B = FULL_B, 131072
    try:
        whole = _full_agent(scg, torch, FULL_B, 0, order=5, K=8, name="hard", window=8)
        whole.run(8)
        st, act = whole.s.cpu(), whole.action.cpu()
        dW = whole.options.dW.double().cpu()
        tr_sum = whole.options.trace.double().sum(dim=(1, 2)).cpu()
        cnt = whole.options.cnt.cpu()
        del whole
        torch.cuda.empty_cache()
        w4 = _full_agent(scg, torch, FULL_B, 0, order=5, K=8, name="hard", window=4)
        w4.run(8)
        assert torch.equal(w4.s.cpu(), st) and torch.equal(w4.action.cpu(), act)
        d4 = w4.options.dW.double().cpu()
        assert float((d4 - dW).abs().max()) <= 1e-4 * max(1.0, float(dW.abs().max()))
        t4 = w4.options.trace.double().sum(dim=(1, 2)).cpu()
        assert float((t4 - tr_sum).abs().max()) <= 1e-4 * max(1.0, float(tr_sum.abs().max()))
        del w4
        torch.cuda.empty_cache()
        sdW, scnt, sts = torch.zeros_like(dW), torch.zeros_like(cnt), []
        for i in range(2):
            sh = _full_agent(scg, torch, FULL_B // 2, i * FULL_B // 2, order=5, K=8, name="hard", window=8)
            sh.run(8)
            sdW += sh.options.dW.double().cpu()
            scnt += sh.options.cnt.cpu()
            sts.append(sh.s.cpu())
            del sh
            torch.cuda.empty_cache()
        assert torch.equal(torch.cat(sts, dim=1), st) and torch.equal(scnt, cnt)
        assert float((sdW - dW).abs().max()) <= 1e-4 * max(1.0, float(dW.abs().max()))
    finally:
        FULL_B = saved


def test_checkpoint_resume(scg, torch, tmp_path):
    """save() in the middle of a sync interval, load() into a fresh agent, continue: same trajectory as the original."""
    _, a = _paired_agents(scg, torch, 3000, 3, 4, "hard", 17, sync_interval=8, option_timeout=5, epsilon=0.1)
    a.run(13)                                   # mid-interval: 5 steps of the second window are open
    path = str(tmp_path / "ckpt.npz")
    a.save(path)
    _, b = _paired_agents(scg, torch, 3000, 3, 4, "hard", 17, sync_interval=8, option_timeout=5, epsilon=0.1)
    b.run(3)                                    # same configuration, different history: load() must override all of it
    b.load(path)
    assert b.t == a.t == 13
    a.run(11)
    b.run(11)
    torch.cuda.synchronize()
    assert torch.equal(a.s, b.s) and torch.equal(a.action, b.action) and torch.equal(a.option, b.option)
    assert float((a.options.W - b.options.W).abs().max()) <= 1e-6 * max(1.0, float(a.options.W.abs().max()))
    assert float((a.options.trace - b.options.trace).abs().max()) <= 1e-5 * max(1.0, float(a.options.trace.abs().max()))
    assert a.counters()["episodes"] == b.counters()["episodes"]
    with pytest.raises(ValueError):
        _, c = _paired_agents(scg, torch, 100, 3, 4, "hard", 1)
        c.load(path)


def test_two_device_agents_equal_single_device_agent(scg, torch):
    """Row (e) end to end: the env batch split over two GPUs (one agent per device, weight deltas exchanged by the
    peer-memory kernel every sync interval) reproduces the single-GPU run: states bit-identical, replicas identical,
    weights equal to rounding."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    import ctypes as C
    from skill_chaining_with_graphs_b200._lib import check
    lib = scg.load_library()
    Bh = 4096
    kw = dict(window=0, order=3, K=4, name="hard")
    global FULL_B
    saved, FULL_B = FULL_B, 2 * Bh
    halves, xs = [], []
    try:
        with torch.cuda.device(0):
            whole = _full_agent(scg, torch, 2 * Bh, 0, **kw)
            whole.cfg.sync_interval = 8
        for r in range(2):
            with torch.cuda.device(r):
                h = _full_agent(scg, torch, Bh, r * Bh, **kw)
                h.cfg.sync_interval = 8
                x = C.c_void_p()
                check(lib.scg_xchg_create(h.options.ctx, r, 2, C.byref(x)))
                halves.append(h); xs.append(x)
        for r in range(2):
            with torch.cuda.device(r):
                torch.zeros(1, device=f"cuda:{1 - r}").to(f"cuda:{r}")      # peer access both ways
        ptrs = (C.c_void_p * 2)()
        for r in range(2):
            p = C.c_void_p()
            check(lib.scg_xchg_local_ptr(xs[r], C.byref(p)))
            ptrs[r] = p
        for r in range(2):
            check(lib.scg_xchg_connect_ptrs(xs[r], ptrs))
            halves[r]._xchg = xs[r]
        for _ in range(3):                       # three sync intervals, launched back to back without host syncs
            for r in range(2):
                with torch.cuda.device(r):
                    halves[r].run(8)
        with torch.cuda.device(0):
            whole.run(24)
        for r in range(2):
            torch.cuda.synchronize(r)
        st = torch.cat([halves[0].s.cpu(), halves[1].s.cpu()], dim=1)
        assert torch.equal(st, whole.s.cpu())
        assert torch.equal(halves[0].options.W.cpu(), halves[1].options.W.cpu())
        assert not halves[0].peer_sync_timed_out() and not halves[1].peer_sync_timed_out()
        w = whole.options.W.cpu()
        assert float((halves[0].options.W.cpu() - w).abs().max()) <= 1e-6 * max(1.0, float(w.abs().max()))
        assert float(w.abs().max()) > 0
        g = halves[0].n_success_global.cpu()
        assert torch.equal(g, halves[1].n_success_global.cpu())
    finally:
        FULL_B = saved
        for r in range(2):
            if r < len(halves):
                halves[r]._xchg = None
        for x in xs:
            lib.scg_xchg_destroy(x)


def test_run_host_equals_run(scg, torch):
    """run_host (host state in / out once per call) == the device-resident run."""
    (_, a), (_, b) = (_paired_agents(scg, torch, 3000, 3, 3, "easy", 8, sync_interval=4, epsilon=0.05) for _ in range(2))
    hs, ha = b.s.cpu().numpy().copy(), b.action.cpu().numpy().copy()
    for _ in range(3):
        a.run(4)
        hs, ha, r, f, d = b.run_host(hs, ha, 4)
    assert np.array_equal(hs, a.s.cpu().numpy()) and np.array_equal(ha, a.action.cpu().numpy())
    # (the host path re-evaluates Q_o(s, a) at the start of every call instead of carrying it: TD errors agree to rounding)
    assert np.array_equal(f, a.flags.cpu().numpy())
    assert_close(d, a.delta.cpu().numpy(), rtol=1e-5)
    assert float((a.options.W - b.options.W).abs().max()) <= 1e-5 * max(1.0, float(a.options.W.abs().max()))


def test_host_step_equals_device_steps_large_ragged_batch(scg, torch):
    """The host-buffer step against the device-resident step loop on a larger, ragged batch (not a tile multiple),
    across window sweeps and syncs.  (A two-stream variant that overlapped the halves' copies and kernels was
    measured at +2.6 % e2e and dropped.)"""
    B = 20000 + 13
    (_, a), (_, c) = (_paired_agents(scg, torch, B, 3, 3, "hard", 6, sync_interval=3, epsilon=0.05, option_timeout=4)
                      for _ in range(2))
    hs, ha = c.s.cpu().numpy().copy(), c.action.cpu().numpy().copy()
    for t in range(10):
        a.invalidate()                           # the host path re-evaluates Q_o(s, a) every call: make the twin do the same
        a.step()
        hs, r, f, ha, d = c.step_host(hs, ha)
        assert np.array_equal(hs, a.s.cpu().numpy()), f"state, step {t}"
        assert np.array_equal(ha, a.action.cpu().numpy()) and np.array_equal(f, a.flags.cpu().numpy())
        # (the slab reduction adds with atomics: after the first apply the weights, hence the TD errors, agree to rounding)
        assert np.array_equal(r, a.reward.cpu().numpy())
        assert_close(d, a.delta.cpu().numpy(), rtol=1e-5)
    torch.cuda.synchronize()
    assert torch.equal(a.option, c.option) and torch.equal(a.options.cnt, c.options.cnt)
    assert float((c.options.W - a.options.W).abs().max()) <= 1e-6 * max(1.0, float(a.options.W.abs().max()))
    assert float((c.options.trace - a.options.trace).abs().max()) <= 1e-5 * max(1.0, float(a.options.trace.abs().max()))
