"""The oracle's forward-view window form (OptionSet(windowed=True).flush) against its dense per-step sweep at every window
length the device sweep accepts (1 .. 32 steps, include/scg_b200.h SCG_WIN_MAX).  The GPU parity tests of long windows
(tests/test_gpu_long_windows.py) compare the device with both forms, so both are pinned here first, on the CPU.

One fixed batch of recorded steps serves every length T (a window of its first T steps, then one of the next T): envs
that terminate exactly at each step index, envs that never terminate (pure decay over the whole window), envs with two
or three terminations, steps masked out, option changes after every termination, and a non-zero trace at the window
start (the carry-in)."""
import numpy as np
import pytest

import oracle
from oracle.option import OptionSet

WIN_MAX = 32
B, K = 160, 3
HP = dict(gamma=0.95, lam=0.8, alpha=0.05, seed=1)


def _batch():
    """Steps 0..63 of the fixed batch (the second 32 repeat the first's terminations and masks): (S, A, r, S2, A2, done,
    mask, option) per step, the initial weights and traces."""
    omap = oracle.PinballMap.from_name("easy")
    rng = np.random.default_rng(0)
    done = np.zeros((WIN_MAX, B), dtype=bool)
    done[np.arange(WIN_MAX), np.arange(WIN_MAX)] = True               # envs 0..31: one termination, at step b
    # envs 32..63: none (pure decay); envs 64..95: two terminations; envs 96..127: three
    for i, b in enumerate(range(64, 96)):
        done[[i % WIN_MAX, (i * 7 + 8) % WIN_MAX], b] = True
    for i, b in enumerate(range(96, 128)):
        done[[(i * 3) % WIN_MAX, (i * 5 + 15) % WIN_MAX, (i * 11 + 23) % WIN_MAX], b] = True
    done[:, 128:] = rng.random((WIN_MAX, B - 128)) < 0.15              # envs 128..159: random
    mask = np.ones((WIN_MAX, B), dtype=bool)
    mask[2::3, 128:] = rng.random((len(range(2, WIN_MAX, 3)), B - 128)) < 0.7   # steps some envs sit out
    mask[5, 40:48] = False
    done, mask = np.concatenate([done, done]), np.concatenate([mask, mask])
    opt = np.zeros((2 * WIN_MAX, B), dtype=np.int32)
    o = rng.integers(0, K, B).astype(np.int32)
    steps = []
    for t in range(2 * WIN_MAX):
        opt[t] = o
        S, S2 = omap.sample_free_states(rng, B), omap.sample_free_states(rng, B)
        A, A2 = rng.integers(0, 5, B), rng.integers(0, 5, B)
        r = rng.standard_normal(B).astype(np.float32)
        steps.append((S, A, r, S2, A2, done[t], mask[t], o.copy()))
        ch = done[t] & mask[t]                                        # an env changes option only after a termination
        o = np.where(ch, (o + 1 + rng.integers(0, K - 1, B)) % K, o).astype(np.int32)
    W = (rng.standard_normal((K, 5, 81)) * 0.05).astype(np.float32)
    E0 = (rng.standard_normal((B, 5, 81)) * 0.3).astype(np.float32)
    return steps, done, mask, opt, W, E0


BATCH = _batch()


def test_fixed_batch_covers_the_window_edges():
    """The batch has what the sweep must get right at every length: a termination at each step index, envs with none,
    with two and with three, masked steps, and options that change after terminations."""
    steps, done, mask, opt, _, _ = BATCH
    done, mask, opt = done[:WIN_MAX], mask[:WIN_MAX], opt[:WIN_MAX]
    dn = done & mask
    assert dn.any(axis=1).all()                                       # a termination at every step index
    n_term = dn.sum(axis=0)
    assert (n_term == 0).sum() >= 32 and (n_term == 2).any() and (n_term >= 3).any()
    assert (~mask).any() and (opt[1:] != opt[:-1]).any(axis=1).sum() >= 16


@pytest.mark.parametrize("T", range(1, WIN_MAX + 1))
def test_windowed_form_equals_dense_form_at_every_window_length(T):
    """One window of T steps (frozen weights), flushed once: the forward view's fp64 G_t and c_t give the dense sweep's
    traces to 1e-6 and its dW to 1e-6 of max |dW|, and the same counts.  Then a second window of T steps on top of the
    first (the next T steps of the batch), so the trace carried across a flush is also checked."""
    steps, _, _, _, W, E0 = BATCH
    d, w = OptionSet(K, 2, B, **HP), OptionSet(K, 2, B, windowed=True, **HP)
    for o in (d, w):
        o.W[:] = W
        o.trace[:] = E0
    for rep in range(2):
        for t in range(T):
            S, A, r, S2, A2, dn, m, o = steps[rep * T + t]
            dd = d.update(S, A, r, S2, A2, dn, o, m)
            dw = w.update(S, A, r, S2, A2, dn, o, m)
            assert np.array_equal(dd, dw)
            d.tick(); w.tick()
        w.flush()
        what = f"T = {T}, window {rep}"
        assert np.abs(w.trace - d.trace).max() < 1e-6, what
        assert np.abs(w.dW - d.dW).max() < 1e-6 * max(1.0, np.abs(d.dW).max()), what
        assert np.array_equal(w.cnt, d.cnt), what
    assert np.abs(d.dW).max() > 0 and np.abs(d.trace).max() > 0


@pytest.mark.parametrize("sync_interval", [13, 16, 32])
def test_windowed_agent_equals_dense_agent_long_windows(sync_interval):
    """The whole oracle agent with windows of 13, 16 and 32 steps (a window is a sync interval) == the dense agent:
    same trajectories, weights after every apply to 1e-6, traces to 1e-5."""
    kw = dict(map="hard", batch=64, order=2, max_options=3, seed=5, sync_interval=sync_interval, option_timeout=6,
              epsilon=0.2, alpha=0.01, max_episode_steps=40)
    d = oracle.SkillChainAgent(oracle.AgentConfig(**kw))
    w = oracle.SkillChainAgent(oracle.AgentConfig(windowed=True, **kw))
    rng = np.random.default_rng(0)
    W = (rng.standard_normal(d.options.W.shape) * 0.2).astype(np.float32)
    d.options.W[:] = W; w.options.W[:] = W
    for t in range(2 * sync_interval + 3):
        od, ow = d.step(), w.step()
        assert np.array_equal(od["state"], ow["state"]) and np.array_equal(od["action"], ow["action"])
        assert np.allclose(od["delta"], ow["delta"], atol=1e-5 * max(1.0, np.abs(od["delta"]).max()))
        if (t + 1) % sync_interval == 0:
            assert np.abs(d.options.W - w.options.W).max() < 1e-6
    assert np.abs(d.options.W - W).max() > 1e-4
    w.options.flush()
    assert np.abs(d.options.trace - w.options.trace).max() < 1e-5
