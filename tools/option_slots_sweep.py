"""Cost of the window sweep's option slots beyond the shared accumulator, and of the top-level update's list rounds.

    python tools/option_slots_sweep.py [--k-used 8,9,12,16] [--reps 20] [--top-batch 1048576,131072] [--out FILE]

Sweep: the order-5 sweep at the configs[2] per-GPU shape (hard map, 131,072 envs, T = 8).  An agent with 16 option
slots records one window of 8 steps; the option ids of its records are then rewritten so that every env runs one option
for the whole window - either spread evenly over the k_used slots in use, or all on the highest slot (at k_used > 8 a
slot that accumulates in global memory: in chain mode the gestating slot, the highest id, takes the rest of the map) -
and the same window is swept `reps` times (scg_agent_flush with the window re-opened).  Time per sweep launch from the
library's CUDA-event profiling (kind 1).

Top-level update: order 3, 4 option slots, top_level=True, T = 8, at each --top-batch; the window is flushed `reps`
times and k_top's device time is read from torch.profiler.

Prints one JSON line per measurement (and appends them to --out).  Needs a GPU.
"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def _agent(scg, torch, B, order, K, name, n_active, **kw):
    from oracle_replay import default_theta
    cfg = scg.AgentConfig(map=name, batch=B, order=order, max_options=K, seed=11, window=16, sync_interval=1000,
                          option_timeout=5, epsilon=0.1, alpha=5e-3, **kw)
    ag = scg.SkillChainAgent(cfg, scg.PinballMap.from_name(name))
    dev = ag.options.W.device
    gen = torch.Generator(device=dev).manual_seed(0)
    ag.options.set_weights(torch.randn(ag.options.W.shape, generator=gen, device=dev) * 0.5)
    theta = default_theta(K)
    ag.options.theta.copy_(torch.as_tensor(theta))
    ag.n_active = n_active
    ag.active_mask = (1 << n_active) - 1
    ag.run(8)                                            # one open window of 8 recorded steps (window capacity 16)
    torch.cuda.synchronize()
    assert int(ag._struct.win_len) == 8
    return ag


def _reflush(ag):
    ag._struct.win_len = 8
    ag.flush()


def sweep(scg, torch, k_used, spread, reps):
    B = 131072
    ag = _agent(scg, torch, B, 5, 16, "hard", k_used - 1)
    rec = ag.win_rec[:8]                                 # (8, B, 8) float32; column 5 holds the meta bits
    meta = rec[:, :, 5].contiguous().view(torch.int32)
    if spread == "even":
        o = (torch.arange(B, device=rec.device, dtype=torch.int32) % k_used)[None, :].expand(8, B)
    else:
        o = torch.full((8, B), k_used - 1, device=rec.device, dtype=torch.int32)
    meta = (meta & ~0xFF00) | (o << 8)
    rec[:, :, 5] = meta.view(torch.float32)
    for _ in range(3):
        _reflush(ag)
    torch.cuda.synchronize()
    ag.profile_begin(4 * reps + 16, kinds=(1,))
    for _ in range(reps):
        _reflush(ag)
    torch.cuda.synchronize()
    ms, n = ag.profile_end()
    return dict(what="k_window", order=5, map="hard", B=B, T=8, k_used=k_used, records=spread,
                ms_per_launch=ms[1] / max(n[1], 1), launches=n[1])


def top(scg, torch, B, reps):
    ag = _agent(scg, torch, B, 3, 4, "easy", 2, top_level=True, alpha_top=1e-3, epsilon_top=0.15)
    events = int(((ag.ev_hist[:8, :B] & 0x80) != 0).sum())
    for _ in range(3):
        _reflush(ag)
    torch.cuda.synchronize()
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            _reflush(ag)
        torch.cuda.synchronize()
    us, n = 0.0, 0
    for ka in prof.key_averages():
        if "k_top" in ka.key:
            us += getattr(ka, "self_device_time_total", 0.0) or getattr(ka, "device_time_total", 0.0)
            n += ka.count
    return dict(what="k_top", order=3, K=4, B=B, T=8, event_bytes=8 * B, events=events, ms_per_launch=us / max(n, 1) / 1e3,
                launches=n)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--k-used", default="8,9,12,16")
    ap.add_argument("--top-batch", default="1048576,131072")
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    import skill_chaining_with_graphs_b200 as scg
    assert torch.cuda.is_available(), "needs a GPU"
    scg.load_library()
    rows = []
    for k in [int(v) for v in args.k_used.split(",") if v]:
        for spread in ("even", "highest"):
            rows.append(sweep(scg, torch, k, spread, args.reps))
            print(json.dumps(rows[-1]), flush=True)
    for B in [int(v) for v in args.top_batch.split(",") if v]:
        rows.append(top(scg, torch, B, args.reps))
        print(json.dumps(rows[-1]), flush=True)
    if args.out:
        with open(args.out, "a") as f:
            for r in rows:
                f.write(json.dumps(r) + "\n")


if __name__ == "__main__":
    main()
