#!/usr/bin/env python
"""Run full skill chaining on a map until the option chain reaches the start state (or a wall-clock budget ends), then
measure what the discovered chain is worth: BASELINE.json's "a full skill chain discovered on the hard map in under one
wall-clock minute".

    python tools/discover_chain.py --map hard --batch 65536 --options 8 [--graph] [--no-top-level]

What makes the discovery meaningful (round 1's was not: with one start position and examples labelled only by "hit", the
first classifier already covered the start):
  * many start states: episodes begin at the map's start and at --starts random free-space positions, so option executions
    begin all over the map and the classifiers see positives and negatives everywhere;
  * an example is positive only if the option reached its target within --horizon steps of where it started
    (AgentConfig.init_horizon), so an initiation set is a neighbourhood of its target and the chain has to grow link by
    link from the goal back to the start;
  * options are chosen by the learned top-level SMDP value function (AgentConfig.top_level), not by slot order.
The controller runs on the device (one kernel per manage() call); the host only polls the mirror to time-stamp promotions.
After discovery a fresh batch of envs, all at the map's own start, runs the chain greedily (epsilon = 0) for one episode
each: the success rate and the steps to the goal are reported, next to the same numbers for the untrained agent.
With --option-log CAP every option execution of the run is logged on the device (AgentConfig.option_log) and polled after
each chunk; the final JSON then carries per-option totals for the whole run ("options": executions, hit and label rates,
mean duration, the count of each outcome flag, the share of env-steps spent in the option) - how each link of the chain
was used, and why its executions stopped.  A poll waits for the device and copies the new records to the host, so the
run's clocks (--budget, --train-seconds, wall_s and the promotion times) leave the polls out: a logged run takes the same
steps in the same clock time as an unlogged one, up to the overlap of host and device work that each poll's wait gives
up and the example-ring pass that each poll runs in place of the next manage().  The time the polls took is reported
as option_poll_s.
With --draw PATH the greedy evaluation after discovery also logs the trajectories of its first --draw-envs envs
(AgentConfig.trajectory_envs) and the script writes PATH, an SVG of the map, each active option's initiation set (64 x 64
positions at zero velocity) and those greedy paths coloured by the running option (tools/chain_svg.py); the final JSON
names it as "drawing".
With --occupancy G the training agent counts every env-step by option and cell of a G x G grid (AgentConfig.occupancy_grid);
the final JSON then carries, per option, its share of all env-steps and the fraction of the free-space cells (cells that
hold a position sampled uniformly from free space) that it visited, and --draw shades each option's visited cells under
its initiation set's outline.
"""
import argparse
import json
import os
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from learning_curve import OptionTally  # noqa: E402


def evaluate(scg, torch, base_map, src, args, n_env=4096, trained=True, draw=None, occupancy=None):
    """Greedy episodes from the map's own start with (a copy of) the agent's weights, classifiers and option graph.
    draw: SVG path - the first args.draw_envs envs' trajectories and the initiation sets are drawn there, over the
    training run's occupancy counts when given."""
    traj = dict(trajectory_envs=tuple(range(min(args.draw_envs, n_env))),
                trajectory_log=min(args.draw_envs, n_env) * (args.max_episode_steps + 64)) if draw else {}
    cfg = scg.AgentConfig(map=args.map, batch=n_env, order=args.order, max_options=args.options, gamma=0.99, lam=0.9,
                          alpha=0.0, epsilon=0.0, sync_interval=8, option_timeout=args.option_timeout,
                          max_episode_steps=args.max_episode_steps, gestation_successes=1 << 30, graph=args.graph,
                          top_level=not args.no_top_level, alpha_top=0.0, epsilon_top=0.0, seed=123, **traj)
    ev = scg.SkillChainAgent(cfg, base_map)
    if trained:
        ev.options.set_weights(src.options.W)
        ev.options.theta.copy_(src.options.theta)
        c = src.controller_state(sync=True)
        ev.parents_host[:] = np.array(c["parents"], dtype=np.uint32)
        ev._ctl.n_active, ev._ctl.active_mask = c["n_active"], c["active_mask"]
        ev._push_ctl()
    st = ev.run_episode(max_steps=args.max_episode_steps, manage_every=64)
    goals = int(ev.stats[1])
    if draw:
        from chain_svg import initiation_grid, render
        c = ev.controller_state(sync=True)
        grid = initiation_grid(ev.options, c["active_mask"])
        with open(draw, "w") as f:
            f.write(render(base_map, ev.trajectories(), init_grid=grid, occupancy=occupancy,
                           title=f"{args.map} map: {c['n_active']} active options, greedy paths of {args.draw_envs} envs"
                                 + (", shaded where each option ran in training" if occupancy is not None else "")))
    return dict(success_rate=goals / n_env, finished=st["finished"], mean_return=st["mean_return"], steps=st["steps"])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--map", default="hard")
    ap.add_argument("--batch", type=int, default=65536)
    ap.add_argument("--order", type=int, default=3)
    ap.add_argument("--options", type=int, default=8)
    ap.add_argument("--graph", action="store_true")
    ap.add_argument("--no-top-level", action="store_true")
    ap.add_argument("--budget", type=float, default=55.0)
    ap.add_argument("--alpha", type=float, default=2e-3)
    ap.add_argument("--alpha-top", type=float, default=1e-3)
    ap.add_argument("--epsilon", type=float, default=0.1)
    ap.add_argument("--gestation", type=int, default=20000)
    ap.add_argument("--train-seconds", type=float, default=25.0, help="keep learning this long after the chain is complete")
    ap.add_argument("--horizon", type=int, default=120)
    ap.add_argument("--option-timeout", type=int, default=120)
    ap.add_argument("--max-episode-steps", type=int, default=1500)
    ap.add_argument("--starts", type=int, default=255)
    ap.add_argument("--chunk", type=int, default=64)
    ap.add_argument("--min-chain", type=int, default=3)
    ap.add_argument("--option-log", type=int, default=0, metavar="CAP",
                    help="log every option execution (ring of CAP records, polled every chunk) and report per-option totals")
    ap.add_argument("--draw", default=None, metavar="PATH", help="write an SVG of the chain and the greedy paths here")
    ap.add_argument("--draw-envs", type=int, default=32, help="greedy envs whose paths are drawn")
    ap.add_argument("--occupancy", type=int, default=0, metavar="G",
                    help="count every training env-step by option and cell of a G x G grid and report where each option ran")
    args = ap.parse_args()
    import torch
    import skill_chaining_with_graphs_b200 as scg
    base = scg.PinballMap.from_name(args.map)
    rng = np.random.default_rng(0)
    extra = base.sample_free_states(rng, args.starts)[:, :2] if args.starts > 0 else np.zeros((0, 2), np.float32)
    starts = [tuple(float(v) for v in p) for p in base.starts] + [(float(x), float(y)) for x, y in extra]
    train_map = scg.PinballMap(float(base.ball_r), tuple(float(v) for v in base.target), starts,
                               [p.tolist() for p in base.polygons])
    cfg = scg.AgentConfig(map=args.map, batch=args.batch, order=args.order, max_options=args.options, gamma=0.99, lam=0.9,
                          alpha=args.alpha, epsilon=args.epsilon, sync_interval=8, option_timeout=args.option_timeout,
                          max_episode_steps=args.max_episode_steps, gestation_successes=args.gestation,
                          example_capacity=8192, clf_steps=300, clf_lr=2.0, graph=args.graph, option_bonus=1000.0,
                          top_level=not args.no_top_level, alpha_top=args.alpha_top, epsilon_top=0.1,
                          init_horizon=args.horizon, option_log=args.option_log, occupancy_grid=args.occupancy)
    ag = scg.SkillChainAgent(cfg, train_map)
    tally = OptionTally([0, 1 << 32], args.options) if args.option_log else None
    opt = dict(seen=0, lost=0, s=0.0)

    def poll_options():
        if tally is not None:
            torch.cuda.synchronize()             # the steps queued so far run on the clock, the poll does not
            p0 = time.perf_counter()
            ex = ag.option_executions(since=opt["seen"])
            opt["lost"] += ex["total"] - opt["seen"] - len(ex["step"])
            opt["seen"] = ex["total"]
            tally.add(ex)
            opt["s"] += time.perf_counter() - p0

    def clock():                                 # wall clock less the time spent in polls of the option log
        return time.perf_counter() - opt["s"]
    before = evaluate(scg, torch, base, ag, args, trained=False)
    start = torch.tensor([[float(base.starts[0][0]), float(base.starts[0][1]), 0.0, 0.0]], device="cuda")
    torch.cuda.synchronize()
    t0 = clock()
    log, steps, seen, done = [], 0, 0, False

    def start_covered(n_active):
        return bool(ag.options.initiation(start)[0, :n_active].any()) if n_active else False

    # skill chaining stops creating options once an initiation set covers the start state (or the slots run out)
    while clock() - t0 < args.budget and not done:
        ag.run(args.chunk)
        ag.manage()                                   # one kernel on the stream; nothing waits for it
        steps += args.chunk
        poll_options()
        c = ag.controller_state(sync=False)           # the host mirror: promotions show up here a moment later
        if c["n_promotions"] > seen:
            seen = c["n_promotions"]
            covered = start_covered(c["n_active"])
            log.append(dict(t=round(clock() - t0, 3), steps=steps, n_active=c["n_active"],
                            promoted_at_step=c["last_promotion_step"], start_covered=covered))
            print(json.dumps(log[-1]), flush=True)
            done = (covered and c["n_active"] >= args.min_chain) or c["n_active"] >= args.options - 1
    torch.cuda.synchronize()
    wall = clock() - t0
    # the chain is in place: keep learning the option policies and the top-level values for a while
    t1 = clock()
    train_steps = 0
    while clock() - t1 < args.train_seconds:
        if tally is None:
            ag.run(16 * args.chunk)
        else:                                         # the same steps, with a poll of the option log after each chunk
            for _ in range(16):
                ag.run(args.chunk)
                poll_options()
        ag.manage()
        train_steps += 16 * args.chunk
        torch.cuda.synchronize()
    train_wall = clock() - t1
    c = ag.controller_state(sync=True)
    cnt = ag.counters()
    # how much of the free space each initiation set covers, and whether it contains the map's start
    probe = torch.as_tensor(base.sample_free_states(np.random.default_rng(1), 20000)).cuda()
    inside = ag.options.initiation(probe)[:, :c["n_active"]].float().mean(dim=0).cpu().numpy().tolist() if c["n_active"] else []
    occ = ag.occupancy() if args.occupancy else None
    after = evaluate(scg, torch, base, ag, args, trained=True, draw=args.draw,
                     occupancy=occ["counts"] if occ is not None else None)
    options = {}
    if occ is not None:
        G = occ["grid"]
        free_xy = base.sample_free_states(np.random.default_rng(2), 200000)[:, :2]
        free = np.zeros((G, G), dtype=bool)
        free[np.clip((free_xy[:, 1] * np.float32(G)).astype(np.int64), 0, G - 1),
             np.clip((free_xy[:, 0] * np.float32(G)).astype(np.int64), 0, G - 1)] = True
        counts = occ["counts"]
        options["occupancy"] = dict(
            grid=G, env_steps=occ["env_steps"], free_cells=int(free.sum()),
            share_of_env_steps=[round(int(counts[o].sum()) / max(occ["env_steps"], 1), 4) for o in range(len(counts))],
            free_cells_visited=[round(float(((counts[o] > 0) & free).sum()) / free.sum(), 3) for o in range(len(counts))])
    if tally is not None:
        poll_options()
        options.update(options=tally.rows(0, (steps + train_steps) * args.batch), option_executions=opt["seen"],
                       option_executions_lost=opt["lost"], option_poll_s=round(opt["s"], 3))
    print(json.dumps(dict(map=args.map, batch=args.batch, graph=args.graph, top_level=not args.no_top_level,
                          wall_s=round(wall, 3), train_after_s=round(train_wall, 2), train_after_steps=train_steps, steps=steps, env_steps=steps * args.batch, n_active=c["n_active"],
                          chain_complete=done, start_covered=start_covered(c["n_active"]), parents=c["parents"],
                          initiation_set_fraction_of_free_space=[round(v, 3) for v in inside],
                          goals=cnt["goals"], episodes=cnt["episodes"], mean_return=cnt["mean_return"],
                          n_success=cnt["n_success"].tolist(), promotions=log,
                          greedy_from_start_untrained=before, greedy_from_start_after_discovery=after, **options,
                          **(dict(drawing=args.draw) if args.draw else {}))))


if __name__ == "__main__":
    main()
