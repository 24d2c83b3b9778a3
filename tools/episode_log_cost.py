#!/usr/bin/env python
"""What a device log costs: the configs[1] shape (easy map, 65,536 envs, order 3, 4 options, sync every 8 steps) with
the log off and on (--log episode: AgentConfig.episode_log = 1 << 20; --log option: AgentConfig.option_log = 1 << 20;
--log trajectory: the first --trajectory-envs envs tracked, AgentConfig.trajectory_log = 1 << 20; --log occupancy: the
occupancy grid, AgentConfig.occupancy_grid = --grid), alternated --reps times in one process.  Each measurement is
--blocks blocks of run(64) + manage() (the controller's ring pass, which also fills the log) after a warm-up, timed with
CUDA events; one JSON line per measurement and a summary line with the medians.  Short episodes (--max-episode-steps) and short option executions (--option-timeout) make many
records per step.

    python tools/episode_log_cost.py [--log episode|option|trajectory|occupancy] [--trajectory-envs N] [--grid G]
                                     [--reps 3] [--blocks 10] [--out DIR]
"""
import argparse
import json
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def measure(scg, torch, capacity, args):
    if args.log == "trajectory":
        log = dict(trajectory_envs=tuple(range(args.trajectory_envs)), trajectory_log=capacity) if capacity else {}
    elif args.log == "occupancy":
        log = dict(occupancy_grid=capacity)
    else:
        log = {f"{args.log}_log": capacity}
    cfg = scg.AgentConfig(map="easy", batch=args.batch, order=3, max_options=4, sync_interval=8, seed=1,
                          max_episode_steps=args.max_episode_steps, option_timeout=args.option_timeout, **log)
    ag = scg.SkillChainAgent(cfg)
    for _ in range(2):                      # warm-up: every kernel of the block loaded, the log ring touched
        ag.run(64)
        ag.manage()
    torch.cuda.synchronize()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    ev[0].record()
    for _ in range(args.blocks):
        ag.run(64)
        ag.manage()
    ev[1].record()
    torch.cuda.synchronize()
    ms = ev[0].elapsed_time(ev[1]) / (64 * args.blocks)
    cnt = ag.counters()
    out = dict(log=args.log, capacity=capacity, ms_per_step=ms, env_steps_per_s=args.batch / (ms * 1e-3),
               episodes=int(cnt["episodes"]), option_executions=int(cnt["n_success"].sum() + cnt["n_fail"].sum()))
    if capacity and args.log == "occupancy":
        out["env_steps_counted"] = ag.occupancy()["env_steps"]
    elif capacity:
        read = dict(episode=ag.episodes, option=ag.option_executions, trajectory=ag.trajectories)[args.log]
        out["records_logged"] = read(since=1 << 62)["total"]
    del ag
    torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--blocks", type=int, default=10)
    ap.add_argument("--batch", type=int, default=65536)
    ap.add_argument("--log", default="episode", choices=["episode", "option", "trajectory", "occupancy"])
    ap.add_argument("--trajectory-envs", type=int, default=1024, help="--log trajectory: envs tracked")
    ap.add_argument("--grid", type=int, default=64, help="--log occupancy: cells per side of the grid")
    ap.add_argument("--max-episode-steps", type=int, default=100, help="short episodes: many log records per step")
    ap.add_argument("--option-timeout", type=int, default=250, help="short option executions: many option records per step")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    import skill_chaining_with_graphs_b200 as scg
    rows = []
    for _ in range(args.reps):
        for cap in (0, args.grid if args.log == "occupancy" else 1 << 20):
            rows.append(measure(scg, torch, cap, args))
            print(json.dumps(rows[-1]), flush=True)
    off = [r["ms_per_step"] for r in rows if not r["capacity"]]
    on = [r["ms_per_step"] for r in rows if r["capacity"]]
    summary = dict(device=torch.cuda.get_device_name(0), log=args.log,
                   **(dict(trajectory_envs=args.trajectory_envs) if args.log == "trajectory" else {}),
                   **(dict(grid=args.grid) if args.log == "occupancy" else {}), ms_per_step_off=off, ms_per_step_on=on,
                   median_off=float(np.median(off)), median_on=float(np.median(on)),
                   on_over_off=float(np.median(on) / np.median(off)))
    print(json.dumps(summary))
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        name = dict(trajectory=f"trajectory{args.trajectory_envs}", occupancy=f"occupancy{args.grid}").get(args.log, args.log)
        with open(os.path.join(args.out, f"{name}_log_cost.jsonl"), "w") as f:
            for r in rows + [summary]:
                f.write(json.dumps(r) + "\n")


if __name__ == "__main__":
    main()
