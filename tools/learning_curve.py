#!/usr/bin/env python
"""Train the skill-chaining agent and write its learning curves from the device episode log (AgentConfig.episode_log):
every finished episode's return, length and whether it reached the goal, binned against env-steps and against episodes.

    python tools/learning_curve.py --map easy --batch 65536 --options 4 [--no-top-level] --steps 6000 --out DIR

The agent runs in chunks of --chunk steps with the option-creation controller (manage()) after each; after each chunk
episodes(since=...) returns the episodes finished since the last poll, so no episode is lost as long as one chunk
produces fewer than --capacity of them (the number lost, if any, is reported).  Output, in DIR:
  curve_env_steps.jsonl   one line per bin of agent steps: env_steps (at the bin's end), episodes, mean_return,
                          goal_rate, mean_length
  curve_episodes.jsonl    one line per bin of consecutive episodes in (step, env) order: the same fields, with
                          episodes_end (episodes finished by the bin's end) in place of env_steps
  summary.json            configuration, device, totals, the controller's promotions and the wall time
With --option-log CAP the device option log (AgentConfig.option_log) is polled after each chunk as well, and
  options_env_steps.jsonl one line per (bin of agent steps, option): executions that ended in the bin, hit_rate,
                          label_rate, mean_duration, the count of each outcome flag, and env_step_share - the summed
                          durations of those executions over the bin's env-steps (the share of the batch's time spent in
                          the option, credited to the bin in which each execution ended)
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def device_info(torch):
    """Card name and power limit as the driver reports them (read only)."""
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=30).stdout.strip().splitlines()
        if out:
            name, limit = (v.strip() for v in out[0].split(","))
            info.update(smi_name=name, power_limit=limit)
    except Exception as e:      # the curve does not depend on it
        info["power_limit"] = f"unavailable ({e})"
    return info


def bin_rows(idx_end, ret, length, goal, edges):
    """Bins [edges[i], edges[i+1]) of the sorted key idx_end -> (n, mean return, goal rate, mean length) per bin."""
    lo = np.searchsorted(idx_end, edges[:-1], side="left")
    hi = np.searchsorted(idx_end, edges[1:], side="left")
    rows = []
    for a, b in zip(lo, hi):
        n = int(b - a)
        rows.append(dict(episodes=n,
                         mean_return=float(ret[a:b].astype(np.float64).mean()) if n else None,
                         goal_rate=float(goal[a:b].mean()) if n else None,
                         mean_length=float(length[a:b].astype(np.float64).mean()) if n else None))
    return rows


class OptionTally:
    """Running sums over option-log records (SkillChainAgent.option_executions) per (bin of agent steps, option):
    executions, summed duration and the count of each outcome flag.  Records are added as they are polled, so a long run
    needs no more host memory than its bins."""

    def __init__(self, edges, n_options):
        from skill_chaining_with_graphs_b200.agent import OPTION_OUTCOMES
        self.outcomes = OPTION_OUTCOMES
        self.edges = np.asarray(edges, dtype=np.int64)
        shape = (len(self.edges) - 1, n_options)
        self.n, self.dur = np.zeros(shape, np.int64), np.zeros(shape, np.int64)
        self.flags = {k: np.zeros(shape, np.int64) for k in OPTION_OUTCOMES}

    def add(self, log):
        b = np.searchsorted(self.edges, log["step"].astype(np.int64), side="right") - 1
        keep = (b >= 0) & (b < self.n.shape[0])
        at = (b[keep], log["option"][keep])
        np.add.at(self.n, at, 1)
        np.add.at(self.dur, at, log["duration"][keep].astype(np.int64))
        for k in self.outcomes:
            np.add.at(self.flags[k], at, log[k][keep].astype(np.int64))

    def rows(self, i, env_steps):
        """One dict per option for bin i, whose agent steps amount to `env_steps` env-steps."""
        out = []
        for o in range(self.n.shape[1]):
            n = int(self.n[i, o])
            row = dict(option=o, executions=n,
                       hit_rate=self.flags["hit"][i, o] / n if n else None,
                       label_rate=self.flags["label"][i, o] / n if n else None,
                       mean_duration=self.dur[i, o] / n if n else None)
            row.update({k: int(self.flags[k][i, o]) for k in self.outcomes})
            row["env_step_share"] = float(self.dur[i, o]) / env_steps if env_steps else None
            out.append({k: float(v) if isinstance(v, np.floating) else v for k, v in row.items()})
        return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--map", default="easy")
    ap.add_argument("--batch", type=int, default=65536)
    ap.add_argument("--order", type=int, default=3)
    ap.add_argument("--options", type=int, default=4)
    ap.add_argument("--no-top-level", action="store_true", help="choose options 'first active' instead of by Q_top")
    ap.add_argument("--steps", type=int, default=6000, help="agent steps (each steps every env once)")
    ap.add_argument("--chunk", type=int, default=128, help="steps between polls of the log (and manage() calls)")
    ap.add_argument("--capacity", type=int, default=1 << 20, help="episode log ring, in records")
    ap.add_argument("--max-episode-steps", type=int, default=500)
    ap.add_argument("--option-timeout", type=int, default=100)
    ap.add_argument("--gestation-successes", type=int, default=256)
    ap.add_argument("--alpha", type=float, default=2e-3)
    ap.add_argument("--epsilon", type=float, default=0.1)
    ap.add_argument("--sync-interval", type=int, default=8)
    ap.add_argument("--bins", type=int, default=50)
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--option-log", type=int, default=0, metavar="CAP",
                    help="also log every option execution (option log ring of CAP records) and write options_env_steps.jsonl")
    ap.add_argument("--out", required=True)
    args = ap.parse_args()

    import torch
    import skill_chaining_with_graphs_b200 as scg
    if not torch.cuda.is_available():
        raise SystemExit("learning_curve.py needs a CUDA device")
    cfg = scg.AgentConfig(map=args.map, batch=args.batch, order=args.order, max_options=args.options,
                          alpha=args.alpha, epsilon=args.epsilon, sync_interval=args.sync_interval, seed=args.seed,
                          option_timeout=args.option_timeout, max_episode_steps=args.max_episode_steps,
                          gestation_successes=args.gestation_successes, top_level=not args.no_top_level,
                          episode_log=args.capacity, option_log=args.option_log)
    ag = scg.SkillChainAgent(cfg)
    parts, seen, lost = [], 0, 0
    # against env-steps: bins of agent steps; an episode that ended at agent step t belongs to env-step (t + 1) * batch
    edges = np.linspace(0, args.steps, args.bins + 1).round().astype(np.int64)
    tally = OptionTally(edges, args.options) if args.option_log else None
    opt_seen = opt_lost = 0
    t0 = time.time()
    done = 0
    while done < args.steps:
        n = min(args.chunk, args.steps - done)
        ag.run(n)
        done += n
        ag.manage()
        new = ag.episodes(since=seen)
        lost += new["total"] - seen - len(new["step"])
        seen = new["total"]
        parts.append(new)
        if tally is not None:
            ex = ag.option_executions(since=opt_seen)
            opt_lost += ex["total"] - opt_seen - len(ex["step"])
            opt_seen = ex["total"]
            tally.add(ex)
    torch.cuda.synchronize()
    wall = time.time() - t0
    log = {k: np.concatenate([p[k] for p in parts]) for k in ("step", "env", "ret", "length", "goal")}
    ctl = ag.controller_state(sync=True)

    os.makedirs(args.out, exist_ok=True)
    step = log["step"].astype(np.int64)
    with open(os.path.join(args.out, "curve_env_steps.jsonl"), "w") as f:
        for e, row in zip(edges[1:], bin_rows(step, log["ret"], log["length"], log["goal"], edges)):
            f.write(json.dumps(dict(env_steps=int(e) * args.batch, **row)) + "\n")
    # against episodes: bins of consecutive episodes (the log is in (step, env) order)
    n_ep = len(step)
    eedges = np.linspace(0, n_ep, min(args.bins, max(n_ep, 1)) + 1).round().astype(np.int64)
    with open(os.path.join(args.out, "curve_episodes.jsonl"), "w") as f:
        for e, row in zip(eedges[1:], bin_rows(np.arange(n_ep), log["ret"], log["length"], log["goal"], eedges)):
            f.write(json.dumps(dict(episodes_end=int(e), **row)) + "\n")
    summary = dict(config={k: v for k, v in vars(args).items() if k != "out"}, device=device_info(torch),
                   agent_steps=done, env_steps=done * args.batch, episodes=int(seen), episodes_lost=int(lost),
                   goals=int(log["goal"].sum()), mean_return=float(log["ret"].astype(np.float64).mean()) if n_ep else None,
                   n_active_end=ctl["n_active"], promotions=ctl["n_promotions"], wall_s=wall)
    if tally is not None:
        with open(os.path.join(args.out, "options_env_steps.jsonl"), "w") as f:
            for i, e in enumerate(edges[1:]):
                for row in tally.rows(i, int(edges[i + 1] - edges[i]) * args.batch):
                    f.write(json.dumps(dict(env_steps=int(e) * args.batch, **row)) + "\n")
        summary.update(option_executions=int(opt_seen), option_executions_lost=int(opt_lost))
    with open(os.path.join(args.out, "summary.json"), "w") as f:
        json.dump(summary, f, indent=1)
    print(json.dumps(summary))


if __name__ == "__main__":
    main()
