#!/usr/bin/env python
"""bench.py - Pinball env-steps/s including option Q-eval + Sarsa(lambda) update (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

A "step" is one lock-step agent step over the whole env batch: a fused kernel does env step (K1) ->
initiation classifiers + Q evaluation + eps-greedy + TD error (K2+K4) -> 32-byte step record, for the
`sync_interval` consecutive steps of a window in one launch (nothing couples the envs while the weights are
frozen); then the window's records are folded into the traces and weight deltas by one Sarsa(lambda) sweep
(K3, forward-view form), followed by the cross-GPU exchange and the weight apply.  The option-creation
controller (SkillChainAgent.manage: one kernel on the stream) runs every 64 steps inside the timed region.
Workload at every N: BASELINE.json configs[1] per GPU - Pinball 'easy', 65,536 envs, order-3 Fourier
basis, 4 option slots, 2 preset active logistic initiation classifiers (the controller promotes the third in the
warm-up) - weak scaling: each rank owns its own 65,536-env slice.  Synthetic data: random free-space start
states, random-init weights.

Prints ONE JSON line (rank 0).  The timed region is exactly K = --steps agent steps, cut into blocks of one sync
interval each (CUDA events at the block boundaries, max over ranks per block); `value` = env-steps of the full blocks
over all ranks / their summed time, state resident in HBM; `e2e` = K steps through SkillChainAgent.step_host
(host buffers, H2D and D2H inside the timed region) in the same blocks, with a per-step breakdown; `roofline` = the
window trace-sweep kernel's algorithmic bytes / its CUDA-event time against the measured HBM copy peak;
`cpu_baseline` = the NumPy oracle timed on this box;
`north_star_config` = the configs[2] per-GPU shape (hard map, order 5, 8 options, 131,072 envs) measured in the same
process; `sync` (N > 1) = microseconds per weight exchange, peer-memory kernel vs NCCL.
--impl reference times the stand-in reference (the NumPy oracle: the reference repository has no
code) on all host cores for the same metric.

--dump-outputs DIR writes what the timed path left after its last step (rank 0's envs) as DIR/<name>.npy, so that two
builds can be compared output for output: the same arguments give the same inputs on every run.  The weight-delta sum
uses floating-point atomics, so weights differ between runs in the last bits and an env whose arg-max is a near-tie can
take another action.  Over a short run this touches a few envs (2 of 65,536 at --steps 20 --warmup 3 on a B200); over
thousands of steps learning amplifies it and most env states differ, so compare builds on short runs.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "Pinball env-steps/s incl. option Q-eval+Sarsa(lambda) update"
UNIT = "env-steps/s"
MANAGE_EVERY = 64          # steps between calls of the option-creation controller (SkillChainAgent.manage)


def workload(args):
    return dict(map=args.map, batch=args.batch, order=args.order, max_options=args.options,
                sync_interval=args.sync_interval, gamma=0.99, lam=0.9, alpha=1e-3, epsilon=0.05, seed=0,
                option_timeout=250, max_episode_steps=2000, graph=bool(getattr(args, "graph", False)))


def wl_episode_steps(args):
    return workload(args)["max_episode_steps"]


def gpu_only(args):
    """AgentConfig fields that only the GPU backend has."""
    return dict(sync_backend=args.sync_backend, window=args.window)


def configs_label(args):
    """Which BASELINE.json config this workload is (built from the arguments, not assumed)."""
    graph = bool(getattr(args, "graph", False))
    if args.map == "easy" and args.order == 3 and args.options == 4 and args.batch == 65536 and not graph:
        return "configs[1]"
    if args.map == "hard" and args.order == 5 and args.options == 8 and args.batch == 131072:
        return "configs[4] (option-graph variant of configs[2])" if graph else "configs[2] per-GPU shape"
    return "custom" + (" (option-graph variant)" if graph else "")


def config_json(args, n_gpus):
    F = (args.order + 1) ** 4
    T = args.window or min(args.sync_interval, 8)
    return {
        "workload": f"{configs_label(args)}: Pinball '{args.map}', {args.batch} envs per GPU, order-{args.order} Fourier "
                    f"(F={F}), {args.options} option slots ({N_PRESET_ACTIVE} preset active initiation classifiers, the "
                    f"controller promotes further ones), sync every {args.sync_interval} steps",
        "controller": f"SkillChainAgent.manage() every {MANAGE_EVERY} steps inside the timed region (one kernel on the "
                      "stream: decision, classifier fit and promotion on the device)",
        "envs_per_gpu": args.batch, "global_envs": args.batch * n_gpus, "order": args.order,
        "options": args.options, "sync_interval": args.sync_interval, "map": args.map,
        "parallelism": f"env-sharded x{n_gpus}, sum of (dW, cnt) over ranks every sync interval "
                       f"({'one NVLink peer-memory exchange+apply kernel' if getattr(args, 'sync_backend', 'p2p') == 'p2p' else 'NCCL all-reduce'})",
        "episode_phase": "ep_steps uniformly random in [0, max_episode_steps) at the start (steady state of a long run)",
        "l2": f"traces {args.batch * 5 * F * 4 / 2**20:.0f} MiB per GPU > 126 MiB L2, swept once per {T}-step window "
              "(inputs larger than L2; no explicit flush)",
    }


N_PRESET_ACTIVE = 2


def setup_classifiers(theta):
    """Two synthetic active options so the classifier / termination / re-selection path runs:
    option 0 accepts x >= 0.6, option 1 accepts y <= 0.45 (quadratic features unused)."""
    theta[:] = 0
    theta[0, :3] = [-6.0, 10.0, 0.0]
    theta[1, :3] = [4.5, 0.0, -10.0]


# ---- clocks ------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.index)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
            except Exception:
                continue
            for name, v in zip(names, r[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


# ---- CPU legs (the only places that execute oracle/) ----------------------------------------------
def _cpu_worker(wl, batch, steps, seed, q, warmup=1):
    import oracle
    wl = dict(wl, batch=batch, seed=seed)
    ag = oracle.SkillChainAgent(oracle.AgentConfig(**wl))
    rng = np.random.default_rng(seed)
    ag.env.reset(states=ag.map.sample_free_states(rng, batch))
    ag.options.W[:] = (rng.standard_normal(ag.options.W.shape) * 0.1).astype(np.float32)
    setup_classifiers(ag.options.theta)
    ag.active[:N_PRESET_ACTIVE] = True
    ag.n_active = N_PRESET_ACTIVE
    ag.ep_steps[:] = rng.integers(0, wl["max_episode_steps"], batch).astype(np.int32)      # random episode phases, as on the GPU
    ag.parents[1], ag.parents[2] = (np.uint32(1 | (1 << 31)), np.uint32(3 | (1 << 31))) if wl.get("graph") else (1, 2)
    for _ in range(max(warmup, 1)):             # untimed warm-up
        ag.step()
    ag.manage()
    t0 = time.perf_counter()
    for i in range(steps):
        ag.step()
        if (i + 1) % MANAGE_EVERY == 0:         # the option-creation controller, as in run_episode
            ag.manage()
    q.put((batch * steps, time.perf_counter() - t0))


def cpu_oracle_rate(wl, batch, steps, procs, warmup=1):
    """env-steps/s of the NumPy oracle agent: `procs` processes, each its own `batch`-env agent."""
    import multiprocessing as mp
    if procs > 1:      # one single-threaded oracle per core instead of oversubscribed BLAS pools
        for v in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS"):
            os.environ[v] = "1"
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    ps = [ctx.Process(target=_cpu_worker, args=(wl, batch, steps, 1000 + i, q, warmup)) for i in range(procs)]
    t0 = time.perf_counter()
    for p in ps:
        p.start()
    res = [q.get() for _ in ps]
    for p in ps:
        p.join()
    wall = time.perf_counter() - t0
    total = sum(r[0] for r in res)
    slowest = max(r[1] for r in res)
    return total / slowest, wall


def run_reference(args):
    """The reference arm: the stand-in reference (NumPy oracle) on all host cores."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = len(os.sched_getaffinity(0))
    procs = max(1, cores)
    # bounded sample: size each step (one pass over `batch` envs per core) so K steps take about a minute
    batch = int(min(args.cpu_batch, max(256, (60 * 12000 // max(args.steps, 1)) // 256 * 256)))
    wl = workload(args)
    t_all = time.perf_counter()
    rate, _ = cpu_oracle_rate(wl, batch, args.steps, procs, warmup=min(args.warmup, 10))
    wall = time.perf_counter() - t_all
    ms = 1e3 * (batch * procs) / rate
    sample = (f"{procs} processes x {batch} envs x {args.steps} steps of the same workload "
              f"(NumPy oracle SkillChainAgent.step; the reference repository has no code)")
    line = {
        "impl": "reference", "metric": METRIC, "value": rate, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic", "config": config_json(args, args.gpus),
        "cpu_baseline": {"value": rate, "unit": UNIT, "cores": procs, "kind": "port", "sample": sample},
        "e2e": {"value": rate, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0, "wall_s": wall,
    }
    print(json.dumps(line), flush=True)


# ---- GPU arm -----------------------------------------------------------------------------------------
def k3_traffic(order, batch, T):
    """ncu dram bytes per k_window launch for this (order, envs, window) if a capture of it is committed, else None."""
    path = os.path.join(ROOT, "profiles", "k3_traffic.json")
    try:
        tj = json.load(open(path))
    except Exception:
        return None
    for e in (tj if isinstance(tj, list) else [tj]):
        if e.get("kernel") == "k_window" and e.get("order", 3) == order and e.get("envs", 65536) == batch and \
                e.get("window_steps", 8) == T:
            return e.get("dram_bytes_per_launch")
    return None


def make_agent(scg, torch, args, rank, world):
    """The bench agent: random free-space start states, random-init weights (the same on every rank), two preset
    active initiation classifiers, the third option gestating."""
    B = args.batch
    gmap = scg.PinballMap.from_name(args.map)
    rng = np.random.default_rng(1234 + rank)
    S = gmap.sample_free_states(rng, B)
    cfg = scg.AgentConfig(**workload(args), env_offset=rank * B, **gpu_only(args))
    ag = scg.SkillChainAgent(cfg, gmap, initial_states=S)
    wrng = np.random.default_rng(7)
    ag.options.set_weights((wrng.standard_normal(tuple(ag.options.W.shape)) * 0.1).astype(np.float32))
    theta = np.zeros((args.options, 6), dtype=np.float32)
    setup_classifiers(theta)
    ag.options.theta.copy_(torch.as_tensor(theta))
    ag.active_mask, ag.n_active = (1 << N_PRESET_ACTIVE) - 1, N_PRESET_ACTIVE
    # steady state of a long run: the envs are at uniformly random phases of their episodes (all of them starting
    # at step 0 would time out together 2000 steps later and restart from the one start state in lock-step)
    ag.ep_steps.copy_(torch.as_tensor(rng.integers(0, wl_episode_steps(args), B).astype(np.int32)))
    GOAL = 1 << 31
    ag.parents_host[1], ag.parents_host[2] = (1 | GOAL, 3 | GOAL) if args.graph else (1, 2)
    ag._push_parents()
    return ag


def block_sizes(steps, per_block):
    """`steps` steps as consecutive blocks of `per_block` steps; the last block holds the remainder."""
    return [per_block] * (steps // per_block) + ([steps % per_block] if steps % per_block else [])


def timed_blocks(torch, ag, sizes, barrier):
    """Exactly sum(sizes) agent steps, device-resident, as consecutive blocks of the given sizes with CUDA events at the
    block boundaries (windows, syncs and the controller's 64-step cadence run on across blocks), queued behind the work
    already on the stream.  Returns per-block milliseconds."""
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(len(sizes) + 1)]
    ev[0].record()
    t_done = 0
    for i, n in enumerate(sizes):
        left = n
        while left > 0:                                         # full skill chaining: steps + the controller
            k = min(left, MANAGE_EVERY - t_done % MANAGE_EVERY)
            ag.run(k)
            t_done += k
            left -= k
            if t_done % MANAGE_EVERY == 0:
                ag.manage()
        if i == len(sizes) - 1:
            ag.flush()                                          # a partial last window is swept inside the timed region
        ev[i + 1].record()
    barrier()
    return [ev[i].elapsed_time(ev[i + 1]) for i in range(len(sizes))]


def ms_per_step(blocks, sizes, per_block):
    """Time per step of the full blocks, or of all blocks if none is full (a last, partial block carries the sweep of
    a whole window for fewer steps)."""
    full = [b for b, n in zip(blocks, sizes) if n == per_block]
    return sum(full) / (len(full) * per_block) if full else sum(blocks) / sum(sizes)


DUMP_MAX_BYTES = 64 * 10 ** 6


def last_step_outputs(ag, max_bytes=DUMP_MAX_BYTES):
    """What a caller of SkillChainAgent.run holds after its last step, as float32 / float64 arrays: per env the state,
    reward, termination flags (bit fields, exact in float64), next action, option and TD error, and the option weights.
    If the per-env arrays would pass `max_bytes`, a fixed seeded sample of the envs is kept and `env_index` names them."""
    per_env = dict(state=ag.state.cpu().numpy(), reward=ag.reward.cpu().numpy(),
                   flags=ag.flags.cpu().numpy().view(np.uint32).astype(np.float64),
                   action=ag.action.cpu().numpy().astype(np.float32), option=ag.option.cpu().numpy().astype(np.float32),
                   td_error=ag.delta.cpu().numpy())
    out = dict(weights=ag.options.W.cpu().numpy())
    B = len(per_env["reward"])
    bytes_per_env = sum(a.nbytes for a in per_env.values()) // max(B, 1) + 8      # + 8: its env_index entry
    n = min(B, (max_bytes - out["weights"].nbytes) // bytes_per_env)
    if n < B:
        idx = np.sort(np.random.default_rng(0).choice(B, n, replace=False))
        out["env_index"] = idx.astype(np.float64)
        per_env = {k: v[idx] for k, v in per_env.items()}
    out.update(per_env)
    return out


def stage_pass(torch, ag, T, n_windows=8):
    """Untimed-by-the-headline side pass: CUDA events around every launch kind (costs ~5 us per step, so it is not done
    in the timed region): -> (ms per launch, launches) for [fused step, sweep, dW reduction, apply / exchange]."""
    n_side = n_windows * T
    ag.profile_begin(8 * n_side + 16, kinds=(0, 1, 2, 3, 4, 5))
    ag.run(n_side)
    ag.manage()
    torch.cuda.synchronize()
    ms, n = ag.profile_end()
    return [ms[k] / n[k] if n[k] else 0.0 for k in range(len(ms))], n, n_side


def run_ours(args):
    import torch
    import torch.distributed as dist
    import skill_chaining_with_graphs_b200 as scg

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise scg.ScgError("bench.py needs a GPU (no CPU fallback); use --impl reference for the CPU arm")
    torch.cuda.set_device(local)
    if world > 1 and args.pin_cores:
        # one process per GPU: give each rank its own slice of the host cores (its launch thread, its copies' staging and
        # the NCCL helper threads then do not migrate over the other ranks' cores)
        cores = sorted(os.sched_getaffinity(0))
        per = len(cores) // world
        if per >= 1:
            os.sched_setaffinity(0, set(cores[local * per:(local + 1) * per]))
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("MASTER_PORT", "29500")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    lib = scg.load_library()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def reduce_max(vals):
        if world == 1:
            return [float(v) for v in vals]
        t = torch.tensor(vals, dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return [float(v) for v in t]

    def measure(a, steps, n_warm, live_kind=True, dump=False):
        """Warm up, then time exactly `steps` steps in blocks of one sync interval -> dict of per-rank-max block times
        and kernel timings (and, with dump=True, the outputs of the last timed step)."""
        ag = make_agent(scg, torch, a, rank, world)
        backend = a.sync_backend
        if world > 1 and a.sync_backend == "p2p" and ag._xchg is None:
            backend = "nccl"                                   # the agent fell back (it said why on stderr): report what ran
        B, T = a.batch, ag.win_cap
        ag.warm_up_controller()
        if live_kind:                                           # create the profiling events before the queue is filled
            ag.profile_begin(steps + 64, kinds=(1,))
            ag.profile_end()
        for lo in range(0, n_warm, MANAGE_EVERY):
            ag.run(min(MANAGE_EVERY, n_warm - lo))
        ag.manage()                                             # the preset gestating option qualifies within the warm-up
        barrier()
        # the controller period after that promotion runs ~5 % slower than the steady state, so it ends the warm-up; it is
        # queued after the barrier so that the GPU is still busy with it when the timed region starts (the first block
        # then carries no launch latency)
        ag.run(MANAGE_EVERY)
        ag.manage()
        launches0 = lib.scg_launch_count()
        if live_kind:
            ag.profile_begin(steps + 64, kinds=(1,))               # events around the dominant kernel only, live
        sizes = block_sizes(steps, a.sync_interval)
        t0 = ag.t
        blocks = timed_blocks(torch, ag, sizes, barrier)
        steps_run = ag.t - t0                                   # the library's own step counter
        live_ms, live_n = ag.profile_end() if live_kind else ([0.0] * 6, [0] * 6)
        launches = lib.scg_launch_count() - launches0
        outputs = last_step_outputs(ag) if dump else None
        blocks = reduce_max(blocks)                             # per block: the slowest rank
        side_ms, side_n, n_side = stage_pass(torch, ag, T)
        if ag.peer_sync_timed_out():
            raise scg.ScgError("a cross-GPU weight exchange timed out during the bench: no valid number")
        per_step = ms_per_step(blocks, sizes, a.sync_interval)
        k3_ms = live_ms[1] / live_n[1] if live_n[1] else side_ms[1]
        return dict(ag=ag, backend=backend, blocks=blocks, sizes=sizes, steps_run=steps_run, ms_per_step=per_step, k3_ms=k3_ms,
                    k3_launches=live_n[1], side_ms=side_ms, side_n=side_n, n_side=n_side, launches=launches,
                    ctl=ag.controller_state(sync=True), outputs=outputs)

    n_warm = max(args.warmup, 16)          # at least two windows, so the preset gestating option has qualified by the end
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    m = measure(args, args.steps, n_warm, dump=bool(args.dump_outputs))
    ag, B, T = m["ag"], args.batch, m["ag"].win_cap
    args.sync_backend = m["backend"]
    dumped = None
    if m["outputs"] is not None and rank == 0:
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, arr in m["outputs"].items():
            np.save(os.path.join(args.dump_outputs, name + ".npy"), arr)
        dumped = {"dir": args.dump_outputs, "bytes": sum(arr.nbytes for arr in m["outputs"].values()),
                  "envs": len(m["outputs"]["reward"]), "arrays": sorted(m["outputs"])}
    # ---- e2e: K steps through the host-buffer API, in the same blocks ----
    def e2e_blocks(step_fns):
        out = []
        for fn in step_fns:
            barrier()
            t0 = time.perf_counter()
            fn()
            torch.cuda.synchronize()
            out.append((time.perf_counter() - t0) * 1e3)
        return reduce_max(out)

    hs = ag.s.cpu().numpy().copy()
    ha = ag.action.cpu().numpy().copy()
    host = dict(s=hs, a=ha, i=0)

    def host_steps(n):
        for _ in range(n):
            s2, r, f, a2, d = ag.step_host(host["s"], host["a"])
            host["s"], host["a"] = s2, a2                       # views of the pinned result buffers, fed straight back
            host["i"] += 1
            if host["i"] % MANAGE_EVERY == 0:
                ag.manage()

    for _ in range(3):
        host["s"], r, f, host["a"], d = ag.step_host(host["s"], host["a"])
    e2e = e2e_blocks([lambda n=n: host_steps(n) for n in m["sizes"]])
    e2e_ms = ms_per_step(e2e, m["sizes"], args.sync_interval) * args.steps

    # where an end-to-end step goes: the pieces timed one by one with CUDA events (pinned host buffers, this stream)
    def ev_time(fn, reps=20):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        fn()
        torch.cuda.synchronize()
        a.record()
        for _ in range(reps):
            fn()
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b) / reps * 1e3

    hbuf = ag._host[0]
    dS, dO = ag.s.clone(), ag._out.clone()
    pin_out = torch.empty((4, B), dtype=torch.float32).pin_memory()
    brk = {
        "h2d_state_action_us": ev_time(lambda: (ag.s.copy_(hbuf["s"], non_blocking=True), ag.action.copy_(hbuf["a"], non_blocking=True))),
        "d2h_state_results_us": ev_time(lambda: (hbuf["s2"].copy_(dS, non_blocking=True), pin_out.copy_(dO, non_blocking=True))),
    }

    def one_step():
        ag.invalidate()
        ag.step()

    # the single-step launches themselves, from the library's own events around each launch (a Python loop of 40 us
    # calls would time the host, not the kernel)
    ag.profile_begin(4 * ag.win_cap + 8, kinds=(0,))
    for _ in range(2 * ag.win_cap):
        one_step()
    torch.cuda.synchronize()
    ms1, n1 = ag.profile_end()
    brk["step_kernel_single_step_requeried_q_us"] = ms1[0] / max(n1[0], 1) * 1e3
    brk["sweep_reduce_apply_ring_per_step_us"] = (m["k3_ms"] + m["side_ms"][2] + m["side_ms"][3] + m["side_ms"][4]) * 1e3 / ag.win_cap
    brk["measured_total_us"] = e2e_ms * 1e3 / args.steps
    resid = brk["measured_total_us"] - sum(v for k, v in brk.items() if k != "measured_total_us")
    brk["host_and_launch_latency_us"] = max(resid, 0.0)
    if resid < 0:      # the pieces overlap in the pipelined host step (and are timed after the end-to-end blocks)
        brk["pieces_exceed_total_by_us"] = -resid
    brk["note"] = ("pieces timed one by one; scg_agent_step_host pipelines them over 2 parts of the batch (copy in / step / copy "
                   "out on three streams), so they add up to more than the total; the sweep / apply chain of a full window "
                   "must finish before the next step's Q evaluation")
    # informational: the same loop for a caller that needs the state only once per sync interval (run_host)
    Ts = args.sync_interval
    hw = dict(s=ag.s.cpu().numpy().copy(), a=ag.action.cpu().numpy().copy())
    n_calls = max(args.steps // Ts, 1)

    def host_window():
        hw["s"], hw["a"], r, f, d = ag.run_host(hw["s"], hw["a"], Ts)

    host_window()
    e2e_win_ms = float(np.median(e2e_blocks([host_window] * n_calls)))
    clocks = sampler.stop() if rank == 0 else None
    # ---- cross-GPU sync: the peer-memory kernel against two NCCL all-reduces + apply on the same payload ----
    sync_cmp = None
    if world > 1:
        from skill_chaining_with_graphs_b200.sync import allreduce_deltas
        o = ag.options
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
        reps = 50
        for i in range(reps + 5):
            if i == 5:
                barrier()
                ev[0].record()
            allreduce_deltas(o._dW, o._cnt, ag.pg)
            o.apply()
        ev[1].record()
        torch.cuda.synchronize()
        nccl_us = reduce_max([ev[0].elapsed_time(ev[1]) / reps * 1e3])[0]
        sync_cmp = {"p2p_kernel_us": reduce_max([m["side_ms"][3] * 1e3])[0] if m["backend"] == "p2p" else None,
                    "nccl_allreduce_x2_plus_apply_us": nccl_us, "payload_bytes": int(o._dW.numel() * 4 + o._cnt.numel() * 4),
                    "note": "per sync, max over ranks; the p2p figure includes the wait for the slowest rank to arrive"}
    # ---- the north-star configuration, in the same process, at every N ----
    north = None
    if not args.no_north_star and configs_label(args) == "configs[1]":
        del ag, m["ag"]
        torch.cuda.empty_cache()
        na = argparse.Namespace(**vars(args))
        na.map, na.order, na.options, na.batch, na.window = "hard", 5, 8, 131072, 0
        nm = measure(na, 320, 16)
        F5 = 6 ** 4
        nb = 8 * 5 * F5 + 32 * nm["ag"].win_cap
        north = {"workload": config_json(na, world)["workload"], "value": na.batch * world / (nm["ms_per_step"] * 1e-3),
                 "unit": UNIT, "ms_per_step": nm["ms_per_step"], "steps": 320, "steps_per_block": na.sync_interval,
                 "blocks_ms": nm["blocks"],
                 "n_active_end": nm["ctl"]["n_active"],
                 "k_window": {"avg_launch_ms": nm["k3_ms"], "achieved_gbs": na.batch * nb / (nm["k3_ms"] * 1e-3) / 1e9 if nm["k3_ms"] else None,
                              "algorithmic_bytes_per_launch": na.batch * nb},
                 "stages_ms_per_launch": {"fused_step": nm["side_ms"][0], "k3_window_sweep": nm["side_ms"][1],
                                          "dw_reduce": nm["side_ms"][2], "apply_or_exchange": nm["side_ms"][3],
                                          "example_ring_pass": nm["side_ms"][4], "controller": nm["side_ms"][5]}}
        del nm
    if rank == 0:
        F = (args.order + 1) ** 4
        total_env_steps = B * world * args.steps
        value = B * world / (m["ms_per_step"] * 1e-3)
        peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
        if os.path.exists(peaks_path):
            peak, which = float(json.load(open(peaks_path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        else:
            peak, which = 6650.0, "fallback (B200_PROFILING.md)"
        bytes_per_env = 8 * 5 * F + 32 * T              # trace read + write once per window, T 32-byte records
        k3_ms = m["k3_ms"]
        achieved = B * bytes_per_env / (k3_ms * 1e-3) / 1e9 if k3_ms > 0 else 0.0
        side, side_n, n_side = m["side_ms"], m["side_n"], m["n_side"]
        per_step = [side[k] * side_n[k] / n_side for k in range(4)]     # ms per agent step of each stage (side pass)
        per_step[1] = k3_ms * (side_n[1] / n_side)                      # the sweep: its live timing
        tot = sum(per_step)
        if north is not None:
            north["k_window"]["frac_of_hbm_peak"] = (north["k_window"]["achieved_gbs"] or 0.0) / peak
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": m["ms_per_step"], "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": config_json(args, world),
            "timed_region": {"steps": args.steps, "steps_run": m["steps_run"], "total_ms": sum(m["blocks"]),
                             "blocks": len(m["blocks"]), "steps_per_block": args.sync_interval,
                             "block_ms_min": min(m["blocks"]), "block_ms_max": max(m["blocks"]), "blocks_ms": m["blocks"],
                             "warmup_steps_run": n_warm + MANAGE_EVERY,
                             "note": "exactly `steps` steps, in blocks of one sync interval (its fused steps, trace sweeps "
                                     "and weight apply; the last block takes the remainder and the sweep of a partial "
                                     "window), each bracketed by CUDA events, max over ranks per block; value = steps of "
                                     "the full blocks / their summed time (of all blocks if none is full); the controller "
                                     "runs every 64 steps inside the timed region"},
            "roofline": {"kernel": "k_window (K3 Sarsa(lambda) trace sweep, forward-view window form)", "bound": "hbm",
                         "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": k3_traffic(args.order, B, T),
                         "peak_source": which, "algorithmic_bytes_per_launch": B * bytes_per_env,
                         "bytes_per_env_step": bytes_per_env / T, "window_steps": T,
                         "avg_launch_ms": k3_ms, "launches": m["k3_launches"],
                         "share_of_step": (per_step[1] / tot) if tot else None},
            "stages_ms_per_step": {"fused_step_k1_k2_k4": per_step[0], "k3_window_sweep": per_step[1],
                                   "dw_reduce": per_step[2], "apply": per_step[3],
                                   "example_ring_pass": side[4] * side_n[4] / n_side,
                                   "controller_kernel_ms_per_launch": side[5],
                                   "fused_step_avg_launch_ms": side[0], "steps_per_fused_launch": n_side / max(side_n[0], 1),
                                   "note": "k3_window_sweep timed live in the timed region; the other stages in a separate "
                                           f"{n_side}-step pass (events around every launch cost ~5 us per step)"},
            # north_star also asks for the FP32 view of the feature + Q part (K2): 18 F flop per env-step, counted
            # against the nominal FP32 FMA rate at the maximum SM clock (148 SMs x 128 lanes x 2 flop)
            "k2_fp32": {"kernel": "k_agent_step (K1+K2+K4; only K2's 18*F flop per env-step are counted)",
                        "flop_per_env_step": 18 * F, "achieved_tflops": B * 18 * F / (per_step[0] * 1e-3) / 1e12
                        if per_step[0] > 0 else None, "peak_tflops_nominal": 148 * 128 * 2 * 1.965e9 / 1e12},
            "e2e": {"value": total_env_steps / (e2e_ms * 1e-3), "unit": UNIT,
                    "h2d_bytes_per_step": B * scg.SkillChainAgent.HOST_H2D_BYTES_PER_ENV,
                    "d2h_bytes_per_step": B * scg.SkillChainAgent.HOST_D2H_BYTES_PER_ENV,
                    "blocks_ms": e2e, "breakdown_per_step": brk,
                    "api": "SkillChainAgent.step_host -> scg_agent_step_host (pinned host buffers)"},
            "e2e_per_sync_interval": {"value": B * world * Ts / (e2e_win_ms * 1e-3), "unit": UNIT, "calls": n_calls,
                                      "h2d_bytes_per_call": B * 20, "d2h_bytes_per_call": B * 32, "steps_per_call": Ts,
                                      "api": "SkillChainAgent.run_host: host state in / out once per sync interval "
                                             "(informational; `e2e` above copies every step)"},
            "controller_state_end": m["ctl"], "sync": sync_cmp, "north_star_config": north,
            "gpu_launches": int(m["launches"]), "clocks": clocks, "dump_outputs": dumped,
        }
        if world == 1 and not args.no_cpu:
            cores = max(1, len(os.sched_getaffinity(0)))
            rate, wall = cpu_oracle_rate(workload(args), args.cpu_batch, args.cpu_steps, cores)
            line["cpu_baseline"] = {
                "value": rate, "unit": UNIT, "cores": cores, "kind": "port",
                "sample": f"NumPy oracle SkillChainAgent.step, {args.cpu_batch} envs x {args.cpu_steps} steps of the "
                          f"same workload in each of {cores} single-threaded processes ({wall:.1f} s wall)"}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=2000, help="timed agent steps")
    ap.add_argument("--warmup", type=int, default=16)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--map", default="easy")
    ap.add_argument("--batch", type=int, default=65536, help="envs per GPU")
    ap.add_argument("--order", type=int, default=3)
    ap.add_argument("--options", type=int, default=4)
    ap.add_argument("--sync-interval", type=int, default=8)
    ap.add_argument("--cpu-batch", type=int, default=4096)
    ap.add_argument("--cpu-steps", type=int, default=40)
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--sync-backend", default="p2p", choices=["p2p", "nccl"])
    ap.add_argument("--window", type=int, default=0, help="steps per trace sweep (0 = min(sync interval, 8))")
    ap.add_argument("--pin-cores", type=int, default=0, help="N > 1: pin each rank to its own slice of the host cores")
    ap.add_argument("--no-north-star", action="store_true", help="skip the extra configs[2]-shape measurement")
    ap.add_argument("--graph", action="store_true", help="option-graph variant (configs[4]): an option's targets are the "
                    "initiation sets of ALL earlier options and the goal, so chains merge")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed step (rank 0's envs) to DIR/<name>.npy, at most 64 MB")
    args = ap.parse_args()
    if args.steps < 1 or args.sync_interval < 1:
        ap.error("--steps and --sync-interval must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the GPU path's outputs (--impl ours)")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
