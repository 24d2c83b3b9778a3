"""Batched skill-chaining agent on B200: the fused lock-step step (one kernel: K1 + K2 + K4), the
windowed Sarsa(lambda) sweep (K3, once per window), the low-rate option-creation controller, and the
cross-GPU weight-delta sync.  Same interface and semantics as the CPU oracle's SkillChainAgent
(oracle/agent.py, which stands in for the reference - the reference has no code:
/root/reference/README.md:1-2).

    agent = SkillChainAgent(AgentConfig(map="easy", batch=65536, max_options=4))
    stats = agent.run_episode(max_steps=2000)

Multi-GPU: one process per GPU, each owning a contiguous env slice (`env_offset`); every
`sync_interval` steps dW and cnt are summed over ranks by ONE kernel over NVLink peer memory (k_sync,
csrc/scg_xchg.cu; `sync_backend="nccl"` keeps an NCCL all-reduce path) and every rank applies the same update
(weights stay bit-identical across ranks).

The option-creation controller runs on the device (csrc/scg_ctl.cu): manage() queues one kernel that checks the
gestating option's success count, fits its initiation classifier on its example ring (across ranks: on the union of
the ranks' rings, exchanged over peer memory) and promotes it in device memory; the host only learns of it from a
host-mapped mirror and never waits for the device.
"""
import ctypes as C
from dataclasses import dataclass

import numpy as np

from . import _lib
from ._lib import check, ptr, AgentStruct, CtlStruct, GOAL_BIT, N_ACTIONS
from .option import OptionSet
from .pinball import PinballMap
from .sync import allreduce_deltas, allreduce_scalar_sum, fit_union, world_size


@dataclass
class AgentConfig:
    map: str = "easy"
    batch: int = 1
    order: int = 3
    max_options: int = 4
    gamma: float = 0.99
    lam: float = 0.9
    alpha: float = 1e-3
    epsilon: float = 0.05
    sync_interval: int = 1
    seed: int = 0
    env_offset: int = 0
    option_bonus: float = 1000.0
    option_timeout: int = 250
    max_episode_steps: int = 2000
    gestation_successes: int = 32
    example_capacity: int = 4096
    clf_steps: int = 200
    clf_lr: float = 1.0
    event_history: int = 64       # steps of option-termination events kept on the device between example-ring passes
    episode_log: int = 0          # records in the device episode log ring (every finished episode: step, env, return,
                                  # length, goal; read with episodes()); 0: no log
    option_log: int = 0           # records in the device option log ring (every option execution: step, env, option,
                                  # duration, outcome, start and end; read with option_executions()); 0: no log
    trajectory_envs: tuple = ()   # local indices of the envs whose every step is logged on the device (state, action,
                                  # option, TD error, outcome; read with trajectories()); () with trajectory_log = 0: no log
    trajectory_log: int = 0       # records in the device trajectory log ring (32 bytes each, len(trajectory_envs) per step)
    occupancy_grid: int = 0       # G: every env-step counted on the device by (option, cell of a G x G grid over the map);
                                  # read with occupancy().  A power of two in 1..128; 0: no grid
    init_horizon: int = 1 << 30   # an example is positive iff the option hit a target within this many steps of its start
    merge_overlap: float = 0.0    # graph mode: an older option's initiation set becomes a target of the next option iff at
                                  # least this fraction of the promoted option's positive examples lies inside it (0: all)
    graph: bool = False
    cull: bool = True
    window: int = 0          # steps per trace sweep; 0 = min(sync_interval, 8)
    deterministic: bool = False   # fixed-order reduction of the weight deltas: runs reproduce bit for bit (slightly slower)
    sync_backend: str = "p2p"   # multi-rank weight-delta exchange: "p2p" (one kernel over NVLink peer memory) or "nccl"
    top_level: bool = False     # option choice by the learned SMDP value function Q_top (oracle/agent.py) instead of "first active"
    alpha_top: float = 1e-3
    epsilon_top: float = 0.05
    sync_timeout_s: float = 30.0   # how long a peer-memory exchange waits for the other ranks before failing (ScgError)

    def __post_init__(self):
        occupancy_grid_size(self.occupancy_grid)


OCCUPANCY_GRID_MAX = 128


def occupancy_grid_size(g):
    """AgentConfig.occupancy_grid as an int: 0 (off) or a power of two in 1..OCCUPANCY_GRID_MAX; else ValueError."""
    if isinstance(g, bool) or int(g) != g or not (g == 0 or (1 <= g <= OCCUPANCY_GRID_MAX and int(g) & (int(g) - 1) == 0)):
        raise ValueError(f"occupancy_grid must be 0 (off) or a power of two in 1..{OCCUPANCY_GRID_MAX}, not {g!r}")
    return int(g)


class SkillChainAgent:
    def __init__(self, cfg, pmap=None, process_group=None, initial_states=None):
        import torch
        if not torch.cuda.is_available():
            raise _lib.ScgError("SkillChainAgent needs a CUDA device: there is no CPU fallback")
        self.torch = torch
        self.lib = _lib.load()
        self.cfg = cfg
        self.map = pmap if pmap is not None else PinballMap.from_name(cfg.map)
        self.pg = process_group
        B, K = cfg.batch, cfg.max_options
        dev = torch.device("cuda", torch.cuda.current_device())
        self.device = dev
        self.top_slots = -(-K // N_ACTIONS) if cfg.top_level else 0
        self.options = OptionSet(K, cfg.order, B, cfg.gamma, cfg.lam, cfg.alpha, cfg.epsilon, cfg.seed,
                                 cfg.env_offset, dev, deterministic=cfg.deterministic, top_slots=self.top_slots,
                                 alpha_top=cfg.alpha_top)
        self.options._pre_read = self.flush        # dW / trace reads see the open window folded in
        f32 = dict(dtype=torch.float32, device=dev)
        i32 = dict(dtype=torch.int32, device=dev)
        self.win_cap = int(cfg.window) if cfg.window else max(1, min(int(cfg.sync_interval), 8))
        if not 1 <= self.win_cap <= _lib.WIN_MAX:
            raise ValueError(f"window must be in 1..{_lib.WIN_MAX}")
        self._sbuf = (torch.zeros((4, B), **f32), torch.zeros((4, B), **f32))
        # reward, flags, action, delta back to back: the host-buffer step returns them with one copy
        self._out = torch.zeros((4, B), **f32)
        self.reward, self.delta = self._out[0], self._out[3]
        self.flags, self.action = self._out[1].view(torch.int32), self._out[2].view(torch.int32)
        self.option = torch.zeros(B, **i32)
        self.t_opt = torch.zeros(B, **i32)
        self.ep_steps = torch.zeros(B, **i32)
        self.start_xy = torch.zeros((B, 2), **f32)
        self.ep_return = torch.zeros(B, **f32)
        self.ep_count = torch.zeros(B, **i32)               # finished episodes per env
        self.last_return = torch.zeros(B, **f32)            # task return of each env's last finished episode
        self.q_carry = torch.zeros(B, **f32)
        self.win_rec = torch.zeros((self.win_cap, B, 8), **f32)
        # option-termination events (one byte per env-step + the option's start position) wait here until the
        # controller needs the example rings: one ring pass per manage() instead of one per window
        self.ev_cap = max(int(cfg.event_history), 2 * self.win_cap)
        self.ev_hist = torch.zeros((self.ev_cap, max(B, 1)), dtype=torch.uint8, device=dev)
        self.ev_pos = torch.zeros((self.ev_cap, max(B, 1), 2), **f32)
        # top-level learner: s0 = (start_xy, start_vxy), discounted return and discount of the running option, and the
        # SMDP update records of the open window
        self.start_vxy = torch.zeros((B, 2), **f32)
        self.opt_ret = torch.zeros(B, **f32)
        self.opt_disc = torch.ones(B, **f32)
        self.win_top = torch.zeros((self.win_cap if cfg.top_level else 0, max(B, 1), 8), **f32)
        # controller state: a device block (struct scg_ctl) the kernels read and scg_agent_manage updates in place
        self.ctl = torch.zeros(32, **i32)
        self._ctl = CtlStruct()
        self._ctl.parents[0] = GOAL_BIT
        self.parents_host = np.ctypeslib.as_array(self._ctl.parents)[:K]     # view: edit, then _push_parents()
        self._ex_xy = torch.zeros((K, cfg.example_capacity, 2), **f32)
        self._ex_label = torch.zeros((K, cfg.example_capacity), dtype=torch.uint8, device=dev)
        self._ex_count = torch.zeros(K, dtype=torch.int64, device=dev)
        # (sized for every weight slot: the cross-GPU exchange carries one success counter per slot)
        self._n_success = torch.zeros(_lib.MAX_OPTIONS, **i32)
        self._n_fail = torch.zeros(_lib.MAX_OPTIONS, **i32)
        self._n_success_global = torch.zeros(_lib.MAX_OPTIONS, **i32)
        self.n_success, self.n_fail, self.n_success_global = self._n_success[:K], self._n_fail[:K], self._n_success_global[:K]
        self.stats = torch.zeros(4, dtype=torch.int64, device=dev)
        # episode log (optional): the step kernel marks episode ends in the event bytes and keeps (return, length) in
        # ev_ep; the ring pass appends them to the log ring _ep_log ([capacity][4]: step, env, return bits,
        # length | goal << 31) and counts them in _ep_log_count
        if int(cfg.episode_log) < 0:
            raise ValueError("episode_log must be >= 0")
        if cfg.episode_log:
            self.ev_ep = torch.zeros((self.ev_cap, max(B, 1), 2), **f32)
            self._ep_log = torch.zeros((int(cfg.episode_log), 4), **i32)
            self._ep_log_count = torch.zeros(1, dtype=torch.int64, device=dev)
        else:
            self.ev_ep = self._ep_log = self._ep_log_count = None
        # option log (optional): at every termination the step kernel keeps (end x, end y, duration, option | outcome)
        # in ev_opt beside the event byte; the ring pass appends every termination to _opt_log ([capacity][8], the
        # records of include/scg_b200.h) and counts them in _opt_log_count
        if int(cfg.option_log) < 0:
            raise ValueError("option_log must be >= 0")
        if cfg.option_log:
            self.ev_opt = torch.zeros((self.ev_cap, max(B, 1), 4), **f32)
            self._opt_log = torch.zeros((int(cfg.option_log), 8), **i32)
            self._opt_log_count = torch.zeros(1, dtype=torch.int64, device=dev)
        else:
            self.ev_opt = self._opt_log = self._opt_log_count = None
        # trajectory log (optional): scg_agent_traj gathers the tracked envs' step records and event bytes of the open
        # window into _traj_log ([capacity][8], the records of include/scg_b200.h) at every flush and every read
        envs = sorted(int(b) for b in cfg.trajectory_envs)
        if int(cfg.trajectory_log) < 0:
            raise ValueError("trajectory_log must be >= 0")
        if bool(envs) != bool(cfg.trajectory_log):
            raise ValueError("trajectory_envs and trajectory_log are set together (both or neither)")
        if len(set(envs)) != len(envs):
            raise ValueError("trajectory_envs has duplicates")
        if envs and not (0 <= envs[0] and envs[-1] < B):
            raise ValueError(f"trajectory_envs must lie in [0, {B})")
        if envs:
            self._traj_env = torch.tensor(envs, **i32)
            self._traj_log = torch.zeros((int(cfg.trajectory_log), 8), **i32)
            self._traj_log_count = torch.zeros(1, dtype=torch.int64, device=dev)
        else:
            self._traj_env = self._traj_log = self._traj_log_count = None
        # occupancy grid (optional): scg_agent_occupancy adds every env-step of the open window to _occ ([K][G][G]
        # uint64 counts held as int64, indexed [option, iy, ix]) at every flush and every read
        G = occupancy_grid_size(cfg.occupancy_grid)
        self._occ = torch.zeros((K, G, G), dtype=torch.int64, device=dev) if G else None
        # initial state, option and action (oracle/agent.py __init__)
        s = self._sbuf[0]
        if initial_states is not None:
            st = torch.as_tensor(np.asarray(initial_states, dtype=np.float32)).to(dev).reshape(B, 4)
            s.copy_(st.t())
        else:
            check(self.lib.scg_reset(self.map.handle, B, None, ptr(s[0]), ptr(s[1]), ptr(s[2]), ptr(s[3]), cfg.seed, 0,
                                     cfg.env_offset, _lib.current_stream()))
        self.start_xy.copy_(s[:2].t())
        self.start_vxy.copy_(s[2:].t())
        self.options.pack()
        self.action.copy_(self.options.act(None, self.option, step=0xFFFFFFFF, stream=_lib.STREAM_RESELECT, soa=s))
        self._struct = self._make_struct()
        self._push_ctl()
        self.options._on_weights_changed = self._weights_changed
        self._xchg = None
        if world_size(self.pg) > 1 and cfg.sync_backend == "p2p":
            # every rank must end up on the same backend: agree on whether the peer mapping worked everywhere
            try:
                x, err = self._connect_peers(), None
            except Exception as e:          # e.g. CUDA IPC unavailable between these devices
                x, err = None, e
            ok = torch.tensor([1 if x is not None else 0], dtype=torch.int32, device=dev)
            ok = int(allreduce_scalar_sum(ok, self.pg))
            if ok == world_size(self.pg):
                self._xchg = x
                check(self.lib.scg_xchg_set_timeout(x, float(cfg.sync_timeout_s)))
            else:
                if x is not None:
                    self.lib.scg_xchg_destroy(x)
                import sys
                print(f"[scg] peer-memory sync unavailable on {world_size(self.pg) - ok} rank(s) ({err}); "
                      "using the NCCL all-reduce path", file=sys.stderr)

    def _connect_peers(self):
        """Create this rank's exchange buffer and map every peer's through CUDA IPC (handles travel over
        torch.distributed once).  The handle exchange is collective, so a rank that failed locally still takes part
        and every rank then sees the failure."""
        dist = self.torch.distributed
        rank, world = dist.get_rank(self.pg), dist.get_world_size(self.pg)
        x, mine, err = C.c_void_p(), None, None
        try:
            check(self.lib.scg_xchg_create(self.options.ctx, rank, world, C.byref(x)))
            buf = (C.c_ubyte * self.lib.scg_xchg_handle_bytes())()
            check(self.lib.scg_xchg_handle(x, buf))
            mine = bytes(buf)
        except Exception as e:
            err = e
        handles = [None] * world
        dist.all_gather_object(handles, mine, group=self.pg)
        try:
            if err is not None or any(h is None for h in handles):
                raise err or _lib.ScgError("a peer could not export its exchange buffer")
            check(self.lib.scg_xchg_connect(x, C.c_char_p(b"".join(handles))))
        except Exception:
            if x:
                self.lib.scg_xchg_destroy(x)
            raise
        return x

    def __del__(self):
        try:
            if getattr(self, "_xchg", None):
                self.lib.scg_xchg_destroy(self._xchg)
                self._xchg = None
        except Exception:
            pass

    # -- controller state --------------------------------------------------------------------------
    def _push_ctl(self):
        """Host copy of the controller state -> device block and host mirror (setup, tests, checkpoints)."""
        g = self._struct
        check(self.lib.scg_agent_set_ctl(self.options.ctx, C.byref(g), C.byref(self._ctl), _lib.current_stream()))

    _push_parents = _push_ctl

    def _poll(self):
        """Pick up promotions the device has made since the last look (host-mapped mirror, no device sync)."""
        m = CtlStruct()
        check(self.lib.scg_agent_poll(self.options.ctx, C.byref(m)))
        if m.n_promotions > self._ctl.n_promotions or m.manage_calls > self._ctl.manage_calls:
            C.memmove(C.byref(self._ctl), C.byref(m), C.sizeof(CtlStruct))
            self._struct.n_active = max(int(self._struct.n_active), int(m.n_active))

    @property
    def n_active(self):
        """Number of active options as far as the host knows (exact after controller_state(sync=True))."""
        self._poll()
        return int(self._ctl.n_active)

    @n_active.setter
    def n_active(self, v):
        self.controller_state(sync=True)       # start from the device's current state, then override
        self._ctl.n_active = int(v)
        self._push_ctl()

    @property
    def active_mask(self):
        self._poll()
        return int(self._ctl.active_mask)

    @active_mask.setter
    def active_mask(self, v):
        self.controller_state(sync=True)
        self._ctl.active_mask = int(v)
        self._push_ctl()

    def controller_state(self, sync=True):
        """dict(n_active, active_mask, n_promotions, last_promotion_step, parents); sync=True waits for the stream so
        the values are exact, sync=False returns what the mirror shows now."""
        if sync:
            self.torch.cuda.current_stream().synchronize()
        self._poll()
        c = self._ctl
        return dict(n_active=int(c.n_active), active_mask=int(c.active_mask), n_promotions=int(c.n_promotions),
                    last_promotion_step=int(c.last_promotion_step), parents=[int(v) for v in c.parents[:self.options.K]])

    # example rings: the step kernel leaves termination events with the step records; they reach the rings at the next
    # flush / manage, or here when somebody looks
    def _ring(self):
        check(self.lib.scg_agent_ring(self.options.ctx, C.byref(self._struct), _lib.current_stream()))

    @property
    def ex_xy(self):
        self._ring()
        return self._ex_xy

    @property
    def ex_label(self):
        self._ring()
        return self._ex_label

    @property
    def ex_count(self):
        self._ring()
        return self._ex_count

    # -- episode log ------------------------------------------------------------------------------
    def episodes(self, since=0, gather=False):
        """The finished episodes logged on the device (AgentConfig.episode_log > 0), brought up to date first (ring pass).
        Returns a dict of NumPy arrays in (step, env) order - step (uint32: the agent step at which the episode ended),
        env (uint32: global env id), ret (float32: task return), length (int32: steps), goal (bool: reached the goal,
        else timed out) - for the records with index >= `since` that are still in the ring, and `total`, the number of
        episodes ever logged.  Polling with since = the previous call's total returns each episode once; when more than
        the capacity arrived in between, the oldest are gone (total - since - len(step) of them).
        gather=True (several ranks): every rank's records, all-gathered over the process group and merged by (step, env);
        `since` is then one value per rank (or one for all), `total` the sum and `totals` the per-rank counts."""
        if not self.cfg.episode_log:
            raise _lib.ScgError("the episode log is off: build the agent with AgentConfig(episode_log=capacity)")
        return self._read_log(self._ep_log, self._ep_log_count, decode_episode_records, since, gather)

    def option_executions(self, since=0, gather=False):
        """The option executions logged on the device (AgentConfig.option_log > 0), brought up to date first (ring pass):
        one record per option termination.  Returns a dict of NumPy arrays in (step, env) order - step (uint32: the agent
        step at which the option terminated), env (uint32: global env id), option (int32), duration (int32: steps the
        execution ran), the outcome flags (bool; every one that holds is set) hit (reached one of its targets), label
        (the example label: hit within init_horizon steps), env_done (the episode ended at the goal), option_timeout,
        left (an active option whose initiation set does not hold at the state reached), episode_timeout, and start,
        end (float32 (n, 2): where the execution began and the state it reached, before any env reset) - plus `total`.
        `since` and `gather` work as for episodes()."""
        if not self.cfg.option_log:
            raise _lib.ScgError("the option log is off: build the agent with AgentConfig(option_log=capacity)")
        return self._read_log(self._opt_log, self._opt_log_count, decode_option_records, since, gather)

    def trajectories(self, since=0, gather=False):
        """The steps of the tracked envs logged on the device (AgentConfig.trajectory_envs / trajectory_log), brought up
        to date first (scg_agent_traj gathers the open window's steps without flushing it, so reading does not change
        what the agent learns): one record per (step, tracked env).  Returns a dict of NumPy arrays in (step, env) order -
        step (uint32: agent step t; the record is the state at which step t began and what happened in it), env (uint32:
        global env id), state (float32 (n, 4): s_t, bit-identical to the agent's state), action, option (int32: what
        was taken at s_t), delta (float32: the step's TD error), term (the option terminated at this step), label (the
        example label: hit within init_horizon steps), episode_end, goal (the episode ended here, at the goal) (bool) -
        plus `total`.  `since` and `gather` work as for episodes()."""
        if self._traj_log is None:
            raise _lib.ScgError("the trajectory log is off: build the agent with AgentConfig(trajectory_envs=..., "
                                "trajectory_log=capacity)")
        check(self.lib.scg_agent_traj(self.options.ctx, C.byref(self._struct), _lib.current_stream()))
        return self._read_log(self._traj_log, self._traj_log_count, decode_trajectory_records, since, gather)

    def occupancy(self, gather=False):
        """The occupancy grid (AgentConfig.occupancy_grid = G), brought up to date first (scg_agent_occupancy counts the
        open window's steps without flushing it, so reading does not change what the agent learns).  Every env-step
        since the agent was built adds 1 to the cell of the option running during it and of the state at which it began:
        cell i = min(max(int(x * G), 0), G - 1) along x, likewise along y.  Returns dict(counts=uint64 (K, G, G) indexed
        [option, iy, ix], grid=G, env_steps=counts.sum()).  Counts are cumulative: subtract two reads for an interval.
        gather=True (several ranks): the counts summed over the process group, plus per_rank, each rank's env_steps."""
        if self._occ is None:
            raise _lib.ScgError("the occupancy grid is off: build the agent with AgentConfig(occupancy_grid=G)")
        check(self.lib.scg_agent_occupancy(self.options.ctx, C.byref(self._struct), _lib.current_stream()))
        counts = self._occ.cpu().numpy().view(np.uint64)
        out = dict(counts=counts, grid=int(counts.shape[1]), env_steps=int(counts.sum()))
        if not gather:
            return out
        parts = [out]
        if world_size(self.pg) > 1:
            parts = [None] * world_size(self.pg)
            self.torch.distributed.all_gather_object(parts, out, group=self.pg)
        return merge_occupancy(parts)

    def _read_log(self, ring, count, decode, since, gather):
        """Records with index >= since still in a device log ring (record i at row i % capacity), decoded, plus `total`;
        with gather=True across a process group, every rank's merged by (step, env)."""
        torch = self.torch
        multi = gather and world_size(self.pg) > 1
        if multi:
            since = since[torch.distributed.get_rank(self.pg)] if np.ndim(since) else since
        self._ring()
        total = int(count.item())
        cap = ring.shape[0]
        lo = max(int(since), total - cap, 0)
        n = max(total - lo, 0)
        s0 = lo % cap
        if s0 + n <= cap:
            rows = ring[s0:s0 + n]
        else:                               # the range wraps around the end of the ring
            rows = torch.cat([ring[s0:], ring[:s0 + n - cap]])
        out = decode(rows.cpu().numpy())
        out["total"] = total
        if not multi:
            return out
        parts = [None] * world_size(self.pg)
        torch.distributed.all_gather_object(parts, out, group=self.pg)
        return merge_episodes(parts)

    # -- plumbing --------------------------------------------------------------------------------

    def _make_struct(self):
        cfg, o, g = self.cfg, self.options, AgentStruct()
        g.B, g.K, g.order = cfg.batch, o.K, o.order
        g.env_offset, g.example_capacity, g.seed = cfg.env_offset, cfg.example_capacity, cfg.seed
        g.gamma, g.lam, g.epsilon, g.option_bonus = cfg.gamma, cfg.lam, cfg.epsilon, cfg.option_bonus
        g.option_timeout, g.max_episode_steps, g.cull = cfg.option_timeout, cfg.max_episode_steps, int(cfg.cull)
        g.alpha, g.win_cap = cfg.alpha, self.win_cap
        g.step = g.window_steps = g.win_len = g.carry_valid = g.ring_len = g.ev_len = g.n_active = 0
        g.ev_cap = self.ev_cap
        g.graph, g.gestation_successes = int(bool(cfg.graph)), int(cfg.gestation_successes)
        g.clf_steps, g.clf_lr = int(cfg.clf_steps), float(cfg.clf_lr)
        g.top_slots, g.alpha_top, g.epsilon_top = self.top_slots, float(cfg.alpha_top), float(cfg.epsilon_top)
        g.init_horizon = int(min(cfg.init_horizon, 1 << 30))
        g.merge_overlap = float(cfg.merge_overlap)
        g.goal_x, g.goal_y = float(self.map.target[0]), float(self.map.target[1])
        s, s2 = self._sbuf
        g.x, g.y, g.vx, g.vy = (s[i].data_ptr() for i in range(4))
        g.x2, g.y2, g.vx2, g.vy2 = (s2[i].data_ptr() for i in range(4))
        for name in ("action", "option", "t_opt", "ep_steps", "start_xy", "ep_return", "reward", "flags", "delta",
                     "q_carry", "win_rec", "ev_hist", "ev_pos", "ctl", "n_success", "n_fail", "n_success_global", "stats",
                     "ep_count", "last_return", "start_vxy", "opt_ret", "opt_disc"):
            setattr(g, name, getattr(self, name).data_ptr())
        g.ex_xy, g.ex_label, g.ex_count = self._ex_xy.data_ptr(), self._ex_label.data_ptr(), self._ex_count.data_ptr()
        g.win_top = self.win_top.data_ptr() if cfg.top_level else None
        if cfg.episode_log:
            g.episode_capacity = int(cfg.episode_log)
            g.ev_ep, g.ep_log, g.ep_log_count = self.ev_ep.data_ptr(), self._ep_log.data_ptr(), self._ep_log_count.data_ptr()
        if cfg.option_log:
            g.option_capacity = int(cfg.option_log)
            g.ev_opt, g.opt_log, g.opt_log_count = (self.ev_opt.data_ptr(), self._opt_log.data_ptr(),
                                                    self._opt_log_count.data_ptr())
        if self._traj_log is not None:
            g.traj_n, g.traj_capacity = len(self._traj_env), int(cfg.trajectory_log)
            g.traj_env, g.traj_log, g.traj_log_count = (self._traj_env.data_ptr(), self._traj_log.data_ptr(),
                                                        self._traj_log_count.data_ptr())
        if self._occ is not None:
            g.occ_grid, g.occ_counts = int(self._occ.shape[1]), self._occ.data_ptr()
        g.trace, g.W, g.Wt, g.theta = o._trace.data_ptr(), o.W.data_ptr(), o.Wt.data_ptr(), o.theta.data_ptr()
        g.dW, g.cnt = o._dW.data_ptr(), o._cnt.data_ptr()
        return g

    def _sync_struct(self):
        g = self._struct
        if self._xchg is not None and self.peer_sync_timed_out():
            raise _lib.ScgError("a peer rank did not arrive at a cross-GPU weight exchange within "
                                f"{self.cfg.sync_timeout_s} s: the weight replicas are out of step")
        return g

    @property
    def t(self):
        return int(self._struct.step)

    @property
    def s(self):
        """(4, B) SoA tensor holding the current state."""
        a, b = self._sbuf
        return a if self._struct.x == a[0].data_ptr() else b

    @property
    def state(self):
        """(B, 4) copy of the current state."""
        return self.s.t().contiguous()

    def _weights_changed(self, applied=False):
        """Hook called by the OptionSet when its weights change (set_weights, apply)."""
        self._struct.carry_valid = 0
        if applied:
            self._struct.window_steps = 0

    def invalidate(self):
        """Call after changing state, action, option or weights from outside: the carried Q_o(s, a)
        is stale and the next step re-evaluates it."""
        self._struct.carry_valid = 0

    # -- the hot path ----------------------------------------------------------------------------
    def step(self):
        """One lock-step agent step for the whole batch (oracle/agent.py SkillChainAgent.step)."""
        self.run(1)

    def run(self, n_steps):
        """`n_steps` lock-step agent steps, with the weight sync every `sync_interval` steps.  The whole loop
        runs inside the library (scg_agent_run): on one rank the sync is the apply kernel, across ranks the
        peer-memory exchange kernel.  With sync_backend="nccl" it returns to Python at every sync for the
        NCCL all-reduce."""
        g = self._sync_struct()
        st = _lib.current_stream()
        n, T = int(n_steps), int(self.cfg.sync_interval)
        if world_size(self.pg) == 1 or self._xchg is not None:
            check(self.lib.scg_agent_run(self.map.handle, self.options.ctx, C.byref(g), n, T, self._xchg, st))
            self.options.window_steps = int(g.window_steps)
            return
        while n > 0:
            k = min(n, T - int(g.window_steps))
            check(self.lib.scg_agent_run(self.map.handle, self.options.ctx, C.byref(g), k, 0, None, st))
            n -= k
            if int(g.window_steps) >= T:
                self.sync()

    def flush(self):
        """Fold the open window's step records into dW and the traces (scg_agent_flush)."""
        g = self._struct
        if int(g.win_len) > 0:
            check(self.lib.scg_agent_flush(self.options.ctx, C.byref(g), _lib.current_stream()))

    def step_host(self, state, action):
        """The same step for a caller that keeps state and actions in host memory (as a user of the
        oracle's NumPy agent does): `state` float32 (4, B) SoA and `action` int32 (B,) are copied
        host->device, the fused step runs, and (next_state (4, B), reward, flags, next_action,
        td_error) come back as views of pinned host buffers that the next call overwrites.  Traces
        and weights stay on the device."""
        torch = self.torch
        B = self.cfg.batch
        if getattr(self, "_host", None) is None:
            pin = lambda shape, dt: torch.empty(shape, dtype=dt).pin_memory()
            def mk():
                out = pin((4, B), torch.float32)      # reward, flags, next action, TD error rows, back to back
                return dict(s=pin((4, B), torch.float32), a=pin((B,), torch.int32), s2=pin((4, B), torch.float32),
                            r=out[0], f=out[1].view(torch.int32), a2=out[2].view(torch.int32), d=out[3])
            self._host = [mk(), mk()]                       # ping-pong: results of call i are inputs of call i+1
            self._host_np = [{k: v.numpy() for k, v in h.items()} for h in self._host]
            self._host_i = 0
        prev, prev_np = self._host[self._host_i], self._host_np[self._host_i]
        cur, cur_np = self._host[1 - self._host_i], self._host_np[1 - self._host_i]
        if state is prev_np["s2"]:
            src_s = prev["s2"]                              # previous result fed straight back: already pinned
        else:
            cur_np["s"][...] = state
            src_s = cur["s"]
        if action is prev_np["a2"]:
            src_a = prev["a2"]
        else:
            cur_np["a"][...] = action
            src_a = cur["a"]
        g = self._sync_struct()
        check(self.lib.scg_agent_step_host(self.map.handle, self.options.ctx, C.byref(g), ptr(src_s), ptr(src_a),
                                           ptr(cur["s2"]), ptr(cur["r"]), ptr(cur["f"]), ptr(cur["a2"]), ptr(cur["d"]),
                                           _lib.current_stream()))
        self._host_i = 1 - self._host_i
        self.options.window_steps = int(g.window_steps)
        if int(g.window_steps) >= self.cfg.sync_interval:
            self.sync()
        return cur_np["s2"], cur_np["r"], cur_np["f"], cur_np["a2"], cur_np["d"]

    def run_host(self, state, action, n_steps):
        """`n_steps` steps for a caller that only needs the state every `n_steps` steps: `state` (4, B) and `action`
        (B,) go host->device once, the steps run device-resident (with the syncs that fall due), and (state, action,
        last reward, last flags, last td_error) come back once, as views of pinned host buffers that the next call
        overwrites (feeding them straight back skips the host-side copy)."""
        torch = self.torch
        B = self.cfg.batch
        if getattr(self, "_hostw", None) is None:
            pin = lambda shape, dt: torch.empty(shape, dtype=dt).pin_memory()
            h = dict(s=pin((4, B), torch.float32), a=pin((B,), torch.int32), s2=pin((4, B), torch.float32),
                     out=pin((4, B), torch.float32))
            h["a2"] = h["out"][2].view(torch.int32)
            self._hostw = h
            self._hostw_np = dict(s=h["s"].numpy(), a=h["a"].numpy(), s2=h["s2"].numpy(), a2=h["a2"].numpy(),
                                  r=h["out"][0].numpy(), f=h["out"][1].view(torch.int32).numpy(), d=h["out"][3].numpy())
        h, hn = self._hostw, self._hostw_np
        if state is hn["s2"]:
            src_s = h["s2"]
        else:
            hn["s"][...] = state
            src_s = h["s"]
        if action is hn["a2"]:
            src_a = h["a2"]
        else:
            hn["a"][...] = action
            src_a = h["a"]
        if world_size(self.pg) == 1 or self._xchg is not None:
            # the whole call stays inside the library: copies in, n_steps steps with their syncs, copies out
            g = self._sync_struct()
            out = h["out"]
            check(self.lib.scg_agent_run_host(self.map.handle, self.options.ctx, C.byref(g), ptr(src_s), ptr(src_a),
                                              int(n_steps), int(self.cfg.sync_interval), self._xchg, ptr(h["s2"]),
                                              ptr(out[0]), ptr(out[1]), ptr(out[2]), ptr(out[3]), _lib.current_stream()))
            self.options.window_steps = int(g.window_steps)
        else:
            self.s.copy_(src_s, non_blocking=True)
            self.action.copy_(src_a, non_blocking=True)
            self.invalidate()
            self.run(n_steps)
            h["s2"].copy_(self.s, non_blocking=True)
            h["out"].copy_(self._out, non_blocking=True)
            torch.cuda.current_stream().synchronize()
        return hn["s2"], hn["a2"], hn["r"], hn["f"], hn["d"]

    HOST_H2D_BYTES_PER_ENV = 20      # state 16 + action 4
    HOST_D2H_BYTES_PER_ENV = 32      # next state 16 + reward 4 + flags 4 + next action 4 + TD error 4

    PROF_KINDS = 6

    def profile_begin(self, max_events, kinds=(0, 1, 2, 3, 4, 5)):
        """Record CUDA events around the launches of the given kinds (0 step, 1 window sweep, 2 reduce, 3 apply /
        exchange, 4 example-ring pass, 5 controller kernel)."""
        check(self.lib.scg_profile_begin(self.options.ctx, int(max_events), sum(1 << k for k in kinds)))

    def profile_end(self):
        """-> (ms per kind, launches per kind) for [fused step, window sweep, dW reduction, apply, ring pass, controller]."""
        ms = (C.c_float * self.PROF_KINDS)()
        n = (C.c_int * self.PROF_KINDS)()
        check(self.lib.scg_profile_end(self.options.ctx, ms, n))
        return [float(v) for v in ms], [int(v) for v in n]

    def sync(self):
        """Flush the window, sum its dW / cnt over ranks (if any) and apply: one library call (scg_agent_sync) on one
        rank or over peer memory; with the NCCL backend the all-reduce runs between the flush and the apply."""
        o, g = self.options, self._struct
        if world_size(self.pg) == 1 or self._xchg is not None:
            check(self.lib.scg_agent_sync(o.ctx, C.byref(g), self._xchg, _lib.current_stream()))
            o.window_steps = 0
            return
        self.flush()
        allreduce_deltas(o._dW, o._cnt, self.pg)
        o.window_steps = int(g.window_steps)
        o.apply()

    def peer_sync_timed_out(self):
        """True if a peer failed to show up at some sync (the exchange kernel gives up after ~2 s)."""
        if self._xchg is None:
            return False
        v = C.c_int()
        check(self.lib.scg_xchg_status(self._xchg, C.byref(v)))
        return bool(v.value)

    # -- low-rate controller ---------------------------------------------------------------------
    def examples(self, k):
        n = int(min(int(self.ex_count[k]), self.cfg.example_capacity))
        return self._ex_xy[k, :n].clone(), self._ex_label[k, :n].clone()

    def manage(self, wait=False):
        """The option-creation controller (oracle/agent.py manage): promote the gestating option once it has enough
        successes.  Queues ONE kernel on the stream (scg_agent_manage): decision, classifier fit and promotion all happen
        in device memory, so the agent loop never waits for the host.  Multi-GPU: success counts are the sums the last
        weight exchange left on every rank (same decision everywhere), and the classifier is fit on the union of the
        ranks' example rings - per-step gradient sums travel over NVLink peer memory and are added in rank order, so
        theta is bit-identical on every rank and equal to one fit on the concatenated examples.  Call it right after a
        sync (manage_every a multiple of sync_interval) for the counts to be current.
        Returns True if the host has learned of a new promotion since the last call: exact with wait=True (waits for
        the stream), otherwise possibly one call late."""
        before = int(self._ctl.n_promotions)
        if world_size(self.pg) > 1 and self._xchg is None:
            self._manage_host()                    # NCCL backend: host-driven, same union fit through all-reduces
        else:
            g = self._sync_struct()
            check(self.lib.scg_agent_manage(self.options.ctx, C.byref(g), self._xchg, _lib.current_stream()))
        if wait:
            self.torch.cuda.current_stream().synchronize()
        self._poll()
        return int(self._ctl.n_promotions) > before

    def _manage_host(self):
        """manage() for the NCCL backend (no peer mapping): the counters and the per-step gradient sums of the fit go
        through all-reduces; every rank ends with the same theta, equal to one fit on the union of the rings."""
        cfg, K, torch = self.cfg, self.options.K, self.torch
        self._poll()
        g = int(self._ctl.n_active)
        if g >= K - 1:
            return
        # the device counter is 32 bits and wraps: read it as unsigned, sum over ranks in 64 bits
        n_succ = int(allreduce_scalar_sum(self.n_success[g:g + 1].to(torch.int64) & 0xFFFFFFFF, self.pg))
        if n_succ < cfg.gestation_successes:
            return
        X, y = self.examples(g)
        o = self.options

        def grad_sum(theta):                      # this rank's sum_i (p_i - y_i) psi_i
            if X.shape[0] == 0:
                return torch.zeros(6, dtype=torch.float32, device=self.device)
            o.theta[g].copy_(theta)
            return o.clf_grad(g, X, y) * float(X.shape[0])

        theta = fit_union(grad_sum, int(X.shape[0]), torch.zeros(6, dtype=torch.float32, device=self.device),
                          cfg.clf_steps, cfg.clf_lr, self.pg)
        o.theta[g].copy_(theta)
        n = g + 1
        self._ctl.active_mask |= (1 << g)
        self._ctl.n_active = n
        self._ctl.n_promotions += 1
        self._ctl.last_promotion_step = int(self._struct.step)
        if cfg.graph and cfg.merge_overlap > 0.0:
            raise _lib.ScgError("merge detection (merge_overlap > 0) needs the device controller (sync_backend='p2p')")
        self.parents_host[n] = (((1 << n) - 1) | GOAL_BIT) if cfg.graph else (1 << (n - 1))
        self._push_ctl()

    def warm_up_controller(self):
        """Run the controller's code path once without effect (first launches load the kernels lazily; with the NCCL
        backend the first collective sets up its communicator): a later promotion then costs what it costs in steady
        state.  Restores everything it touched."""
        torch = self.torch
        if world_size(self.pg) > 1 and self._xchg is None:
            _ = int(allreduce_scalar_sum(self.n_success[0:1].to(torch.int64) & 0xFFFFFFFF, self.pg))
            _ = fit_union(lambda th: th * 0, 0, torch.zeros(6, dtype=torch.float32, device=self.device), 1, 1.0, self.pg)
        else:
            thr, self._struct.gestation_successes = self._struct.gestation_successes, 0x7FFFFFFF   # never promotes
            check(self.lib.scg_agent_manage(self.options.ctx, C.byref(self._struct), self._xchg, _lib.current_stream()))
            self._struct.gestation_successes = thr
        torch.cuda.synchronize()

    # -- checkpoint / resume (SURVEY.md section 5) ----------------------------------------------------
    _CKPT_TENSORS = ("action", "option", "t_opt", "ep_steps", "start_xy", "ep_return", "_ex_xy", "_ex_label", "_ex_count",
                     "n_success", "n_fail", "n_success_global", "stats", "q_carry", "ep_count", "last_return", "start_vxy",
                     "opt_ret", "opt_disc")

    def _logs(self):
        """(checkpoint name, ring, count) of each device log that is on."""
        return [(name, ring, count) for name, ring, count in (("ep_log", self._ep_log, self._ep_log_count),
                                                              ("opt_log", self._opt_log, self._opt_log_count),
                                                              ("traj_log", self._traj_log, self._traj_log_count))
                if ring is not None]

    def save(self, path):
        """Write everything needed to resume this rank (option weights, classifiers, option graph, per-env state and
        traces, counters) to `path` (.npz).  The open window is folded in first."""
        self.flush()
        self._ring()
        o, g = self.options, self._struct
        c = self.controller_state(sync=True)
        arrs = {k.lstrip("_"): getattr(self, k).cpu().numpy() for k in self._CKPT_TENSORS}
        for name, ring, count in self._logs():
            arrs.update({name: ring.cpu().numpy(), name + "_count": count.cpu().numpy()})
        if self._occ is not None:
            arrs["occ_counts"] = self._occ.cpu().numpy()
        arrs.update(W=o.W.cpu().numpy(), theta=o.theta.cpu().numpy(), trace=o._trace.cpu().numpy(),
                    dW=o._dW.cpu().numpy(), cnt=o._cnt.cpu().numpy(), state=self.s.cpu().numpy(),
                    parents=np.array(c["parents"], dtype=np.uint32),
                    meta=np.array([c["n_active"], c["active_mask"], int(g.step), int(g.window_steps), c["n_promotions"],
                                   c["last_promotion_step"]], dtype=np.int64))
        np.savez(path, **arrs)

    def load(self, path):
        """Restore a checkpoint written by save() into an agent built with the same AgentConfig."""
        torch = self.torch
        z = np.load(path)
        o, g = self.options, self._struct
        if tuple(z["W"].shape) != tuple(o.W.shape) or z["state"].shape != tuple(self.s.shape):
            raise ValueError("checkpoint does not match this agent's configuration")
        if self._occ is not None and "occ_counts" in z.files and z["occ_counts"].shape != tuple(self._occ.shape):
            raise ValueError(f"checkpoint occupancy grid {z['occ_counts'].shape} does not match this agent's "
                             f"{tuple(self._occ.shape)}")
        self.flush()
        for k in self._CKPT_TENSORS:
            getattr(self, k).copy_(torch.as_tensor(z[k.lstrip("_")]))
        o.W.copy_(torch.as_tensor(z["W"]))
        o.theta.copy_(torch.as_tensor(z["theta"]))
        o._trace.copy_(torch.as_tensor(z["trace"]))
        o._dW.copy_(torch.as_tensor(z["dW"]))
        o._cnt.copy_(torch.as_tensor(z["cnt"]))
        o.pack()
        self.s.copy_(torch.as_tensor(z["state"]))
        for name, ring, count in self._logs():     # (a checkpoint without a log resumes with an empty one)
            log, total = np.zeros(tuple(ring.shape), dtype=np.int32), 0
            if name in z.files and name + "_count" in z.files:
                old, total = z[name], int(z[name + "_count"][0])
                # the records that fit this agent's ring keep their index i, so they sit at slot i % capacity
                idx = np.arange(max(0, total - min(len(log), len(old))), total, dtype=np.int64)
                log[idx % len(log)] = old[idx % len(old)]
            ring.copy_(torch.as_tensor(log))
            count.fill_(total)
        if self._occ is not None:                  # (a checkpoint without a grid resumes with zeros)
            if "occ_counts" in z.files:
                self._occ.copy_(torch.as_tensor(z["occ_counts"]))
            else:
                self._occ.zero_()
        self.torch.cuda.current_stream().synchronize()
        self._poll()
        self.parents_host[:] = z["parents"]
        self._ctl.n_active, self._ctl.active_mask = int(z["meta"][0]), int(z["meta"][1])
        if len(z["meta"]) > 4:
            self._ctl.n_promotions, self._ctl.last_promotion_step = int(z["meta"][4]), int(z["meta"][5])
        self._push_ctl()
        g.step, g.window_steps, g.win_len, g.ring_len, g.ev_len = int(z["meta"][2]), int(z["meta"][3]), 0, 0, 0
        g.traj_len = g.occ_len = 0
        o.window_steps = int(z["meta"][3])
        g.carry_valid = 0

    def counters(self):
        """Host copy of the global statistics: episodes, goals, mean finished return, per-option counts."""
        st = self.stats.cpu().numpy()
        ep = int(st[0])
        ret = float(st[2:3].view(np.float64)[0])
        return dict(episodes=ep, goals=int(st[1]), mean_return=(ret / ep) if ep else float("nan"),
                    n_success=self.n_success.cpu().numpy().view(np.uint32).astype(np.int64),
                    n_fail=self.n_fail.cpu().numpy().view(np.uint32).astype(np.int64),
                    n_active=self.n_active)

    def run_episode(self, max_steps=2000, manage_every=64, check_every=None):
        """Step until every env has finished at least one more episode, or `max_steps` steps (oracle/agent.py
        run_episode: same stopping rule, same statistics).  The controller runs every `manage_every` steps.  The
        stopping rule is evaluated every `check_every` steps (default: manage_every; the oracle checks after every step,
        so check_every=1 reproduces its step count exactly, at the price of one host read per step)."""
        torch = self.torch
        check_every = int(check_every or manage_every)
        base = self.ep_count.clone()
        goals0 = int(self.stats[1])
        steps = 0
        while steps < max_steps:
            k = min(check_every - steps % check_every, manage_every - steps % manage_every, max_steps - steps)
            self.run(k)
            steps += k
            if steps % manage_every == 0:
                self.manage()
            if steps % check_every == 0 or steps == max_steps:
                done = (self.ep_count > base).all().to(torch.int32)
                if world_size(self.pg) > 1:      # every rank must leave the loop at the same step (the syncs are collective)
                    done = allreduce_scalar_sum(done, self.pg) == world_size(self.pg)
                if bool(done):
                    break
        fin = self.ep_count > base
        n_fin = int(fin.sum())
        mean_ret = float(self.last_return[fin].double().mean()) if n_fin else float("nan")
        return dict(steps=steps, finished=n_fin, goals=int(self.stats[1]), goals_this_call=int(self.stats[1]) - goals0,
                    mean_return=mean_ret, n_active=self.controller_state(sync=True)["n_active"], env_steps=steps * self.cfg.batch)


def decode_episode_records(rec):
    """[n][4] int32 episode-log records (include/scg_b200.h: step, env, return bits, length | goal << 31) -> dict of
    NumPy arrays step, env (uint32), ret (float32), length (int32), goal (bool)."""
    rec = np.ascontiguousarray(rec, dtype=np.int32).reshape(-1, 4)
    u = rec.view(np.uint32)
    return dict(step=u[:, 0].copy(), env=u[:, 1].copy(), ret=rec[:, 2].copy().view(np.float32),
                length=(u[:, 3] & 0x7FFFFFFF).astype(np.int32), goal=(u[:, 3] >> 31).astype(bool))


# option-log outcome bits of record word 2 (include/scg_b200.h), in bit order from 0x100
OPTION_OUTCOMES = ("hit", "label", "env_done", "option_timeout", "left", "episode_timeout")


def decode_option_records(rec):
    """[n][8] int32 option-log records (include/scg_b200.h: step, env, option | outcome bits, duration, start x, y,
    end x, y) -> dict of NumPy arrays step, env (uint32), option, duration (int32), one bool array per outcome
    (OPTION_OUTCOMES), start, end (float32 (n, 2))."""
    rec = np.ascontiguousarray(rec, dtype=np.int32).reshape(-1, 8)
    u = rec.view(np.uint32)
    out = dict(step=u[:, 0].copy(), env=u[:, 1].copy(), option=(u[:, 2] & 0xF).astype(np.int32),
               duration=rec[:, 3].copy())
    for i, k in enumerate(OPTION_OUTCOMES):
        out[k] = ((u[:, 2] >> (8 + i)) & 1).astype(bool)
    out["start"] = rec[:, 4:6].copy().view(np.float32)
    out["end"] = rec[:, 6:8].copy().view(np.float32)
    return out


# trajectory-log flag bits of record word 6 (include/scg_b200.h), in bit order from 0x10000
TRAJECTORY_FLAGS = ("term", "label", "episode_end", "goal")


def decode_trajectory_records(rec):
    """[n][8] int32 trajectory-log records (include/scg_b200.h: step, env, x, y, vx, vy, action | option << 8 | flag
    bits, delta) -> dict of NumPy arrays step, env (uint32), state (float32 (n, 4)), action, option (int32), delta
    (float32), term, label, episode_end, goal (bool)."""
    rec = np.ascontiguousarray(rec, dtype=np.int32).reshape(-1, 8)
    u = rec.view(np.uint32)
    w = u[:, 6]
    out = dict(step=u[:, 0].copy(), env=u[:, 1].copy(), state=rec[:, 2:6].copy().view(np.float32),
               action=(w & 0x7).astype(np.int32), option=((w >> 8) & 0xFF).astype(np.int32),
               delta=rec[:, 7].copy().view(np.float32))
    for i, k in enumerate(TRAJECTORY_FLAGS):
        out[k] = ((w >> (16 + i)) & 1).astype(bool)
    return out


def merge_episodes(parts):
    """Merge the episodes(), option_executions() or trajectories() results of several ranks (a list in rank order) into one in
    (step, env) order; `total` is the sum of their totals and `totals` the list of them."""
    keys = [k for k in parts[0] if k not in ("total", "totals")]
    cat = {k: np.concatenate([p[k] for p in parts]) for k in keys}
    order = np.lexsort((cat["env"], cat["step"]))
    out = {k: v[order] for k, v in cat.items()}
    out["totals"] = [int(p["total"]) for p in parts]
    out["total"] = sum(out["totals"])
    return out


def merge_occupancy(parts):
    """Merge the occupancy() results of several ranks (a list in rank order): the counts summed, env_steps their total
    and per_rank each rank's env_steps."""
    counts = np.sum([p["counts"] for p in parts], axis=0, dtype=np.uint64)
    return dict(counts=counts, grid=int(parts[0]["grid"]), env_steps=int(counts.sum()),
                per_rank=[int(p["env_steps"]) for p in parts])
