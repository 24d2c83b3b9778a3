/* scg_b200.h - C ABI of the B200-native Pinball / skill-chaining hot path.
 *
 * The reference repository (joedownard/skill-chaining-with-graphs) ships no code and therefore
 * no FFI: /root/reference/README.md:1-2 is the whole repository.  The interface each entry point
 * "replaces" is the Python interface of the committed CPU oracle that stands in for the reference
 * (BASELINE.json north_star: "env.reset/step, Option.initiation/act/update,
 * SkillChainAgent.run_episode").  Each declaration cites the oracle function it mirrors.
 *
 * Conventions
 *   - every function returns 0 on success, a cudaError_t value (> 0) on a CUDA failure, or one
 *     of the SCG_E* codes (< 0) on a bad argument; scg_error_string() describes any of them
 *   - the library never allocates or frees caller buffers; all `float*` / `int*` arguments are
 *     DEVICE pointers unless the function name ends in `_host`
 *   - every launch is asynchronous on `stream` (a cudaStream_t passed as void*; NULL = default)
 *   - no function synchronises the device except the `_host` variants, scg_map_create, scg_xchg_create and
 *     the scratch (re)allocations inside the context (first sweep, first apply) and the map (first scg_step_host)
 *   - one host thread drives one context; entry points are re-entrant, not internally locked.  The weight applies on one
 *     context (scg_apply, scg_agent_sync, scg_agent_run) must be stream-ordered: like W and dW, they share the
 *     context's "blocks done" counter
 *   - actions: 0 +x, 1 +y, 2 -x, 3 -y, 4 none;  A = 5;  F = (order+1)^4;  orders 1..5
 *   - state is structure-of-arrays: x[B], y[B], vx[B], vy[B] (fp32)
 */
#ifndef SCG_B200_H
#define SCG_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SCG_N_ACTIONS 5
#define SCG_N_PSI 6
#define SCG_MAX_OPTIONS 16
#define SCG_MAX_ORDER 5
#define SCG_GOAL_BIT 0x80000000u

/* flags word written by the step (oracle/pinball.py pack_flags) */
#define SCG_FLAG_DONE 1
#define SCG_FLAG_KIND_SHIFT 1   /* 0 none, 1 reflection, 2 reversal (last collision of the step) */
#define SCG_FLAG_EDGE_SHIFT 8   /* edge index inside its obstacle, 8 bits */
#define SCG_FLAG_OBST_SHIFT 16  /* obstacle (polygon) index, 12 bits */

/* Philox stream ids: counter = (global env id, step, stream, 0), key = seed */
#define SCG_STREAM_ACTION 0
#define SCG_STREAM_RESET 1
#define SCG_STREAM_RESELECT 2
#define SCG_STREAM_TOP 3

#define SCG_EINVAL (-1)   /* bad argument */
#define SCG_ENOMEM (-2)   /* host allocation failed */
#define SCG_ELIMIT (-3)   /* map / order / K exceeds a compiled-in limit */
#define SCG_EPEER (-4)    /* a peer rank did not arrive at a cross-GPU exchange within the timeout (sticky) */

typedef struct scg_map scg_map_t; /* opaque: edge table + broad-phase grid, host and device copies */
typedef struct scg_ctx scg_ctx_t; /* opaque: device scratch for the Sarsa(lambda) reduction */
typedef struct scg_xchg scg_xchg_t; /* opaque: peer-memory exchange buffers of the cross-GPU sync */

const char *scg_error_string(int code);
int scg_version(void);

/* ---- map ---------------------------------------------------------------------------------
 * mirrors oracle/pinball.py PinballMap.__init__ (edge table) - same fp32 formulas, same order.
 * verts: n_verts x 2 fp32 HOST; poly_start: n_poly+1 HOST offsets into verts; starts: n_starts x 2.
 * grid_n: broad-phase grid resolution (power of two, <= 128; 0 = default 64). */
int scg_map_create(const float *verts, const int *poly_start, int n_poly, float ball_r, float tx,
                   float ty, float tr, const float *starts, int n_starts, int grid_n, scg_map_t **out);
int scg_map_destroy(scg_map_t *map);
int scg_map_num_edges(const scg_map_t *map);
int scg_map_num_candidates(const scg_map_t *map);
int scg_map_edge_table(const scg_map_t *map, float *edges_out /* HOST [E][8] */,
                       int *obstacle_out /* HOST [E] */, int *local_out /* HOST [E] */);
/* broad-phase grid, for tests: cell_start HOST [G*G+1], cand HOST [n_cand] */
int scg_map_grid(const scg_map_t *map, int *grid_n_out, int *cell_start_out, int *cand_out);

/* ---- K1: batched Pinball step -------------------------------------------------------------
 * mirrors oracle/pinball.py step_scalar / PinballEnv.step.  Out arrays may alias the inputs.
 * cull != 0 uses the broad-phase grid (bit-identical results); 0 tests every edge. */
int scg_step(const scg_map_t *map, int B, const float *x, const float *y, const float *vx,
             const float *vy, const int *action, float *x2, float *y2, float *vx2, float *vy2,
             float *reward, int *flags, int cull, void *stream);
/* mirrors PinballEnv.reset(mask, step): masked envs go to a start position with zero velocity */
int scg_reset(const scg_map_t *map, int B, const uint8_t *mask /* may be NULL = all */, float *x,
              float *y, float *vx, float *vy, uint64_t seed, uint32_t step, uint32_t env_offset,
              void *stream);
/* HOST-buffer variant of scg_step (state in, state/reward/flags out; copies included) */
int scg_step_host(scg_map_t *map, int B, float *state_soa /* HOST [4][B] in/out */,
                  const int *action /* HOST */, float *reward /* HOST */, int *flags /* HOST */,
                  void *stream);

/* ---- K2: Fourier features, Q evaluation, action selection, TD error ------------------------
 * mirrors oracle/fourier.py FourierBasis.features, oracle/option.py OptionSet.q / act / td_error.
 * W is [K][A][F]; Wt is the packed copy the kernels read, made by scg_pack_weights (and kept current by scg_apply /
 * scg_xchg_sync / scg_agent_sync): [K][scg_packed_slot_floats(order)] fp32, a slot holding its features in pairs of 12 floats
 * (w0a w1a w2a w3a | w0b w1b w2b w3b | w4a w4b 0 0) - the operands of the two-wide FMAs, 1.5 16-byte loads per
 * feature - padded so that consecutive slots start 16 bytes apart modulo 128 (shared-memory banks). */
int scg_packed_slot_floats(int order);
int scg_features(int order, int B, const float *x, const float *y, const float *vx, const float *vy,
                 float *phi /* [B][F] */, void *stream);
int scg_pack_weights(int order, int K, const float *W, float *Wt, void *stream);
int scg_q_eval(int order, int K, int B, const float *x, const float *y, const float *vx,
               const float *vy, const int *option, const float *Wt, float *Q /* [B][A] */, void *stream);
int scg_select(int B, const float *Q /* [B][A] */, float epsilon, uint64_t seed, uint32_t step,
               uint32_t stream_id, uint32_t env_offset, int *action, void *stream);
int scg_td_error(int order, int K, int B, const float *x, const float *y, const float *vx,
                 const float *vy, const int *a, const float *r, const float *x2, const float *y2,
                 const float *vx2, const float *vy2, const int *a2, const uint8_t *done,
                 const int *option, const float *Wt, float gamma, float *delta, void *stream);

/* ---- K3: Sarsa(lambda) eligibility traces and weight-delta accumulation --------------------
 * mirrors oracle/option.py OptionSet.update (trace part) and OptionSet.apply.
 * trace is [B][A][F]; dW [K][A][F] and cnt [K] accumulate over the sync window. */
int scg_ctx_create(int order, int K, scg_ctx_t **out);
int scg_ctx_destroy(scg_ctx_t *ctx);
/* on != 0: reproducible runs.  The per-CTA dW slabs are summed in a fixed order (no floating-point atomics) and
 * scg_agent_manage waits for its kernel, so that the host sizes the following launches with exact knowledge of the
 * controller state; together with the deterministic example rings (scg_agent_ring) weights, traces, rings and classifiers
 * then reproduce bit for bit for the same inputs.  Not covered: the top-level learner's window update (k_top adds with
 * atomics) and the double-precision sum of finished returns in `stats` (integer-valued rewards: exact in practice).
 * off (default): one atomic per address per slice, ~1 us per step faster at configs[1]. */
int scg_ctx_set_deterministic(scg_ctx_t *ctx, int on);
/* One dense Sarsa(lambda) step over all of the context's K option slots; any K <= SCG_MAX_OPTIONS (16) at every order
 * (at order 5 the slots beyond 8 accumulate in global memory instead of shared memory). */
int scg_sarsa_update(scg_ctx_t *ctx, int B, const float *x, const float *y, const float *vx,
                     const float *vy, const int *a, const int *option, const float *delta,
                     const uint8_t *done, const uint8_t *mask /* may be NULL */, float gamma_lambda,
                     float *trace, float *dW, int *cnt, void *stream);
/* W += alpha * alpha_scale_f * dW * (window_steps / cnt[k]) for every slot k with cnt[k] > 0, Wt refreshed, dW and cnt
 * zeroed, over all of the context's K slots at its order.  Slots K_opt .. K-1 hold the top-level learner
 * (oracle/option.py OptionSet(top_slots=...)): they are stepped with alpha_top and the mean over the window's events
 * (cnt[k] = event count) instead; K_opt == K: no top-level slots. */
int scg_apply(scg_ctx_t *ctx, int K_opt, float *W, float *Wt, float *dW, int *cnt, float alpha, float alpha_top,
              int window_steps, void *stream);

/* ---- K4: initiation classifiers --------------------------------------------------------------
 * mirrors oracle/option.py OptionSet.initiation_prob / clf_grad / fit_initiation. */
int scg_clf_eval(int B, const float *x, const float *y, const float *theta /* [K][6] */, int K,
                 float *p /* [B][K] */, void *stream);
/* mirrors OptionSet.initiation: inside[b][k] = (theta_k . psi(x_b, y_b) >= 0), the logit formed in fp32 with one rounding
 * per operation in the oracle's order (initiation_logit), so the decision is bit-identical to the oracle's */
int scg_clf_decide(int B, const float *x, const float *y, const float *theta /* [K][6] */, int K,
                   uint8_t *inside /* [B][K] */, void *stream);
int scg_clf_grad(int N, const float *X /* [N][2] */, const uint8_t *y, const float *theta_k /* [6] */,
                 float *grad /* [6], overwritten */, void *stream);
int scg_clf_fit(int N, const float *X, const uint8_t *y, float *theta_k /* [6] in/out */, int steps,
                float lr, void *stream);

/* ---- fused agent pipeline, mirrors oracle/agent.py SkillChainAgent.step ------------------------
 * One step = ONE kernel: env step (K1) -> initiation bits of s' (K4) -> termination / option reward ->
 * Q_o(s', .) (K2) -> eps-greedy a' -> TD error -> 32-byte step record -> env reset -> option re-selection.
 * Q_o(s, a) is carried from the previous step (q_carry) while the weights are unchanged.
 * Sarsa(lambda) runs in the windowed (forward-view) form of oracle/option.py OptionSet.flush: the step
 * records of up to win_cap steps are folded into dW and the per-env traces by ONE trace sweep per
 * window (scg_agent_flush), so the dense traces are read and written once per window, not per step. */
#define SCG_WIN_MAX 32

/* Device-resident controller state (oracle/agent.py: n_active, active, parents).  The step kernel reads it every step;
 * scg_agent_manage's kernel promotes the gestating option in place, so option creation needs no host round trip. */
typedef struct scg_ctl {
    int32_t n_active;              /* options 0 .. n_active-1 are active; slot n_active is the gestating learner */
    uint32_t active_mask;          /* bit k set <=> option k is active */
    int32_t n_promotions;          /* promotions decided on the device so far */
    uint32_t last_promotion_step;  /* agent step at which the last one was decided */
    uint32_t manage_calls;         /* scg_agent_manage launches completed */
    uint32_t reserved[3];
    uint32_t parents[SCG_MAX_OPTIONS]; /* bit j: the initiation set of option j is a target of option k; bit 31: the goal */
} scg_ctl_t;

typedef struct scg_agent {
    /* sizes and hyper-parameters */
    int32_t B, K, order;
    int32_t n_active;                /* the caller's LOWER BOUND of ctl->n_active: sizes the on-chip weight staging and the
                                        sweep's accumulator (options 0 .. n_active); options beyond it still work, through
                                        the global-memory paths.  scg_agent_run raises it from the host mirror by itself. */
    uint32_t graph, env_offset, step, example_capacity;
    uint64_t seed;
    float gamma, lambda, epsilon, option_bonus;
    int32_t option_timeout, max_episode_steps, cull, carry_valid;
    float alpha; int32_t window_steps, win_cap, win_len;
    int32_t ev_cap, ev_len, ring_len; /* event history: capacity in steps (>= 2 * win_cap), steps recorded, steps already
                                        appended to the example rings (ring_len <= ev_len; the open window is the last win_len) */
    int32_t gestation_successes, clf_steps; float clf_lr;   /* controller: promotion threshold, classifier fit */
    int32_t top_slots;               /* 0: options are chosen "first active initiation set"; n = ceil(K / 5): by the top-level
                                        SMDP learner whose weights are slots K .. K+n-1 of W / Wt / dW / cnt (K + n <= 16) */
    float alpha_top, epsilon_top;
    int32_t init_horizon;            /* an example is positive iff the option hit a target within this many steps of its start */
    float merge_overlap, goal_x, goal_y;   /* option graph: merge detection threshold (0: every older option and the goal
                                        are targets), the goal position (oracle/agent.py merged_parents) */
    uint32_t episode_capacity;       /* records in the episode log ring (ep_log); 0 with ev_ep = ep_log = NULL: no log */
    /* per-env state (device) */
    float *x, *y, *vx, *vy;          /* current state s */
    float *x2, *y2, *vx2, *vy2;      /* the other state buffer: a step writes s' here, then the two swap */
    int32_t *action, *option, *t_opt, *ep_steps;
    float *start_xy;                 /* [B][2] position where the current option execution began */
    float *start_vxy;                /* [B][2] velocity there; opt_ret [B] discounted task reward since, opt_disc [B] gamma^steps */
    float *opt_ret, *opt_disc;       /*   (top-level learner only; may be NULL when top_slots == 0) */
    float *ep_return;                /* [B] running task return */
    int32_t *ep_count;               /* [B] finished episodes of each env */
    float *last_return;              /* [B] task return of each env's last finished episode */
    float *reward; int32_t *flags;   /* [B] outputs of the env step */
    float *delta;                    /* [B] TD errors of this step */
    float *q_carry;                  /* [B] Q_o(s, a) of the pending (state, action), valid iff carry_valid */
    float *win_rec;                  /* [win_cap][B][8] step records of the open window */
    uint8_t *ev_hist;                /* [ev_cap][B] option-termination events, one byte per env-step (0 = none), kept until the
                                        example-ring pass has consumed them (scg_agent_ring: at manage / when the history is full) */
    float *ev_pos;                   /* [ev_cap][B][2] where the terminated option had started (written where ev_hist says so) */
    float *win_top;                  /* [win_cap][B][8] top-level SMDP updates of the open window, valid where the event byte says
                                        "terminated": s0 (4), delta_top, option bits (top_slots > 0 only) */
    float *trace;                    /* [B][A][F], as of the last flush */
    /* per-option state (device) */
    float *W, *Wt, *theta, *dW;      /* [K][A][F], [K][scg_packed_slot_floats], [K][6], [K][A][F] */
    int32_t *cnt;                    /* [K] */
    scg_ctl_t *ctl;                  /* controller state */
    float *ex_xy; uint8_t *ex_label; /* [K][cap][2], [K][cap] example rings */
    int64_t *ex_count;               /* [K] examples ever appended; slot of the next one = ex_count % cap */
    int32_t *n_success, *n_fail;     /* [K] */
    int32_t *n_success_global;       /* [K] n_success summed over ranks as of the last cross-GPU sync (multi-rank runs) */
    /* global statistics (device), 4 x 64 bit: [0] episodes, [1] goals (uint64), [2] sum of finished returns (double) */
    int64_t *stats;
    /* episode log (optional: all NULL / 0 = off, and the kernels do exactly the work they do without it).  When on, the
     * step kernel marks every episode end in its event byte and keeps (return, length) beside it; the ring pass appends
     * the episode ends to ep_log in (step, env) order:
     *   record i (16 bytes) at slot i % episode_capacity: uint32 step (agent step at which the episode ended),
     *   uint32 env (global env id), float return, int32 length | goal << 31 (goal 0: the episode timed out).
     * The last episode_capacity records survive.  ev_ep and ep_log are both NULL or both set, with episode_capacity > 0
     * and ep_log_count set. */
    float *ev_ep;                    /* [ev_cap][B][2] at an episode end: its return, its length (int32 bits) */
    uint32_t *ep_log;                /* [episode_capacity][4] the records */
    int64_t *ep_log_count;           /* [1] episodes ever logged; the next one goes to slot ep_log_count % episode_capacity */
    /* option log (optional, same rules as the episode log: all NULL / 0 = off, and the kernels do exactly the work they do
     * without it).  When on, the step kernel keeps, beside every termination's event byte, where the execution ended, how
     * long it ran and why it stopped; the ring pass appends every termination to opt_log in (step, env) order:
     *   record i (32 bytes) at slot i % option_capacity: uint32 step (agent step at which the option terminated),
     *   uint32 env (global env id), uint32 option (bits 0-3) | outcome bits, int32 duration (t_opt at termination, >= 1),
     *   float start x, y (where the execution began), float end x, y (the state the step reached, before any env reset).
     *   Outcome bits (oracle/agent.py SkillChainAgent.step items 3 and 6), every one that holds is set:
     *   0x100 hit (reached one of its targets), 0x200 label (the example label: hit and t_opt <= init_horizon),
     *   0x400 env_done (the episode ended at the goal), 0x800 option_timeout (t_opt >= option_timeout),
     *   0x1000 left (an active option whose initiation set does not hold at s'), 0x2000 episode_timeout.
     * The last option_capacity records survive.  ev_opt, opt_log and opt_log_count are all NULL or all set, with
     * option_capacity > 0. */
    uint32_t option_capacity;        /* records in the option log ring (opt_log); 0 with ev_opt = opt_log = NULL: no log */
    float *ev_opt;                   /* [ev_cap][B][4] at a termination: end x, end y, duration (int32 bits), word 2 of the
                                        record (uint32 bits) */
    uint32_t *opt_log;               /* [option_capacity][8] the records */
    int64_t *opt_log_count;          /* [1] executions ever logged; the next one goes to slot opt_log_count % option_capacity */
    /* trajectory log (optional, same rules: all NULL / 0 = off).  When on, every step of traj_n chosen envs is recorded:
     * scg_agent_traj gathers the open window's step records (win_rec) and event bytes of those envs into traj_log, at
     * every flush and whenever the log is read.  The step kernel's only part is to mark episode ends in the event byte
     * (as with the episode log on).  Records in (step, env) order, traj_n per step, tracked envs in ascending order:
     *   record i (32 bytes) at slot i % traj_capacity: uint32 step (agent step t: the record is the state at which step
     *   t began and what happened in it), uint32 env (global env id; 0xFFFFFFFF with a zero payload for a traj_env entry
     *   outside [0, B)), float x, y, vx, vy (s_t, bit-identical to the agent's state), uint32 action (bits 0-2) |
     *   option << 8 | 0x10000 term (the option terminated at this step) | 0x20000 label (the example label: hit and
     *   t_opt <= init_horizon) | 0x40000 episode end | 0x80000 goal (the episode ended at the goal), float delta (this
     *   step's TD error).
     * The last traj_capacity records survive.  traj_env, traj_log and traj_log_count are all NULL with traj_n =
     * traj_capacity = 0, or all set with 1 <= traj_n <= B and traj_capacity > 0. */
    uint32_t traj_n;                 /* tracked envs; 0: no log */
    const int32_t *traj_env;         /* [traj_n] local env indices, ascending and distinct, each < B (device) */
    uint32_t traj_capacity;          /* records in the trajectory log ring (traj_log) */
    uint32_t *traj_log;              /* [traj_capacity][8] the records */
    int64_t *traj_log_count;         /* [1] records ever logged; record i sits at slot i % traj_capacity */
    int32_t traj_len;                /* steps of the open window already gathered (0 .. win_len; host bookkeeping, like
                                        ring_len: scg_agent_traj sets it to win_len, the flush resets it with win_len) */
    /* occupancy grid (optional: occ_grid = 0 and occ_counts = NULL = off, and the kernels do exactly the work they do
     * without it).  When on, every env-step of every env is counted by the option running during it and the map cell
     * of the state at which it began: scg_agent_occupancy adds the open window's step records (win_rec) to occ_counts,
     * at every flush and whenever the grid is read.  The step kernel has no part in it.  Step t of env b adds 1 to
     *   occ_counts[o][iy][ix], o = the record's option (slots 0 .. K-1, the gestating one included; the top-level
     *   learner's weight slots have no cell), ix = min(max((int)(x * occ_grid), 0), occ_grid - 1) with x the fp32 x of
     *   s_t and the conversion truncating toward zero, iy likewise from y.
     * occ_grid is a power of two in 1 .. 128, so x * occ_grid is exact in fp32.  Counts are cumulative (subtract two
     * reads for an interval), and integer adds make them the same whatever the order of the adds.  occ_counts is NULL
     * iff occ_grid == 0. */
    uint32_t occ_grid;               /* cells per side of the unit square; 0: no grid */
    uint64_t *occ_counts;            /* [K][occ_grid][occ_grid] env-steps per (option, cell) (device) */
    int32_t occ_len;                 /* steps of the open window already counted (0 .. win_len; host bookkeeping, like
                                        traj_len: scg_agent_occupancy sets it to win_len, the flush resets it with win_len) */
} scg_agent_t;

/* One lock-step agent step.  Updates the struct: swaps (x..vy) with (x2..vy2) so that x..vy is the new
 * current state, step += 1, window_steps += 1, win_len += 1, carry_valid = 1; flushes the window when
 * win_len reaches win_cap.  Clear carry_valid whenever state, action, option or weights are changed
 * from outside (scg_apply changes the weights: callers clear it after every apply; scg_agent_sync does). */
int scg_agent_step(const scg_map_t *map, scg_ctx_t *ctx, scg_agent_t *ag, void *stream);
/* Fold the open window into dW and the traces (no-op when win_len == 0).  Accepts any K <= SCG_MAX_OPTIONS (16, the
 * top-level slots included) at every order and batch size.  With the trajectory log on it first gathers the window's
 * remaining steps into the log (scg_agent_traj), and with the occupancy grid on counts them (scg_agent_occupancy);
 * win_len, traj_len and occ_len then return to 0. */
int scg_agent_flush(scg_ctx_t *ctx, scg_agent_t *ag, void *stream);
/* Bring the trajectory log up to date: append the records of the tracked envs for the open window's steps
 * [traj_len, win_len) to traj_log (one small kernel on `stream`), advance *traj_log_count by traj_n per step, and set
 * traj_len = win_len.  It does not flush, so calling it between steps leaves every learning result bit for bit as it
 * would be without the call.  No-op with the log off.  Call it before reading the log. */
int scg_agent_traj(scg_ctx_t *ctx, scg_agent_t *ag, void *stream);
/* Bring the occupancy grid up to date: add the open window's steps [occ_len, win_len) of all B envs to occ_counts (one
 * kernel on `stream`: per-CTA shared-memory bins, then integer adds to occ_counts) and set occ_len = win_len.  It does not flush, so calling it
 * between steps leaves every learning result bit for bit as it would be without the call.  No-op with the grid off.
 * Call it before reading the grid. */
int scg_agent_occupancy(scg_ctx_t *ctx, scg_agent_t *ag, void *stream);
/* Append the option-termination examples of the recorded, not yet processed steps to the example rings
 * (oracle/agent.py step, item 6).  The step kernel only leaves an event byte and a start position per termination; the
 * rings are brought up to date here - by scg_agent_manage, when the event history is full, or on request - so the pass
 * runs once per controller interval, not once per window.  Deterministic: the examples of a step are appended in env order, steps in order,
 * exactly the oracle's sequence, whatever the launch geometry; when more than `example_capacity` examples of one option
 * arrive, the last `example_capacity` survive.  Called by flush and manage; call it before reading the rings.
 * With the episode log on it also brings the log up to date: the same pass appends the episode ends of those steps to
 * ep_log, in the same (step, env) order, and advances *ep_log_count.  Call it before reading the log.  The option log
 * likewise: every termination of those steps goes to opt_log in (step, env) order, and *opt_log_count advances. */
int scg_agent_ring(scg_ctx_t *ctx, scg_agent_t *ag, void *stream);
/* The option-creation controller (oracle/agent.py manage) as ONE kernel on `stream`, no host round trip: if the
 * gestating option g = ctl->n_active has at least gestation_successes successes (n_success[g]; across ranks:
 * n_success_global[g] as of the last exchange, identical on every rank), its initiation classifier is fit on its
 * example ring (clf_steps gradient steps from theta = 0; across ranks on the UNION of the ranks' rings: the per-step
 * gradient sums and example counts are exchanged over NVLink peer memory and added in rank order, so theta is
 * bit-identical on every rank and equal to a single fit on the concatenated examples), option g becomes active and
 * slot g + 1 starts gestating with parents {g} (chain) or {0..g, goal} (graph != 0).  The new state is also written to a
 * host-mapped mirror (scg_agent_poll).  xchg: NULL for a single rank.  Every rank must call it at the same steps. */
int scg_agent_manage(scg_ctx_t *ctx, scg_agent_t *ag, scg_xchg_t *xchg, void *stream);
/* Host copy of the controller state as of the last completed scg_agent_manage / scg_agent_set_ctl, without
 * synchronising the device.  The copy is always one consistent state: a read that overlaps a write of the mirror is
 * retried, for up to 1 ms, and then the last consistent copy is returned (the values only ever grow, so a stale copy is
 * a valid lower bound). */
int scg_agent_poll(scg_ctx_t *ctx, scg_ctl_t *out /* HOST */);
/* Overwrite the controller state from the host (tests, checkpoints): device copy on `stream` + the mirror. */
int scg_agent_set_ctl(scg_ctx_t *ctx, scg_agent_t *ag, const scg_ctl_t *in /* HOST */, void *stream);
/* n_steps steps in one call; when sync_interval > 0 also scg_agent_sync every sync_interval steps.  With
 * sync_interval == 0 the caller syncs: scg_agent_sync, or flush, sum dW / cnt over ranks itself and scg_apply. */
int scg_agent_run(const scg_map_t *map, scg_ctx_t *ctx, scg_agent_t *ag, int n_steps, int sync_interval,
                  scg_xchg_t *xchg, void *stream);
/* The weight sync of the agent: flush the open window, then scg_apply for a single rank (xchg == NULL) or scg_xchg_sync
 * across ranks (dW, cnt and the success counters summed over ranks), with the agent's alpha, alpha_top and window_steps
 * (the top-level slots are K .. K+top_slots-1); then window_steps = 0 and carry_valid = 0.  Profiled as kind 3. */
int scg_agent_sync(scg_ctx_t *ctx, scg_agent_t *ag, scg_xchg_t *xchg, void *stream);

/* ---- S5: cross-GPU weight-delta exchange over NVLink peer memory ---------------------------------
 * mirrors the multi-rank half of oracle/option.py OptionSet.apply (sum dW and cnt over ranks, then the
 * same apply on every rank).  One kernel per sync publishes this rank's dW / cnt, signals and waits on
 * per-slice flags in peer memory, sums every rank's slice in rank order and applies - replicas stay
 * bit-identical.  One process per GPU: exchange scg_xchg_handle() blobs (scg_xchg_handle_bytes() each,
 * CUDA IPC) and call scg_xchg_connect with all of them; one process driving several devices:
 * scg_xchg_connect_ptrs with every rank's scg_xchg_local_ptr (peer access enabled by the caller). */
int scg_xchg_create(scg_ctx_t *ctx, int rank, int world, scg_xchg_t **out);
int scg_xchg_destroy(scg_xchg_t *x);
int scg_xchg_handle_bytes(void);
int scg_xchg_handle(scg_xchg_t *x, void *handle_out /* HOST */);
int scg_xchg_connect(scg_xchg_t *x, const void *all_handles /* HOST [world][handle_bytes] */);
int scg_xchg_local_ptr(scg_xchg_t *x, void **ptr_out);
int scg_xchg_connect_ptrs(scg_xchg_t *x, void *const *peer_ptrs /* HOST [world] device pointers */);
/* *timed_out != 0: some exchange gave up waiting for a peer.  The flag is sticky and lives in host-mapped memory (no
 * device synchronisation to read it); from then on scg_xchg_sync, scg_agent_sync and scg_agent_run return SCG_EPEER. */
int scg_xchg_status(scg_xchg_t *x, int *timed_out);
/* how long an exchange waits for its peers before giving up (default 30 s) */
int scg_xchg_set_timeout(scg_xchg_t *x, double seconds);
/* dW (reduced over this rank's envs) and cnt -> summed over ranks -> W, Wt updated as scg_apply does (order and K of
 * the context the handle was created from, top-level slots K_opt .. K-1); dW and cnt zeroed.
 * nsucc_local [K] (optional): this rank's option success counters; nsucc_global [K] (optional) receives their sum
 * over ranks, identical on every rank, so the controller needs no collective of its own.
 * Every rank must call it the same number of times. */
int scg_xchg_sync(scg_xchg_t *x, int K_opt, float *W, float *Wt, float *dW, int *cnt, float alpha, float alpha_top,
                  int window_steps, const int *nsucc_local, int *nsucc_global, void *stream);

/* HOST-buffer variant of scg_agent_step: the call a user makes who keeps state and actions in
 * host (NumPy) arrays, as with the oracle's SkillChainAgent.  Copies state [4][B] and action [B]
 * host->device, runs the fused step, copies next state, reward, flags, next action and TD error
 * device->host and waits for them.  Traces and weights stay resident on the device.  When the SoA blocks are
 * back to back on both sides and B >= 128 the step is pipelined over two halves of the batch (copy in / step / copy out
 * on three streams); results are identical. */
int scg_agent_step_host(const scg_map_t *map, scg_ctx_t *ctx, scg_agent_t *ag,
                        const float *h_state_soa, const int *h_action, float *h_state2_soa,
                        float *h_reward, int *h_flags, int *h_action2, float *h_delta, void *stream);

/* HOST-buffer variant of scg_agent_run for a caller that only needs the state every n_steps steps: state and action go
 * host->device once, the n_steps steps (with the syncs that fall due) run device-resident inside the library, and next
 * state, last reward / flags / TD error and next action come back once; waits for the copies. */
int scg_agent_run_host(const scg_map_t *map, scg_ctx_t *ctx, scg_agent_t *ag, const float *h_state_soa,
                       const int *h_action, int n_steps, int sync_interval, scg_xchg_t *xchg, float *h_state2_soa,
                       float *h_reward, int *h_flags, int *h_action2, float *h_delta, void *stream);

/* Per-kernel device timing of the agent pipeline with CUDA events on the launch stream.
 * scg_profile_begin arms it (up to max_events kernel launches of the kinds in kind_mask are recorded);
 * scg_profile_end waits for the recorded events and returns, per kind, the summed milliseconds and the
 * launch count: kind 0 fused step kernel, 1 window trace sweep, 2 dW reduction, 3 weight apply / exchange
 * (scg_sarsa_update on the same context runs the same sweep and reduction, and is recorded as kinds 1 and 2).
 * (Events around the step kernels - bit 0 - keep consecutive step kernels from overlapping their prologues.) */
#define SCG_PROF_KINDS 6   /* 0 fused step, 1 window sweep, 2 dW reduction, 3 apply / exchange, 4 example-ring pass, 5 controller */
int scg_profile_begin(scg_ctx_t *ctx, int max_events, int kind_mask);
int scg_profile_end(scg_ctx_t *ctx, float *ms /* HOST [SCG_PROF_KINDS] */, int *count /* HOST [SCG_PROF_KINDS] */);

/* kernel launch counter (this library's launches since load), for bench.py's gpu_launches */
uint64_t scg_launch_count(void);

#ifdef __cplusplus
}
#endif
#endif /* SCG_B200_H */
