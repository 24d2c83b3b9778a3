// scg_agent.cu - the fused lock-step agent step (K1 + K2 + K4 in ONE kernel) and the windowed pipeline.
//
// Mirrors oracle/agent.py SkillChainAgent.step, numbered steps 1-8 of its docstring (the reference
// has no code: /root/reference/README.md:1-2).  Per env step, k_agent_step does
//   1    s2, r_env, flags = env.step(a)                                   (pinball_step, scg_step.cuh)
//   2-3  initiation bits of s2 (K4), termination, option reward
//   4    Q_o(s2, .) (K2), eps-greedy a2, TD error; Q_o(s, a) is carried from the previous step
//        (q_carry) and only recomputed (PAIR variant, weight loads shared) after the weights changed
//   5    a 32-byte step record for the window sweep (state, delta, action/option/termination bits)
//   6-8  example-ring append, env reset, option re-selection + first action under the new option
// Sarsa(lambda) itself runs once per window of up to win_cap steps (k_window in scg_sarsa.cu: the
// forward-view form of oracle/option.py OptionSet.flush), so the dense per-env traces cross HBM once
// per window instead of once per step.  Weight application (and the cross-GPU sum of dW / cnt, scg_xchg.cu)
// happens every sync interval.  Because nothing couples the envs while the weights are frozen, ONE launch runs
// all the steps of a window for every env, with the env's state in registers between the steps.
//
// Kernel design: one thread per env, work handed out per warp (32 envs) and interleaved over the
// persistent CTAs so that every SM gets the same number of warps even at B = 65,536.  Each CTA stages
// the map blob and, when they fit, the packed weight slots in use into shared memory with bulk-TMA copies
// (cp.async.bulk + mbarrier); lanes executing different options then read different banks.
#include <stdlib.h>

#include <algorithm>

#include "scg_common.cuh"
#include "scg_step.cuh"

int scg_launch_window(scg_ctx *ctx, int B, int T, int k_used, const float *rec, float *trace, float gl, float *dW,
                      cudaStream_t st);
int scg_reduce_window(scg_ctx *ctx, int n_slabs, int k_used, float *dW, cudaStream_t st);
int scg_prof_push(scg_ctx *ctx, int kind, cudaStream_t st, bool end);
int scg_launch_top(scg_ctx *ctx, const scg_agent_t *ag, cudaStream_t st);

struct StepArgs {
    scg_agent_t ag;
    const unsigned char *map_blob;
    int blob_bytes, w_bytes;
    int k_stage;      // options whose weights are staged to shared memory (ids 0 .. k_stage-1 are the ones in use)
    int wait_first;   // 1: the previous launch may have written the weights - wait for it before staging them
    int n_steps;      // consecutive steps run by this launch (records go to consecutive slabs of the window)
    int b_begin, b_end;   // envs [b_begin, b_end) are stepped by this launch (b_begin a multiple of 32; normally 0, B)
    float4 *rec;  // this step's slab of the window: [B][2]
    uint8_t *ev;  // this step's slab of the event bytes: [B]
    float2 *pos;  // this step's slab of option start positions: [B]
    float *top;   // this step's slab of the top-level update records: [B][8] (top_slots > 0)
    float2 *ep;   // this step's slab of episode ends (return, length as int bits): [B]; NULL: episode log off
    float4 *opt;  // this step's slab of option terminations (end x, end y, duration bits, record word 2): [B]; NULL: option log off
    int traj;     // trajectory log on: episode ends are marked in the event byte (SCG_EV_EPEND | SCG_EV_GOAL) as with the episode log
};

// Q_slot(z, .) for the lanes of `mask` (a warp-uniform ballot), compacted: N1 lanes share one of those envs, one leading
// multi-index digit c0 each, and the partial sums are folded back to the env's own lane.  `z` and `slot` are the env's
// phasors and weight-table slot (valid on the lanes of mask); q receives the 5 values on those lanes.
template <int N1, bool SMEMW>
__device__ __forceinline__ void warp_compact_q(unsigned mask, bool in_mask, int lane, const float2 z[4], int slot_id,
                                               const float *Wt_staged, int k_opt, int K, const float *Wt_global,
                                               float q[SCG_A]) {
    constexpr int SF = WtLayout<N1>::SLOT_FLOATS;
    constexpr unsigned FULL = 0xffffffffu;
    constexpr int PER = 32 / N1;                                 // envs served per pass
    const int my_rank = __popc(mask & ((1u << lane) - 1u));      // rank of this lane among the lanes of mask
    const int grp = lane / N1, c0 = lane - grp * N1;
    for (int base = 0; base < __popc(mask); base += PER) {
        const unsigned src = __fns(mask, 0, base + grp + 1);     // lane of the (base+grp)-th env of mask
        const bool have = grp < PER && src < 32u;
        const int sl = have ? (int)src : 0;
        float2 zs[4];
#pragma unroll
        for (int dd = 0; dd < 4; ++dd) {
            zs[dd].x = __shfl_sync(FULL, z[dd].x, sl);
            zs[dd].y = __shfl_sync(FULL, z[dd].y, sl);
        }
        const int os = __shfl_sync(FULL, slot_id, sl);
        float qp[SCG_A] = {0.f, 0.f, 0.f, 0.f, 0.f};
        // staged table: option slots 0 .. k_opt-1, then the top-level slots K .. Kall-1; anything else (an option
        // promoted after the host sized this launch) is read through the global path
        const bool staged = os < k_opt || os >= K;
        if (SMEMW && __any_sync(FULL, have && !staged)) {
            if (have) scg_q_c0<N1, false>(c0, zs, WCur<false>(Wt_global, SF, os), qp);
        } else {
            if (have) scg_q_c0<N1, SMEMW>(c0, zs, WCur<SMEMW>(SMEMW ? Wt_staged : Wt_global, SF, SMEMW && os >= K ? os - K + k_opt : os), qp);
        }
#pragma unroll
        for (int dd = 1; dd < N1; ++dd) {                        // group head (c0 == 0) gathers the partial sums
#pragma unroll
            for (int i = 0; i < SCG_A; ++i) {
                const float v = __shfl_down_sync(FULL, qp[i], dd);
                if (c0 == 0) qp[i] += v;
            }
        }
        const int rel = my_rank - base;
        const bool mine = in_mask && rel >= 0 && rel < PER;
        const int head = mine ? rel * N1 : 0;
#pragma unroll
        for (int i = 0; i < SCG_A; ++i) {
            const float v = __shfl_sync(FULL, qp[i], head);
            if (mine) q[i] = v;
        }
    }
}

template <int N1, bool SMEMW, bool PAIR, int NTH, bool TOP>
__global__ void __launch_bounds__(NTH, 512 / NTH) k_agent_step(const __grid_constant__ StepArgs args) {
    extern __shared__ __align__(128) unsigned char smem[];
    __shared__ __align__(8) unsigned long long bar;
    const scg_agent_t &g = args.ag;
    unsigned char *w_smem = smem + ((args.blob_bytes + 127) & ~127);
    // Programmatic dependent launch: let the next step kernel start its prologue (map + weight staging) under
    // this kernel's tail, and do our own staging before waiting for the previous kernel - unless that kernel
    // may have rewritten the weights.
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    if (args.wait_first) asm volatile("griddepcontrol.wait;" ::: "memory");
    // the map moves with one bulk-TMA copy, and so do the weights: a slot of the packed table is contiguous, so the
    // staged table is the option slots in use (0 .. k_opt-1) followed by the top-level learner's slots (K .. Kall-1)
    constexpr int SF = WtLayout<N1>::SLOT_FLOATS, SB = WtLayout<N1>::SLOT_BYTES;
    const int k_opt = args.k_stage - g.top_slots;
    stage3(smem, args.map_blob, args.blob_bytes, w_smem, g.Wt, SMEMW ? k_opt * SB : 0, w_smem + (size_t)k_opt * SB,
           g.Wt + (size_t)g.K * SF, SMEMW ? g.top_slots * SB : 0, &bar);
    if (!args.wait_first) asm volatile("griddepcontrol.wait;" ::: "memory");
    const StepMap m = make_step_map(smem);
    const ScgMapHeader *mh = reinterpret_cast<const ScgMapHeader *>(smem);
    const float *Wt = SMEMW ? reinterpret_cast<const float *>(w_smem) : g.Wt;
    const int K = g.K;
    // controller state lives on the device (scg_agent_manage promotes options in place): the launch was sized with the
    // host's lower bound of n_active (k_stage), the truth is read here
    const int n_act = g.ctl->n_active;
    const uint32_t amask = g.ctl->active_mask;
    const int gest = min(n_act, K - 1);
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, nw = blockDim.x >> 5;
    const int n_tiles = (args.b_end - args.b_begin + 31) >> 5;
    constexpr unsigned FULL = 0xffffffffu;
    // warp-granular work, interleaved over CTAs: tile i goes to CTA i % grid, warp i / grid.  The warp stays
    // converged through the whole tile (lanes past the batch end compute on a clamped index and skip stores).
    // Inside a window nothing couples the envs (the weights are frozen), so a launch runs n_steps consecutive
    // steps of every env with the env's state in registers: one load and one store of the per-env state, one
    // staging of the map and the weights and one launch per window instead of per step.
    for (int tile = w * gridDim.x + blockIdx.x; tile < n_tiles; tile += gridDim.x * nw) {
        const bool valid = args.b_begin + tile * 32 + lane < args.b_end;
        const int b = valid ? args.b_begin + tile * 32 + lane : args.b_end - 1;
        const uint32_t env = g.env_offset + (uint32_t)b;
        float sx = g.x[b], sy = g.y[b], svx = g.vx[b], svy = g.vy[b];
        // (ids poked in from outside are clamped: an out-of-range option or action must not index past the tables)
        int a = min(max(g.action[b], 0), SCG_A - 1), o = min(max(g.option[b], 0), g.K - 1);
        int t_opt = g.t_opt[b], ep = g.ep_steps[b];
        float ret = g.ep_return[b], qc = PAIR ? 0.f : g.q_carry[b];
        float stx = g.start_xy[2 * b], sty = g.start_xy[2 * b + 1];
        // top-level learner: velocity at the option's start, discounted task reward since, gamma^steps
        float stvx = 0.f, stvy = 0.f, oret = 0.f, odisc = 1.f;
        if (TOP) { stvx = g.start_vxy[2 * b]; stvy = g.start_vxy[2 * b + 1]; oret = g.opt_ret[b]; odisc = g.opt_disc[b]; }
        float r_env = 0.f, delta = 0.f;
        int fl = 0;
        for (int s = 0; s < args.n_steps; ++s) {
            const uint32_t step = g.step + (uint32_t)s;
            // 1: env step
            float nx = sx, ny = sy, nvx = svx, nvy = svy;
            if (g.cull) pinball_step<true>(m, nx, ny, nvx, nvy, a, r_env, fl);
            else pinball_step<false>(m, nx, ny, nvx, nvy, a, r_env, fl);
            const bool env_done = (fl & SCG_FLAG_DONE) != 0;
            // 4a: Q_o(s2, .) (and Q_o(s, .) when the carried value is stale: first step after a weight change)
            float2 zb[4];
            scg_phasors(nx, ny, nvx, nvy, zb);
            float qb[SCG_A], qsa = qc;
            // an option promoted after the host sized this launch (o >= k_stage) is not in the staged table: the warp
            // then reads the weights through the global path for this step (rare and transient)
            const bool unstaged = SMEMW && __any_sync(FULL, o >= k_opt);
            if (PAIR && s == 0) {
                float2 za[4];
                scg_phasors(sx, sy, svx, svy, za);
                float qa[SCG_A];
                if (unstaged) scg_q_pair<N1, false>(za, zb, WCur<false>(g.Wt, SF, o), qa, qb);
                else scg_q_pair<N1, SMEMW>(za, zb, WCur<SMEMW>(Wt, SF, o), qa, qb);
                qsa = 0.f;
#pragma unroll
                for (int i = 0; i < SCG_A; ++i) qsa = (i == a) ? qa[i] : qsa;
            } else {
                if (unstaged) scg_q_one<N1, false>(zb, WCur<false>(g.Wt, SF, o), qb);
                else scg_q_one<N1, SMEMW>(zb, WCur<SMEMW>(Wt, SF, o), qb);
            }
            // 2-3: initiation bits of s2, termination, option reward
            const uint32_t bits = scg_init_bits(g.theta, K, amask, nx, ny);
            const uint32_t pm = g.ctl->parents[o];
            const bool hit = (((pm & SCG_GOAL_BIT) != 0) && env_done) || ((bits & pm & ~SCG_GOAL_BIT) != 0);
            t_opt += 1;
            ep += 1;
            const bool left = ((amask >> o) & 1u) && !((bits >> o) & 1u);
            const bool ep_timeout = (ep >= g.max_episode_steps) && !env_done;
            const bool term = env_done || hit || (t_opt >= g.option_timeout) || left || ep_timeout;
            const float r = __fadd_rn(r_env, (hit && !env_done) ? g.option_bonus : 0.f);
            // 4b: a2, TD error
            const int a2 = scg_eps_greedy(qb, g.epsilon, scg_draw(g.seed, env, step, SCG_STREAM_ACTION));
            float qs2 = 0.f;
#pragma unroll
            for (int i = 0; i < SCG_A; ++i) qs2 = (i == a2) ? qb[i] : qs2;
            delta = __fsub_rn(__fadd_rn(r, __fmul_rn(__fmul_rn(g.gamma, term ? 0.f : 1.f), qs2)), qsa);
            ret += r_env;
            if (TOP) {   // SMDP return of the running option (oracle/agent.py: this operation order)
                oret = __fadd_rn(oret, __fmul_rn(odisc, r_env));
                odisc = __fmul_rn(odisc, g.gamma);
            }
            const bool reset = env_done || ep_timeout;
            {   // cnt[o] += 1, one atomic per (warp, option)
                const uint32_t peers = __match_any_sync(FULL, valid ? o : -1);
                if (valid && (__ffs(peers) - 1) == lane) atomicAdd(g.cnt + o, __popc(peers));
            }
            if (valid) {
                // 5: the step record for the window sweep
                const uint32_t meta = (uint32_t)a | ((uint32_t)o << 8) | (term ? SCG_META_ZERO_AFTER : 0u) | SCG_META_ACTIVE;
                float4 *rec = args.rec + ((size_t)s * g.B + b) * 2;
                rec[0] = make_float4(sx, sy, svx, svy);
                rec[1] = make_float4(delta, __uint_as_float(meta), 0.f, 0.f);
                // 6: example for option o's initiation classifier: an event byte per env-step and, at a termination, the
                // option's start position go to the event history; k_ring appends them to the ring in the oracle's order
                // (step, then env) when the controller next needs the rings
                args.ev[(size_t)s * g.B + b] = term ? (uint8_t)(SCG_EV_TERM | ((hit && t_opt <= g.init_horizon) ? SCG_EV_HIT : 0) | o) : (uint8_t)0;
                if (term) {
                    args.pos[(size_t)s * g.B + b] = make_float2(stx, sty);
                    atomicAdd((hit ? g.n_success : g.n_fail) + o, 1);
                    if (args.opt != nullptr) {   // option log: where the execution ended (before the reset), how long, why
                        const uint32_t why = (uint32_t)o | (hit ? SCG_OL_HIT : 0u) | ((hit && t_opt <= g.init_horizon) ? SCG_OL_LABEL : 0u) |
                                             (env_done ? SCG_OL_ENV_DONE : 0u) | ((t_opt >= g.option_timeout) ? SCG_OL_OPTION_TIMEOUT : 0u) |
                                             (left ? SCG_OL_LEFT : 0u) | (ep_timeout ? SCG_OL_EPISODE_TIMEOUT : 0u);
                        args.opt[(size_t)s * g.B + b] = make_float4(nx, ny, __int_as_float(t_opt), __uint_as_float(why));
                    }
                }
                // 7: env reset
                if (reset) {
                    if (args.ep != nullptr || args.traj) {   // episode / trajectory log: the end (always also a termination) goes into the
                        const size_t i = (size_t)s * g.B + b;   // event byte, with the episode log its return and length beside it
                        args.ev[i] |= (uint8_t)(SCG_EV_EPEND | (env_done ? SCG_EV_GOAL : 0u));
                        if (args.ep != nullptr) args.ep[i] = make_float2(ret, __int_as_float(ep));
                    }
                    const uint4 rr = scg_draw(g.seed, env, step, SCG_STREAM_RESET);
                    const int ns = mh->n_starts;
                    const int pick = min((int)__fmul_rn(scg_u01(rr.x), (float)ns), ns - 1);
                    const float2 s0 = reinterpret_cast<const float2 *>(smem + mh->off_starts)[pick];
                    nx = s0.x; ny = s0.y; nvx = 0.f; nvy = 0.f;
                    atomicAdd(reinterpret_cast<unsigned long long *>(g.stats) + 0, 1ull);
                    if (env_done) atomicAdd(reinterpret_cast<unsigned long long *>(g.stats) + 1, 1ull);
                    atomicAdd(reinterpret_cast<double *>(g.stats) + 2, (double)ret);
                    g.ep_count[b] += 1;
                    g.last_return[b] = ret;
                    ret = 0.f;
                    ep = 0;
                }
            }
            // 8: option re-selection.  Terminations are rare, so every Q evaluation they need is compacted inside the
            // warp (warp_compact_q): N1 lanes share one terminated env, one leading digit c0 each.
            int o_next = o, a_next = a2;
            float q_next = qs2;
            const bool tv = term && valid;
            const unsigned tmask = __ballot_sync(FULL, tv);
            if (tmask) {
                float2 zn[4] = {zb[0], zb[1], zb[2], zb[3]};
                uint32_t bn = bits;
                if (tv) {
                    if (reset) {
                        bn = scg_init_bits(g.theta, K, amask, nx, ny);
                        scg_phasors(nx, ny, nvx, nvy, zn);
                    }
                    o_next = bn ? (__ffs(bn) - 1) : gest;
                }
                if (TOP) {
                    // The top-level SMDP learner (oracle/agent.py module docstring).  Q_top(s, j) is row j % 5 of slot
                    // K + j / 5.  (i) max over the admissible slots at s2 for the bootstrap, and - the same pass when the
                    // env was not reset - the greedy choice at s_next; (ii) Q_top(s0, o); (iii) delta_top -> win_top.
                    const uint32_t adm2 = bits | (1u << gest), admn = bn | (1u << gest);
                    float m2 = -INFINITY, mn = -INFINITY;
                    int best = gest;
                    const unsigned rmask = __ballot_sync(FULL, tv && reset);
                    for (int sl = 0; sl < g.top_slots; ++sl) {
                        float qt[SCG_A] = {0.f, 0.f, 0.f, 0.f, 0.f};
                        warp_compact_q<N1, SMEMW>(tmask, tv, lane, zb, K + sl, Wt, k_opt, K, g.Wt, qt);
#pragma unroll
                        for (int i = 0; i < SCG_A; ++i) {
                            const int j = sl * SCG_A + i;
                            if (j < K && ((adm2 >> j) & 1u)) {
                                m2 = fmaxf(m2, qt[i]);
                                if (!reset && qt[i] > mn) { mn = qt[i]; best = j; }     // first admissible maximum
                            }
                        }
                        if (rmask) {          // envs that were reset choose at the start state instead
                            float qr[SCG_A] = {0.f, 0.f, 0.f, 0.f, 0.f};
                            warp_compact_q<N1, SMEMW>(rmask, tv && reset, lane, zn, K + sl, Wt, k_opt, K, g.Wt, qr);
#pragma unroll
                            for (int i = 0; i < SCG_A; ++i) {
                                const int j = sl * SCG_A + i;
                                if (reset && j < K && ((admn >> j) & 1u) && qr[i] > mn) { mn = qr[i]; best = j; }
                            }
                        }
                    }
                    float2 z0[4];
                    scg_phasors(stx, sty, stvx, stvy, z0);
                    float q0v[SCG_A] = {0.f, 0.f, 0.f, 0.f, 0.f};
                    warp_compact_q<N1, SMEMW>(tmask, tv, lane, z0, K + o / SCG_A, Wt, k_opt, K, g.Wt, q0v);
                    if (tv) {
                        float q0 = 0.f;
                        const int row = o - (o / SCG_A) * SCG_A;
#pragma unroll
                        for (int i = 0; i < SCG_A; ++i) q0 = (i == row) ? q0v[i] : q0;
                        const float boot = reset ? 0.f : __fmul_rn(odisc, m2);
                        const float dtop = __fsub_rn(__fadd_rn(oret, boot), q0);
                        float4 *tr = reinterpret_cast<float4 *>(args.top) + ((size_t)s * g.B + b) * 2;
                        tr[0] = make_float4(stx, sty, stvx, stvy);
                        tr[1] = make_float4(dtop, __int_as_float(o), 0.f, 0.f);
                        // eps_top-greedy over the admissible slots at s_next
                        const uint4 rt = scg_draw(g.seed, env, step, SCG_STREAM_TOP);
                        const int n_adm = __popc(admn);
                        const int pick = min((int)__fmul_rn(scg_u01(rt.y), (float)n_adm), n_adm - 1);
                        const int rnd_o = (int)__fns(admn, 0, pick + 1);
                        o_next = (scg_u01(rt.x) < g.epsilon_top) ? rnd_o : best;
                    }
                }
                float qn[SCG_A] = {0.f, 0.f, 0.f, 0.f, 0.f};
                warp_compact_q<N1, SMEMW>(tmask, tv, lane, zn, o_next, Wt, k_opt, K, g.Wt, qn);
                if (tv) {
                    a_next = scg_eps_greedy(qn, g.epsilon, scg_draw(g.seed, env, step, SCG_STREAM_RESELECT));
#pragma unroll
                    for (int i = 0; i < SCG_A; ++i) q_next = (i == a_next) ? qn[i] : q_next;
                    t_opt = 0;
                    stx = nx;
                    sty = ny;
                    if (TOP) { stvx = nvx; stvy = nvy; oret = 0.f; odisc = 1.f; }
                }
            }
            // the next step starts from here
            sx = nx; sy = ny; svx = nvx; svy = nvy;
            a = a_next; o = o_next; qc = q_next;
        }
        if (valid) {
            g.x2[b] = sx; g.y2[b] = sy; g.vx2[b] = svx; g.vy2[b] = svy;
            g.action[b] = a;
            g.option[b] = o;
            g.t_opt[b] = t_opt;
            g.ep_steps[b] = ep;
            g.ep_return[b] = ret;
            g.q_carry[b] = qc;
            g.start_xy[2 * b] = stx;
            g.start_xy[2 * b + 1] = sty;
            if (TOP) { g.start_vxy[2 * b] = stvx; g.start_vxy[2 * b + 1] = stvy; g.opt_ret[b] = oret; g.opt_disc[b] = odisc; }
            g.reward[b] = r_env;
            g.flags[b] = fl;
            g.delta[b] = delta;
        }
    }
}

// ---- launch plumbing --------------------------------------------------------------------------------
template <int N1, bool SMEMW, bool PAIR, int NTH, bool TOP>
static int launch_step_tt(const StepArgs &args, size_t smem, cudaStream_t st) {
    auto kern = k_agent_step<N1, SMEMW, PAIR, NTH, TOP>;
    static ScgKernelCfg cfgc = {};
    int per_sm = 0;
    int rcc = scg_configure(cfgc, kern, NTH, smem, &per_sm);
    if (rcc) return rcc;
    const int sms = scg_num_sms();
    if (per_sm < 1 || sms < 1) return SCG_ELIMIT;
    constexpr int WPC = NTH / 32;                       // warps (tiles in flight) per CTA
    const int n_tiles = (args.b_end - args.b_begin + 31) / 32;
    // enough CTAs for one warp per tile if they all fit at once, else every resident slot
    int grid = (n_tiles + WPC - 1) / WPC;
    if (grid > sms) {   // same number of CTAs on every SM: as many rounds of one CTA per SM as the tiles need, if resident
        const int rounds = std::min(per_sm, (grid + sms - 1) / sms);
        grid = sms * rounds;
    }
    grid = std::max(grid, 1);
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(grid);
    cfg.blockDim = dim3(NTH);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    SCG_CUDA_OK(cudaLaunchKernelEx(&cfg, kern, args));
    ++g_scg_launches;
    return 0;
}

template <int N1, bool SMEMW, bool PAIR, int NTH>
static int launch_step_t(const StepArgs &args, size_t smem, cudaStream_t st) {
    if (args.ag.top_slots > 0) return launch_step_tt<N1, SMEMW, PAIR, NTH, true>(args, smem, st);
    return launch_step_tt<N1, SMEMW, PAIR, NTH, false>(args, smem, st);
}

// mode 0: weights through the read-only global path; 1: staged to shared memory, two 256-thread CTAs per SM;
// 2: staged, one 512-thread CTA per SM (order 5: the options in use take up to ~200 KB)
template <int N1>
static int launch_step_n(const StepArgs &args, int mode, bool pair, cudaStream_t st) {
    const size_t blob = (size_t)((args.blob_bytes + 127) & ~127);
    if (mode == 1) {
        const size_t smem = blob + args.w_bytes;
        return pair ? launch_step_t<N1, true, true, 256>(args, smem, st) : launch_step_t<N1, true, false, 256>(args, smem, st);
    }
    if (mode == 2) {
        const size_t smem = blob + args.w_bytes;
        return pair ? launch_step_t<N1, true, true, 512>(args, smem, st) : launch_step_t<N1, true, false, 512>(args, smem, st);
    }
    return pair ? launch_step_t<N1, false, true, 256>(args, blob, st) : launch_step_t<N1, false, false, 256>(args, blob, st);
}

static int check_agent(const scg_map_t *map, const scg_ctx_t *ctx, const scg_agent_t *ag) {
    if (!map || !ctx || !ag) return SCG_EINVAL;
    if (ag->top_slots < 0 || ag->K + ag->top_slots != ctx->K || ag->order != ctx->order) return SCG_EINVAL;
    if (ag->K < 1 || ag->K + ag->top_slots > SCG_MAX_OPTIONS) return SCG_ELIMIT;
    if (ag->top_slots > 0 && (ag->top_slots * SCG_A < ag->K || !ag->win_top || !ag->start_vxy || !ag->opt_ret || !ag->opt_disc))
        return SCG_EINVAL;
    if (ag->B < 0 || ag->win_cap < 1 || ag->win_cap > SCG_WIN_MAX || ag->win_len < 0 || ag->win_len >= ag->win_cap)
        return SCG_EINVAL;
    if (ag->n_active < 0 || ag->n_active > ag->K - 1 || !ag->ctl || !ag->ev_hist || !ag->ev_pos) return SCG_EINVAL;
    if (ag->ev_cap < 2 * ag->win_cap || ag->ev_len < ag->win_len || ag->ev_len > ag->ev_cap || ag->ring_len < 0 ||
        ag->ring_len > ag->ev_len)
        return SCG_EINVAL;
    if (!scg_episode_log_ok(ag) || !scg_option_log_ok(ag) || !scg_traj_log_ok(ag) || !scg_occupancy_ok(ag))
        return SCG_EINVAL;
    if (map->hdr.blob_bytes > 160 * 1024) return SCG_ELIMIT;
    return 0;
}

// ---- trajectory log --------------------------------------------------------------------------------
// k_traj_gather: the tracked envs' records of window steps [s0, s0 + n_steps), copied out of the step records (win_rec)
// and the event bytes the step kernel left; record r = (step, tracked env) in (step, env) order.  One CTA: it reads the
// count, every thread writes its records (only the last `cap` of this pass, so every slot has one writer), then one
// thread advances the count.  It is launched without programmatic serialization and never triggers its dependents, so
// the next step kernel's griddepcontrol.wait covers all of it before win_rec is rewritten.
#define TRAJ_NT 1024

__global__ void __launch_bounds__(TRAJ_NT) k_traj_gather(const float4 *__restrict__ rec, const uint8_t *__restrict__ ev,
                                                         const int32_t *__restrict__ env, int traj_n, int n_steps, int B,
                                                         uint32_t env_offset, uint32_t step0, uint4 *log,
                                                         long long *count, uint32_t cap) {
    const unsigned long long c0 = (unsigned long long)*count;
    const uint32_t n = (uint32_t)traj_n * (uint32_t)n_steps;
    const uint32_t first = n > cap ? n - cap : 0u;     // records of this pass that the ring keeps
#pragma unroll 4
    for (uint32_t r = first + threadIdx.x; r < n; r += TRAJ_NT) {
        const uint32_t s = r / (uint32_t)traj_n, j = r - s * (uint32_t)traj_n;
        const int b = __ldg(env + j);
        uint4 w0 = make_uint4(step0 + s, 0xFFFFFFFFu, 0u, 0u), w1 = make_uint4(0u, 0u, 0u, 0u);
        if (b >= 0 && b < B) {
            const size_t i = (size_t)s * B + b;
            const float4 st = __ldg(rec + 2 * i), dm = __ldg(rec + 2 * i + 1);
            const uint32_t meta = __float_as_uint(dm.y), e = __ldg(ev + i);
            const uint32_t word = (meta & 7u) | (((meta >> 8) & 0xFFu) << 8) | ((meta & SCG_META_ZERO_AFTER) ? SCG_TL_TERM : 0u) |
                                  ((e & SCG_EV_HIT) ? SCG_TL_LABEL : 0u) | ((e & SCG_EV_EPEND) ? SCG_TL_EPEND : 0u) |
                                  ((e & SCG_EV_GOAL) ? SCG_TL_GOAL : 0u);
            w0 = make_uint4(step0 + s, env_offset + (uint32_t)b, __float_as_uint(st.x), __float_as_uint(st.y));
            w1 = make_uint4(__float_as_uint(st.z), __float_as_uint(st.w), word, __float_as_uint(dm.x));
        }
        const size_t slot = (size_t)((c0 + r) % cap);
        log[2 * slot] = w0;
        log[2 * slot + 1] = w1;
    }
    __syncthreads();                                    // every thread has read the count
    if (threadIdx.x == 0) *count = (long long)(c0 + n);
}

extern "C" int scg_agent_traj(scg_ctx_t *ctx, scg_agent_t *ag, void *stream) {
    if (!ctx || !ag || !scg_traj_log_ok(ag)) return SCG_EINVAL;
    if (!ag->traj_log) return 0;
    if (ag->win_len > ag->win_cap || ag->ev_len < ag->win_len || ag->ev_len > ag->ev_cap || !ag->win_rec || !ag->ev_hist)
        return SCG_EINVAL;
    const int n = ag->win_len - ag->traj_len;
    if (n > 0) {
        // window step s is history row ev_len - win_len + s (as k_top reads it); the ring pass only recycles rows
        // between windows
        const size_t s0 = (size_t)ag->traj_len;
        const size_t row = (size_t)(ag->ev_len - ag->win_len) + s0;
        k_traj_gather<<<1, TRAJ_NT, 0, (cudaStream_t)stream>>>(
            reinterpret_cast<const float4 *>(ag->win_rec) + s0 * ag->B * 2, ag->ev_hist + row * ag->B, ag->traj_env,
            (int)ag->traj_n, n, ag->B, ag->env_offset, ag->step - (uint32_t)ag->win_len + (uint32_t)ag->traj_len,
            reinterpret_cast<uint4 *>(ag->traj_log), reinterpret_cast<long long *>(ag->traj_log_count), ag->traj_capacity);
        SCG_LAUNCH_CHECK();
    }
    ag->traj_len = ag->win_len;
    return 0;
}

// ---- occupancy grid --------------------------------------------------------------------------------
// k_occupancy: the step records of window steps [s0, s0 + n_steps) of all B envs, n = n_steps * B of them back to back
// in win_rec.  A record's option (meta word) and the cell of its (x, y) give its bin, key = (option * grid + iy) * grid
// + ix.  Many envs share a few cells (around the start positions, along walls), so one global atomic per record
// serialises on those addresses: each CTA counts its OCC_REC_PER_CTA records in 32-bit shared-memory bins, then adds
// its non-zero bins to the global counts (red.global.add.u64), at most one add per bin and CTA.  Bins beyond the shared
// memory of one CTA are split into chunks along blockIdx.y; a CTA counts the records whose key falls into its chunk.
// Integer adds make the counts independent of the order of the adds.  Launched like k_traj_gather: no programmatic
// serialization and no trigger, so the next step kernel's griddepcontrol.wait covers all of it before win_rec is
// rewritten.
#define OCC_NT 512
#define OCC_REC_PER_CTA 4096            // records per CTA: < 2^32, so the shared counters cannot overflow
#define OCC_SMEM_BINS 16384             // 64 KiB of shared counters per CTA

__global__ void __launch_bounds__(OCC_NT) k_occupancy(const float4 *__restrict__ rec, size_t n, int K, int grid,
                                                       int chunk_bins, unsigned long long *counts) {
    extern __shared__ uint32_t bins[];
    const int n_bins = K * grid * grid, lo = (int)blockIdx.y * chunk_bins;
    const int hi = min(lo + chunk_bins, n_bins);
    for (int j = threadIdx.x; j < hi - lo; j += OCC_NT) bins[j] = 0u;
    __syncthreads();
    const size_t end = min(n, (size_t)(blockIdx.x + 1) * OCC_REC_PER_CTA);
    for (size_t i = (size_t)blockIdx.x * OCC_REC_PER_CTA + threadIdx.x; i < end; i += OCC_NT) {
        const float2 xy = __ldg(reinterpret_cast<const float2 *>(rec + 2 * i));
        const uint32_t o = (__float_as_uint(__ldg(reinterpret_cast<const float *>(rec + 2 * i + 1) + 1)) >> 8) & 0xFFu;
        if (o >= (uint32_t)K) continue;
        // grid is a power of two: x * grid is exact, and the conversion truncates toward zero (include/scg_b200.h)
        const int ix = min(max(__float2int_rz(__fmul_rn(xy.x, (float)grid)), 0), grid - 1);
        const int iy = min(max(__float2int_rz(__fmul_rn(xy.y, (float)grid)), 0), grid - 1);
        const int key = ((int)o * grid + iy) * grid + ix;
        if (key >= lo && key < hi) atomicAdd(bins + (key - lo), 1u);
    }
    __syncthreads();
    for (int j = threadIdx.x; j < hi - lo; j += OCC_NT) {
        const uint32_t v = bins[j];
        if (v) atomicAdd(counts + lo + j, (unsigned long long)v);
    }
}

extern "C" int scg_agent_occupancy(scg_ctx_t *ctx, scg_agent_t *ag, void *stream) {
    if (!ctx || !ag || !scg_occupancy_ok(ag)) return SCG_EINVAL;
    if (!ag->occ_counts) return 0;
    if (ag->win_len > ag->win_cap || ag->B < 0 || ag->K < 1 || ag->K > SCG_MAX_OPTIONS || !ag->win_rec) return SCG_EINVAL;
    const int n = ag->win_len - ag->occ_len;
    if (n > 0 && ag->B > 0) {
        static ScgKernelCfg cfgc = {};
        int per_sm, rc;
        if ((rc = scg_configure(cfgc, k_occupancy, OCC_NT, OCC_SMEM_BINS * sizeof(uint32_t), &per_sm))) return rc;
        const int grid = (int)ag->occ_grid, n_bins = ag->K * grid * grid;
        const int chunk_bins = std::min(n_bins, OCC_SMEM_BINS);
        const size_t s0 = (size_t)ag->occ_len, m = (size_t)n * ag->B;
        const dim3 blocks((unsigned)((m + OCC_REC_PER_CTA - 1) / OCC_REC_PER_CTA), (unsigned)((n_bins + chunk_bins - 1) / chunk_bins));
        k_occupancy<<<blocks, OCC_NT, chunk_bins * sizeof(uint32_t), (cudaStream_t)stream>>>(
            reinterpret_cast<const float4 *>(ag->win_rec) + s0 * ag->B * 2, m, ag->K, grid, chunk_bins,
            reinterpret_cast<unsigned long long *>(ag->occ_counts));
        SCG_LAUNCH_CHECK();
    }
    ag->occ_len = ag->win_len;
    return 0;
}

extern "C" int scg_agent_flush(scg_ctx_t *ctx, scg_agent_t *ag, void *stream) {
    if (!ctx || !ag) return SCG_EINVAL;
    int rc;
    // the trajectory log and the occupancy grid take the window's last steps before anything else reads or recycles
    // the window
    if ((rc = scg_agent_traj(ctx, ag, stream))) return rc;
    if ((rc = scg_agent_occupancy(ctx, ag, stream))) return rc;
    if (ag->win_len <= 0 || ag->B <= 0) { ag->win_len = ag->traj_len = ag->occ_len = 0; return 0; }
    // option ids in the records are 0 .. n_active (the gestating slot); n_active is the host's lower bound of the
    // device's value: records of an option promoted since then are folded through the sweep's global-memory path
    const int k_used = std::min(ag->K, std::max(ag->n_active, 0) + 1);
    if ((rc = scg_launch_top(ctx, ag, (cudaStream_t)stream))) return rc;     // the top-level learner's SMDP updates
    const int n_slabs = scg_launch_window(ctx, ag->B, ag->win_len, k_used, ag->win_rec, ag->trace, ag->gamma * ag->lambda,
                                          ag->dW, (cudaStream_t)stream);
    if (n_slabs <= 0) return n_slabs == 0 ? SCG_EINVAL : n_slabs;
    if ((rc = scg_reduce_window(ctx, n_slabs, k_used, ag->dW, (cudaStream_t)stream))) return rc;
    ag->win_len = ag->traj_len = ag->occ_len = 0;
    // the event history must have room for the next full window: when it has not, bring the rings up to date now
    if (ag->ev_len + ag->win_cap > ag->ev_cap && (rc = scg_agent_ring(ctx, ag, stream))) return rc;
    return 0;
}

// n consecutive steps (1 <= n <= win_cap - win_len) in one launch; a full window is swept right away unless the
// caller defers that (defer_flush) to queue something of its own first
// b_begin/b_end: step only those envs and leave the bookkeeping to the call that steps the last part (b_end == B):
// scg_agent_step_host pipelines a step over parts of the batch
static int agent_steps(const scg_map_t *map, scg_ctx_t *ctx, scg_agent_t *ag, int n, void *stream,
                       bool defer_flush = false, int b_begin = 0, int b_end = -1) {
    if (b_end < 0) b_end = ag->B;
    cudaStream_t st = (cudaStream_t)stream;
    // promotions happen on the device (scg_agent_manage); the host learns of them from the mirror, without waiting
    if (ctx->h_mirror) ag->n_active = std::max(ag->n_active, std::min((int)ctx->h_mirror->ctl.n_active, ag->K - 1));
    StepArgs args;
    args.ag = *ag;
    args.map_blob = map->d_blob;
    args.blob_bytes = map->hdr.blob_bytes;
    // only the options that can be executed (ids 0 .. n_active) need their weights on chip
    args.k_stage = std::min(ag->K, std::max(ag->n_active, 0) + 1) + ag->top_slots;   // + the top-level learner's slots
    args.w_bytes = args.k_stage * scg_wt_slot_floats(ag->order) * (int)sizeof(float);
    args.rec = reinterpret_cast<float4 *>(ag->win_rec) + (size_t)ag->win_len * ag->B * 2;
    args.ev = ag->ev_hist + (size_t)ag->ev_len * ag->B;
    args.pos = reinterpret_cast<float2 *>(ag->ev_pos) + (size_t)ag->ev_len * ag->B;
    args.top = ag->win_top ? ag->win_top + (size_t)ag->win_len * ag->B * 8 : nullptr;
    args.ep = ag->ev_ep ? reinterpret_cast<float2 *>(ag->ev_ep) + (size_t)ag->ev_len * ag->B : nullptr;
    args.opt = ag->ev_opt ? reinterpret_cast<float4 *>(ag->ev_opt) + (size_t)ag->ev_len * ag->B : nullptr;
    args.traj = ag->traj_log != nullptr;
    args.n_steps = n;
    args.b_begin = b_begin;
    args.b_end = b_end;
    // weights go to shared memory when two CTAs per SM still fit next to the map, or one big CTA
    const size_t need = (size_t)args.w_bytes + args.blob_bytes + 256;
    const int mode = need <= 100 * 1024 ? 1 : (need <= 220 * 1024 ? 2 : 0);
    const bool pair = !ag->carry_valid;
    // a step kernel directly behind another step kernel of the same window may stage the weights early
    args.wait_first = !(ag->carry_valid && ag->win_len > 0 && !(ctx->prof_on && (ctx->prof_mask & 1)));
    int rc;
    if ((rc = scg_prof_push(ctx, 0, st, false))) return rc;
    DISPATCH_ORDER(ag->order, rc = launch_step_n<N1>(args, mode, pair, st));
    if (rc) return rc;
    if ((rc = scg_prof_push(ctx, 0, st, true))) return rc;
    if (b_end < ag->B) return 0;
    std::swap(ag->x, ag->x2); std::swap(ag->y, ag->y2);
    std::swap(ag->vx, ag->vx2); std::swap(ag->vy, ag->vy2);
    ag->step += n;
    ag->window_steps += n;
    ag->win_len += n;
    ag->ev_len += n;
    ag->carry_valid = 1;
    if (ag->win_len >= ag->win_cap && !defer_flush) return scg_agent_flush(ctx, ag, stream);
    return 0;
}

extern "C" int scg_agent_step(const scg_map_t *map, scg_ctx_t *ctx, scg_agent_t *ag, void *stream) {
    int rc = check_agent(map, ctx, ag);
    if (rc) return rc;
    if (ag->B == 0) return 0;
    return agent_steps(map, ctx, ag, 1, stream);
}

extern "C" int scg_agent_run(const scg_map_t *map, scg_ctx_t *ctx, scg_agent_t *ag, int n_steps, int sync_interval,
                             scg_xchg_t *xchg, void *stream) {
    if (n_steps < 0 || sync_interval < 0) return SCG_EINVAL;
    int rc = check_agent(map, ctx, ag);
    if (rc) return rc;
    if (ag->B == 0) return 0;
    for (int done = 0; done < n_steps;) {
        // as many steps as fit before the window is full, the sync is due, or the request ends
        int n = std::min(n_steps - done, ag->win_cap - ag->win_len);
        if (sync_interval > 0) n = std::min(n, std::max(1, sync_interval - ag->window_steps));
        if ((rc = agent_steps(map, ctx, ag, n, stream))) return rc;
        done += n;
        if (sync_interval > 0 && ag->window_steps >= sync_interval && (rc = scg_agent_sync(ctx, ag, xchg, stream)))
            return rc;
    }
    return 0;
}

extern "C" int scg_agent_sync(scg_ctx_t *ctx, scg_agent_t *ag, scg_xchg_t *xchg, void *stream) {
    if (!ctx || !ag || ag->K + ag->top_slots != ctx->K) return SCG_EINVAL;   // the apply covers the context's K slots
    int rc;
    if ((rc = scg_agent_flush(ctx, ag, stream))) return rc;
    if ((rc = scg_prof_push(ctx, 3, (cudaStream_t)stream, false))) return rc;
    if (xchg) rc = scg_xchg_sync(xchg, ag->K, ag->W, ag->Wt, ag->dW, ag->cnt, ag->alpha, ag->alpha_top, ag->window_steps, ag->n_success, ag->n_success_global, stream);
    else rc = scg_apply(ctx, ag->K, ag->W, ag->Wt, ag->dW, ag->cnt, ag->alpha, ag->alpha_top, ag->window_steps, stream);
    if (rc) return rc;
    if ((rc = scg_prof_push(ctx, 3, (cudaStream_t)stream, true))) return rc;
    ag->window_steps = 0;
    ag->carry_valid = 0;
    return 0;
}

// copy `rows` arrays of n bytes each; one cudaMemcpyAsync when they are contiguous on both sides
static int copy_rows(void *const *dst, const void *const *src, int rows, size_t n, cudaMemcpyKind kind, cudaStream_t st) {
    bool contig = true;
    for (int i = 1; i < rows; ++i)
        contig = contig && (const char *)dst[i] == (const char *)dst[0] + i * n && (const char *)src[i] == (const char *)src[0] + i * n;
    if (contig) {
        SCG_CUDA_OK(cudaMemcpyAsync(dst[0], src[0], n * rows, kind, st));
        return 0;
    }
    for (int i = 0; i < rows; ++i) SCG_CUDA_OK(cudaMemcpyAsync(dst[i], src[i], n, kind, st));
    return 0;
}

// One step through host buffers.  The three phases - state and action in, the step kernel, results out - are a chain
// for any one env but not across envs, so the batch is cut into parts (multiples of 32 envs) and pipelined: part p+1
// is copied in while part p is stepped and part p-1 is copied out (PCIe is full duplex; copies in and copies out have
// a stream each, the kernels stay on the caller's stream, events order the three).  Rows of the SoA blocks are moved
// with one pitched copy per block.  Two parts measured fastest (DESIGN.md section 6); small batches, buffers that are not
// back to back and profiled step kernels take the plain sequence.
extern "C" int scg_agent_step_host(const scg_map_t *map, scg_ctx_t *ctx, scg_agent_t *ag, const float *h_state_soa,
                                   const int *h_action, float *h_state2_soa, float *h_reward, int *h_flags,
                                   int *h_action2, float *h_delta, void *stream) {
    if (!map || !ctx || !ag || !h_state_soa || !h_action || !h_state2_soa || !h_reward || !h_flags || !h_action2 ||
        !h_delta)
        return SCG_EINVAL;
    cudaStream_t st = (cudaStream_t)stream;
    const int B = ag->B;
    const size_t n = (size_t)B * sizeof(float);
    int rc;
    if ((rc = check_agent(map, ctx, ag))) return rc;
    // pitched copies need the SoA blocks back to back on both sides (they are in the Python layer: [4][B] tensors)
    auto rows4 = [&](const void *a, const void *b, const void *c, const void *d) {
        return (const char *)b == (const char *)a + n && (const char *)c == (const char *)a + 2 * n && (const char *)d == (const char *)a + 3 * n;
    };
    const bool blocks = rows4(ag->x, ag->y, ag->vx, ag->vy) && rows4(ag->x2, ag->y2, ag->vx2, ag->vy2) &&
                        rows4(ag->reward, ag->flags, ag->action, ag->delta) && rows4(h_reward, h_flags, h_action2, h_delta);
    int parts = SCG_HOST_PARTS_MAX;
    if (!blocks || B < 64 * parts || (ctx->prof_on && (ctx->prof_mask & 1))) parts = 1;
    if (parts == 1) {
        {
            void *dst[4] = {ag->x, ag->y, ag->vx, ag->vy};
            const void *src[4] = {h_state_soa, h_state_soa + B, h_state_soa + 2 * (size_t)B, h_state_soa + 3 * (size_t)B};
            if ((rc = copy_rows(dst, src, 4, n, cudaMemcpyHostToDevice, st))) return rc;
        }
        SCG_CUDA_OK(cudaMemcpyAsync(ag->action, h_action, n, cudaMemcpyHostToDevice, st));
        ag->carry_valid = 0;   // state and action came from outside: Q_o(s, a) must be evaluated
        if (B == 0) return 0;
        if ((rc = agent_steps(map, ctx, ag, 1, stream, /*defer_flush=*/true))) return rc;
        {   // the step swapped the buffers: x..vy is the new state
            void *dst[4] = {h_state2_soa, h_state2_soa + B, h_state2_soa + 2 * (size_t)B, h_state2_soa + 3 * (size_t)B};
            const void *src[4] = {ag->x, ag->y, ag->vx, ag->vy};
            if ((rc = copy_rows(dst, src, 4, n, cudaMemcpyDeviceToHost, st))) return rc;
        }
        {   // reward, flags, next action, TD error: one copy when both sides keep them back to back
            void *dst[4] = {h_reward, h_flags, h_action2, h_delta};
            const void *src[4] = {ag->reward, ag->flags, ag->action, ag->delta};
            if ((rc = copy_rows(dst, src, 4, n, cudaMemcpyDeviceToHost, st))) return rc;
        }
        // The results do not depend on the trace sweep: when this step filled the window, the sweep is queued behind the
        // copies and the host only waits for the copies, so the sweep overlaps the caller's next host-side work and H2D.
        if (!ctx->host_ev) SCG_CUDA_OK(cudaEventCreateWithFlags(&ctx->host_ev, cudaEventDisableTiming));
        SCG_CUDA_OK(cudaEventRecord(ctx->host_ev, st));
        if (ag->win_len >= ag->win_cap && (rc = scg_agent_flush(ctx, ag, stream))) return rc;
        SCG_CUDA_OK(cudaEventSynchronize(ctx->host_ev));
        return 0;
    }
    for (int i = 0; i < 2; ++i)
        if (!ctx->host_st[i]) SCG_CUDA_OK(cudaStreamCreateWithFlags(&ctx->host_st[i], cudaStreamNonBlocking));
    for (int i = 0; i < 2 * SCG_HOST_PARTS_MAX + 1; ++i)
        if (!ctx->host_evs[i]) SCG_CUDA_OK(cudaEventCreateWithFlags(&ctx->host_evs[i], cudaEventDisableTiming));
    if (!ctx->host_ev) SCG_CUDA_OK(cudaEventCreateWithFlags(&ctx->host_ev, cudaEventDisableTiming));
    cudaStream_t s_in = ctx->host_st[0], s_out = ctx->host_st[1];
    cudaEvent_t *ev_in = ctx->host_evs, *ev_step = ctx->host_evs + SCG_HOST_PARTS_MAX, ev_entry = ctx->host_evs[2 * SCG_HOST_PARTS_MAX];
    // whatever the caller queued on its stream (a sweep, the controller) stays ahead of the copies in
    SCG_CUDA_OK(cudaEventRecord(ev_entry, st));
    SCG_CUDA_OK(cudaStreamWaitEvent(s_in, ev_entry, 0));
    ag->carry_valid = 0;       // state and action came from outside: Q_o(s, a) must be evaluated
    // the step writes the new state to x2 .. vy2 (the buffers are swapped by the call that steps the last part)
    float *d_new = ag->x2;
    float *d_out = ag->reward;
    const int per = ((B + parts - 1) / parts + 31) & ~31;
    for (int p = 0; p < parts; ++p) {
        const int b0 = p * per, b1 = std::min(B, b0 + per);
        if (b0 >= b1) { parts = p; break; }
        const size_t w = (size_t)(b1 - b0) * sizeof(float);
        SCG_CUDA_OK(cudaMemcpy2DAsync(ag->x + b0, n, h_state_soa + b0, n, w, 4, cudaMemcpyHostToDevice, s_in));
        SCG_CUDA_OK(cudaMemcpyAsync(ag->action + b0, h_action + b0, w, cudaMemcpyHostToDevice, s_in));
        SCG_CUDA_OK(cudaEventRecord(ev_in[p], s_in));
    }
    for (int p = 0; p < parts; ++p) {
        const int b0 = p * per, b1 = std::min(B, b0 + per);
        const size_t w = (size_t)(b1 - b0) * sizeof(float);
        SCG_CUDA_OK(cudaStreamWaitEvent(st, ev_in[p], 0));
        if ((rc = agent_steps(map, ctx, ag, 1, stream, /*defer_flush=*/true, b0, b1))) return rc;
        SCG_CUDA_OK(cudaEventRecord(ev_step[p], st));
        SCG_CUDA_OK(cudaStreamWaitEvent(s_out, ev_step[p], 0));
        SCG_CUDA_OK(cudaMemcpy2DAsync(h_state2_soa + b0, n, d_new + b0, n, w, 4, cudaMemcpyDeviceToHost, s_out));
        SCG_CUDA_OK(cudaMemcpy2DAsync(h_reward + b0, n, d_out + b0, n, w, 4, cudaMemcpyDeviceToHost, s_out));
    }
    SCG_CUDA_OK(cudaEventRecord(ctx->host_ev, s_out));
    // The results do not depend on the trace sweep: when this step filled the window, the sweep is queued behind the
    // step and the host only waits for the copies, so the sweep overlaps the caller's next host-side work and H2D.
    if (ag->win_len >= ag->win_cap && (rc = scg_agent_flush(ctx, ag, stream))) return rc;
    SCG_CUDA_OK(cudaEventSynchronize(ctx->host_ev));
    return 0;
}

// n_steps steps for a caller that only needs the state every n_steps steps: one host->device copy of state and action,
// the device-resident loop (windows, syncs, exchange), one device->host copy of the results; the loop stays in the library
extern "C" int scg_agent_run_host(const scg_map_t *map, scg_ctx_t *ctx, scg_agent_t *ag, const float *h_state_soa,
                                  const int *h_action, int n_steps, int sync_interval, scg_xchg_t *xchg,
                                  float *h_state2_soa, float *h_reward, int *h_flags, int *h_action2, float *h_delta,
                                  void *stream) {
    if (!map || !ctx || !ag || !h_state_soa || !h_action || !h_state2_soa || !h_reward || !h_flags || !h_action2 ||
        !h_delta || n_steps < 0)
        return SCG_EINVAL;
    cudaStream_t st = (cudaStream_t)stream;
    const size_t n = (size_t)ag->B * sizeof(float);
    int rc;
    {
        void *dst[4] = {ag->x, ag->y, ag->vx, ag->vy};
        const void *src[4] = {h_state_soa, h_state_soa + ag->B, h_state_soa + 2 * (size_t)ag->B, h_state_soa + 3 * (size_t)ag->B};
        if ((rc = copy_rows(dst, src, 4, n, cudaMemcpyHostToDevice, st))) return rc;
    }
    SCG_CUDA_OK(cudaMemcpyAsync(ag->action, h_action, n, cudaMemcpyHostToDevice, st));
    ag->carry_valid = 0;   // state and action came from outside: Q_o(s, a) must be evaluated
    if ((rc = scg_agent_run(map, ctx, ag, n_steps, sync_interval, xchg, stream))) return rc;
    {
        void *dst[4] = {h_state2_soa, h_state2_soa + ag->B, h_state2_soa + 2 * (size_t)ag->B, h_state2_soa + 3 * (size_t)ag->B};
        const void *src[4] = {ag->x, ag->y, ag->vx, ag->vy};
        if ((rc = copy_rows(dst, src, 4, n, cudaMemcpyDeviceToHost, st))) return rc;
    }
    {
        void *dst[4] = {h_reward, h_flags, h_action2, h_delta};
        const void *src[4] = {ag->reward, ag->flags, ag->action, ag->delta};
        if ((rc = copy_rows(dst, src, 4, n, cudaMemcpyDeviceToHost, st))) return rc;
    }
    SCG_CUDA_OK(cudaStreamSynchronize(st));
    return 0;
}

// ---- per-kernel timing ---------------------------------------------------------------------------------
int scg_prof_push(scg_ctx *ctx, int kind, cudaStream_t st, bool end) {
    if (!ctx->prof_on || !((ctx->prof_mask >> kind) & 1)) return 0;
    if (!end) {
        if (ctx->prof_n >= ctx->prof_cap) return 0;
        ctx->prof_kind[ctx->prof_n] = kind;
        SCG_CUDA_OK(cudaEventRecord(ctx->prof_ev[2 * ctx->prof_n], st));
        ctx->prof_open = 1;
    } else if (ctx->prof_open) {
        SCG_CUDA_OK(cudaEventRecord(ctx->prof_ev[2 * ctx->prof_n + 1], st));
        ctx->prof_n += 1;
        ctx->prof_open = 0;
    }
    return 0;
}

extern "C" int scg_profile_begin(scg_ctx_t *ctx, int max_events, int kind_mask) {
    if (!ctx || max_events <= 0) return SCG_EINVAL;
    ctx->prof_mask = kind_mask & ((1 << SCG_PROF_KINDS) - 1);
    if (max_events > ctx->prof_cap) {
        for (int i = 0; i < 2 * ctx->prof_cap; ++i) cudaEventDestroy(ctx->prof_ev[i]);
        free(ctx->prof_ev);
        free(ctx->prof_kind);
        ctx->prof_cap = 0;
        ctx->prof_ev = (cudaEvent_t *)calloc((size_t)2 * max_events, sizeof(cudaEvent_t));
        ctx->prof_kind = (int *)calloc((size_t)max_events, sizeof(int));
        if (!ctx->prof_ev || !ctx->prof_kind) return SCG_ENOMEM;
        for (int i = 0; i < 2 * max_events; ++i) SCG_CUDA_OK(cudaEventCreate(&ctx->prof_ev[i]));
        ctx->prof_cap = max_events;
    }
    ctx->prof_n = 0;
    ctx->prof_open = 0;
    ctx->prof_on = 1;
    return 0;
}

extern "C" int scg_profile_end(scg_ctx_t *ctx, float *ms, int *count) {
    if (!ctx || !ms || !count) return SCG_EINVAL;
    ctx->prof_on = 0;
    for (int k = 0; k < SCG_PROF_KINDS; ++k) { ms[k] = 0.f; count[k] = 0; }
    for (int i = 0; i < ctx->prof_n; ++i) {
        float t = 0.f;
        SCG_CUDA_OK(cudaEventSynchronize(ctx->prof_ev[2 * i + 1]));
        SCG_CUDA_OK(cudaEventElapsedTime(&t, ctx->prof_ev[2 * i], ctx->prof_ev[2 * i + 1]));
        int k = ctx->prof_kind[i] % SCG_PROF_KINDS;
        ms[k] += t;
        count[k] += 1;
    }
    return 0;
}
