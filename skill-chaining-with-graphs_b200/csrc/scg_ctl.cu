// scg_ctl.cu - the option-creation controller on the device (sm_100a): deterministic example rings and the
// promote-and-fit kernel.
//
// Mirrors oracle/agent.py SkillChainAgent.step item 6 (example ring append) and SkillChainAgent.manage (the reference
// has no code: /root/reference/README.md:1-2).
//
// k_ring_count, k_ring_place
//          The step kernel leaves one event byte per env-step (option terminated? hit? which option) and the option's
//          start position in the step record.  The ring pass turns the events of the steps not yet processed into ring
//          appends in exactly the oracle's order - steps in order, envs in order within a step - so the ring contents
//          (including which examples survive once a ring wraps) do not depend on launch geometry or atomic timing:
//          per-CTA per-option counts (k_ring_count) -> exclusive prefix -> slot = (ex_count + rank) % capacity
//          (k_ring_place, launched after it on the same stream), and only the last `capacity` new examples of an option
//          are written (no two writers per slot).  With the episode log on, episode ends are one more bucket after the 16
//          options: counted, ranked (by a 17th warp) and placed by the same two kernels into the log ring, in the same
//          order and with the same one-writer-per-slot rule.  A byte that is both an example and an episode end is
//          ranked in both buckets.  With the option log on, every termination is a record: its rank is its position in
//          the pass's (step, env) order, which the tile's event list already holds, so it needs no count of its own.
// k_manage One CTA.  Reads the gestating option's success count, and if it qualifies fits its logistic initiation
//          classifier on its ring by batch gradient descent from theta = 0, flips the option to active and wires the
//          next gestating slot's parents - all in device memory, so the agent loop never waits for the host.  Across
//          ranks the per-step gradient sums and example counts travel through NVLink peer memory (one flag round per
//          gradient step) and are added in rank order: every rank ends with the bit-identical theta of one fit on the
//          union of all ranks' examples.
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <atomic>
#include <chrono>
#include <mutex>

#include "scg_common.cuh"
#include "scg_xchg.cuh"

int scg_prof_push(scg_ctx *ctx, int kind, cudaStream_t st, bool end);

#define RING_CTAS 128
#define RING_NT 1024
#define RING_TILE (RING_NT * 4)      // bytes per tile: one 32-bit word per thread, coalesced

// scratch layout (unsigned int): [RING_CTAS][16] per-CTA option counts | [RING_CTAS] per-CTA episode ends | done ticket
#define RING_EP (RING_CTAS * SCG_MAX_OPTIONS)
#define RING_DONE (RING_EP + RING_CTAS)
#define RING_WORDS (RING_DONE + 1)
#define RING_BUCKETS (SCG_MAX_OPTIONS + 1)   // bucket 16: episode ends
// flag bits of an event-list entry next to the option id (bits 0-3) and the byte index (bits 8-19)
#define RING_L_HIT 0x10u
#define RING_L_GOAL 0x20u
#define RING_L_EPEND 0x40u

// exclusive prefix of one value per thread over the CTA (1024 threads); *total receives the sum
__device__ __forceinline__ uint32_t ring_block_scan(uint32_t v, uint32_t *warp_sums, uint32_t *total) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint32_t inc = v;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const uint32_t u = __shfl_up_sync(0xffffffffu, inc, d);
        if (lane >= d) inc += u;
    }
    if (lane == 31) warp_sums[warp] = inc;
    __syncthreads();
    if (warp == 0) {
        const uint32_t w = warp_sums[lane];
        uint32_t winc = w;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const uint32_t u = __shfl_up_sync(0xffffffffu, winc, d);
            if (lane >= d) winc += u;
        }
        warp_sums[lane] = winc - w;
        if (lane == 31) *total = winc;
    }
    __syncthreads();
    return warp_sums[warp] + inc - v;
}

// CTA c of both ring kernels owns the contiguous tiles [c * tiles_per_cta, ...) of the flat [step][env] event-byte array
// (n bytes, read as aligned 32-bit words: the view starts `mis` = ev % 4 bytes early).  ring_word: the word at byte
// offset v0 of that view, bytes outside the events [mis, nv) cleared.
__device__ __forceinline__ uint32_t ring_word(const uint32_t *__restrict__ evw, int mis, long long nv, long long v0) {
    if (v0 >= nv) return 0u;
    uint32_t w = __ldg(evw + (v0 >> 2));
    if (v0 < mis) w &= 0xFFFFFFFFu << (8 * (mis - (int)v0));
    if (v0 + 4 > nv) w &= 0xFFFFFFFFu >> (8 * (int)(v0 + 4 - nv));
    return w;
}

// pass A: this CTA's event count per option -> scratch[blockIdx.x][o], and (ep_on) its episode ends -> scratch[RING_EP + c]
__global__ void __launch_bounds__(RING_NT) k_ring_count(int n, const uint8_t *__restrict__ ev, unsigned int *scratch,
                                                        int tiles_per_cta, int ep_on) {
    __shared__ uint32_t cnt_s[RING_BUCKETS];
    const int tid = threadIdx.x;
    const int mis = (int)(reinterpret_cast<uintptr_t>(ev) & 3);
    const uint32_t *evw = reinterpret_cast<const uint32_t *>(ev - mis);
    const long long nv = (long long)n + mis;
    const long long cta_lo = (long long)blockIdx.x * tiles_per_cta * RING_TILE;
    if (tid < RING_BUCKETS) cnt_s[tid] = 0;
    __syncthreads();
    for (int t = 0; t < tiles_per_cta; ++t) {
        uint32_t w = ring_word(evw, mis, nv, cta_lo + (long long)t * RING_TILE + tid * 4);
        if (ep_on) {
            const uint32_t ne = __reduce_add_sync(0xffffffffu, (uint32_t)__popc(w & 0x20202020u));   // SCG_EV_EPEND bytes
            if ((tid & 31) == 0 && ne) atomicAdd(&cnt_s[SCG_MAX_OPTIONS], ne);
        }
        w &= 0x8F8F8F8Fu;
        while (w & 0x80808080u) {
            const int j = (__ffs(w & 0x80808080u) - 1) >> 3;
            atomicAdd(&cnt_s[(w >> (8 * j)) & SCG_EV_OPT], 1u);
            w &= ~(0xFFu << (8 * j));
        }
    }
    __syncthreads();
    if (tid < SCG_MAX_OPTIONS) scratch[blockIdx.x * SCG_MAX_OPTIONS + tid] = cnt_s[tid];
    if (ep_on && tid == SCG_MAX_OPTIONS) scratch[RING_EP + blockIdx.x] = cnt_s[tid];
}

// where k_ring_place writes the episode log and the option log (ep_log / opt_log NULL: that log is off)
struct RingLogs {
    uint4 *ep_log;              // [ep_cap] records (step, env, return bits, length | goal << 31)
    long long *ep_log_count;
    uint32_t ep_cap;
    const float2 *ev_ep;        // (return, length bits) at the pass's first byte, flat [step][env] like the bytes
    uint4 *opt_log;             // [opt_cap][2] records (step, env, option | outcome, duration), (start x, y, end x, y)
    long long *opt_log_count;
    uint32_t opt_cap;
    const float4 *ev_opt;       // (end x, end y, duration bits, option | outcome) at the pass's first byte, like ev_ep
    uint32_t step0;             // agent step of the pass's first step
    int B;
    uint32_t env_offset;
};

// pass B, on the counts of every CTA that k_ring_count (same grid) left in scratch
__global__ void __launch_bounds__(RING_NT) k_ring_place(int n, int K, const uint8_t *__restrict__ ev, const float2 *__restrict__ pos,
                                                        float *ex_xy, uint8_t *ex_label, long long *ex_count, uint32_t cap,
                                                        unsigned int *scratch, int tiles_per_cta, const RingLogs lg) {
    __shared__ uint32_t lst[RING_TILE];                 // this tile's events in flat order: option | RING_L_* | byte index << 8
    __shared__ uint32_t rk[RING_TILE];                  // their rank among the CTA's events of the same option
    __shared__ uint16_t rke[RING_TILE];                 // episode ends: their rank among this tile's episode ends
    __shared__ uint32_t warp_sums[32];
    __shared__ uint32_t base_s[RING_BUCKETS], tot_s[RING_BUCKETS], run_s[RING_BUCKETS];
    __shared__ uint32_t slot0_s[RING_BUCKETS];
    __shared__ uint32_t n_tile_ev, ep0_s;
    const bool ep_on = lg.ep_log != nullptr;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int mis = (int)(reinterpret_cast<uintptr_t>(ev) & 3);
    const uint32_t *evw = reinterpret_cast<const uint32_t *>(ev - mis);
    const long long nv = (long long)n + mis;
    const long long cta_lo = (long long)blockIdx.x * tiles_per_cta * RING_TILE;
    if (tid < SCG_MAX_OPTIONS) { run_s[tid] = 0; slot0_s[tid] = tid < K ? (uint32_t)((unsigned long long)ex_count[tid] % cap) : 0u; }
    if (ep_on && tid == SCG_MAX_OPTIONS) { run_s[tid] = 0; slot0_s[tid] = (uint32_t)((unsigned long long)*lg.ep_log_count % lg.ep_cap); }
    // option log: its slot of rank 0 (read before this CTA's ticket, like the other counts)
    const bool ol_on = lg.opt_log != nullptr;
    const uint32_t oslot0 = ol_on ? (uint32_t)((unsigned long long)*lg.opt_log_count % lg.opt_cap) : 0u;
    // every CTA's per-option totals: threads (c, o) load them with independent loads, 16 threads form this CTA's bases
    // (and with the log on, thread 16 those of the episode ends, loaded behind them)
    const int n_opt_words = (int)gridDim.x * SCG_MAX_OPTIONS;
    for (int i = tid; i < n_opt_words; i += RING_NT) rk[i] = __ldcg(scratch + i);
    if (ep_on)
        for (int i = tid; i < (int)gridDim.x; i += RING_NT) rk[n_opt_words + i] = __ldcg(scratch + RING_EP + i);
    __syncthreads();
    if (tid < SCG_MAX_OPTIONS || (ep_on && tid == SCG_MAX_OPTIONS)) {
        uint32_t b = 0, tt = 0;
        for (int c = 0; c < (int)gridDim.x; ++c) {
            const uint32_t v = tid < SCG_MAX_OPTIONS ? rk[c * SCG_MAX_OPTIONS + tid] : rk[n_opt_words + c];
            if (c < (int)blockIdx.x) b += v;
            tt += v;
        }
        base_s[tid] = b;
        tot_s[tid] = tt;
    }
    __syncthreads();
    // option log: a termination's rank is the terminations of every option in earlier CTAs (obase), then those of this
    // CTA's earlier tiles (orun), then its index in the tile's list; the pass appends otot of them
    uint32_t obase = 0, otot = 0, orun = 0;
    if (ol_on)
        for (int o = 0; o < SCG_MAX_OPTIONS; ++o) { obase += base_s[o]; otot += tot_s[o]; }
    // per tile, the ordered event list (block scan), per-option ranks (warp o walks the list with ballots), then one
    // thread per event places it.  rank = position among this pass's events of the option in (step, env) order; only
    // the last `cap` of them are written, so every slot has exactly one writer.
    for (int t = 0; t < tiles_per_cta; ++t) {
        const long long v0 = cta_lo + (long long)t * RING_TILE + tid * 4;
        const uint32_t w = ring_word(evw, mis, nv, v0);
        const uint32_t flags = w & 0x80808080u;
        uint32_t total = 0;
        uint32_t off = ring_block_scan(__popc(flags), warp_sums, &n_tile_ev);
        total = n_tile_ev;
        if (flags) {
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const uint32_t e = (w >> (8 * j)) & 0xFFu;
                if (e & SCG_EV_TERM)
                    lst[off++] = (e & SCG_EV_OPT) | ((e & SCG_EV_HIT) ? RING_L_HIT : 0u) | ((e & SCG_EV_GOAL) ? RING_L_GOAL : 0u) |
                                 ((e & SCG_EV_EPEND) ? RING_L_EPEND : 0u) | ((uint32_t)(tid * 4 + j) << 8);
            }
        }
        __syncthreads();
        if (warp < SCG_MAX_OPTIONS && total) {
            uint32_t run = run_s[warp];
            for (uint32_t i0 = 0; i0 < total; i0 += 32) {
                const uint32_t i = i0 + lane;
                const bool m = i < total && (lst[i] & SCG_EV_OPT) == (uint32_t)warp;
                const unsigned bal = __ballot_sync(0xffffffffu, m);
                if (m) rk[i] = run + __popc(bal & ((1u << lane) - 1u));
                run += __popc(bal);
            }
            if (lane == 0) run_s[warp] = run;
        } else if (ep_on && warp == SCG_MAX_OPTIONS && total) {     // the episode ends, ranked within the tile
            uint32_t run = 0;
            for (uint32_t i0 = 0; i0 < total; i0 += 32) {
                const uint32_t i = i0 + lane;
                const bool m = i < total && (lst[i] & RING_L_EPEND);
                const unsigned bal = __ballot_sync(0xffffffffu, m);
                if (m) rke[i] = (uint16_t)(run + __popc(bal & ((1u << lane) - 1u)));
                run += __popc(bal);
            }
            if (lane == 0) { ep0_s = run_s[warp]; run_s[warp] += run; }
        }
        __syncthreads();
        for (uint32_t i = tid; i < total; i += RING_NT) {
            const uint32_t e = lst[i], o = e & SCG_EV_OPT;
            const uint32_t rank = base_s[o] + rk[i];
            if ((int)o < K && (unsigned long long)rank + cap >= tot_s[o]) {
                const uint32_t slot = (uint32_t)(((unsigned long long)slot0_s[o] + rank) % cap);
                const long long f = cta_lo + (long long)t * RING_TILE + (e >> 8) - mis;     // flat [step][env] index
                const size_t ei = (size_t)o * cap + slot;
                *reinterpret_cast<float2 *>(ex_xy + 2 * ei) = __ldg(pos + f);
                ex_label[ei] = (e & RING_L_HIT) ? 1 : 0;
            }
            if (ep_on && (e & RING_L_EPEND)) {
                const uint32_t erank = base_s[SCG_MAX_OPTIONS] + ep0_s + rke[i];
                if ((unsigned long long)erank + lg.ep_cap >= tot_s[SCG_MAX_OPTIONS]) {
                    const uint32_t slot = (uint32_t)(((unsigned long long)slot0_s[SCG_MAX_OPTIONS] + erank) % lg.ep_cap);
                    const long long f = cta_lo + (long long)t * RING_TILE + (e >> 8) - mis;
                    const float2 rl = __ldg(lg.ev_ep + f);
                    lg.ep_log[slot] = make_uint4(lg.step0 + (uint32_t)(f / lg.B), lg.env_offset + (uint32_t)(f % lg.B),
                                                 __float_as_uint(rl.x), __float_as_uint(rl.y) | ((e & RING_L_GOAL) ? 0x80000000u : 0u));
                }
            }
            const uint32_t orank = obase + orun + i;
            if (ol_on && (unsigned long long)orank + lg.opt_cap >= otot) {
                const uint32_t slot = (uint32_t)(((unsigned long long)oslot0 + orank) % lg.opt_cap);
                const long long f = cta_lo + (long long)t * RING_TILE + (e >> 8) - mis;
                const float4 q = __ldg(lg.ev_opt + f);
                const float2 p0 = __ldg(pos + f);
                lg.opt_log[2 * (size_t)slot] = make_uint4(lg.step0 + (uint32_t)(f / lg.B), lg.env_offset + (uint32_t)(f % lg.B),
                                                          __float_as_uint(q.w), __float_as_uint(q.z));
                lg.opt_log[2 * (size_t)slot + 1] = make_uint4(__float_as_uint(p0.x), __float_as_uint(p0.y), __float_as_uint(q.x),
                                                              __float_as_uint(q.y));
            }
        }
        orun += total;
        __syncthreads();
    }
    // the last CTA to finish advances the counts (every CTA has read them by then)
    if (scg_last_block(scratch + RING_DONE, gridDim.x)) {
        if (tid < K) ex_count[tid] += (long long)tot_s[tid];
        if (ep_on && tid == SCG_MAX_OPTIONS) *lg.ep_log_count += (long long)tot_s[tid];
        if (ol_on && tid == 0) *lg.opt_log_count += (long long)otot;
    }
}

extern "C" int scg_agent_ring(scg_ctx_t *ctx, scg_agent_t *ag, void *stream) {
    if (!ctx || !ag) return SCG_EINVAL;
    if (ag->ring_len < 0 || ag->ring_len > ag->ev_len || ag->ev_len > ag->ev_cap) return SCG_EINVAL;
    if (!scg_episode_log_ok(ag) || !scg_option_log_ok(ag)) return SCG_EINVAL;
    const int T = ag->ev_len - ag->ring_len;
    cudaStream_t st = (cudaStream_t)stream;
    if (T > 0 && ag->B > 0) {
        if (!ag->ev_hist || !ag->ev_pos || !ag->ex_xy || !ag->ex_label || !ag->ex_count || ag->example_capacity == 0)
            return SCG_EINVAL;
        if (!ctx->d_ring) {
            SCG_CUDA_OK(cudaMalloc((void **)&ctx->d_ring, RING_WORDS * sizeof(unsigned int)));
            SCG_CUDA_OK(cudaMemsetAsync(ctx->d_ring, 0, RING_WORDS * sizeof(unsigned int), st));
        }
        const long long n = (long long)T * ag->B;
        if (n > 0x7fffffffll) return SCG_ELIMIT;
        const long long n_tiles = (n + 3 + RING_TILE - 1) / RING_TILE;              // (+3: the aligned view may start up to 3 bytes early)
        const int tiles_per_cta = (int)((n_tiles + RING_CTAS - 1) / RING_CTAS);
        const int grid = (int)std::max<long long>(1, (n_tiles + tiles_per_cta - 1) / tiles_per_cta);
        const size_t off = (size_t)ag->ring_len * ag->B;
        int rcp;
        if ((rcp = scg_prof_push(ctx, 4, st, false))) return rcp;
        RingLogs lg = {};
        if (ag->ep_log) {
            lg.ep_log = reinterpret_cast<uint4 *>(ag->ep_log);
            lg.ep_log_count = reinterpret_cast<long long *>(ag->ep_log_count);
            lg.ep_cap = ag->episode_capacity;
            lg.ev_ep = reinterpret_cast<const float2 *>(ag->ev_ep) + off;
        }
        if (ag->opt_log) {
            lg.opt_log = reinterpret_cast<uint4 *>(ag->opt_log);
            lg.opt_log_count = reinterpret_cast<long long *>(ag->opt_log_count);
            lg.opt_cap = ag->option_capacity;
            lg.ev_opt = reinterpret_cast<const float4 *>(ag->ev_opt) + off;
        }
        lg.step0 = ag->step - (uint32_t)ag->ev_len + (uint32_t)ag->ring_len;   // step of history slab ring_len
        lg.B = ag->B;
        lg.env_offset = ag->env_offset;
        k_ring_count<<<grid, RING_NT, 0, st>>>((int)n, ag->ev_hist + off, ctx->d_ring, tiles_per_cta, lg.ep_log != nullptr);
        SCG_LAUNCH_CHECK();
        k_ring_place<<<grid, RING_NT, 0, st>>>((int)n, ag->K, ag->ev_hist + off, reinterpret_cast<const float2 *>(ag->ev_pos) + off,
                                               ag->ex_xy, ag->ex_label, reinterpret_cast<long long *>(ag->ex_count),
                                               ag->example_capacity, ctx->d_ring, tiles_per_cta, lg);
        SCG_LAUNCH_CHECK();
        if ((rcp = scg_prof_push(ctx, 4, st, true))) return rcp;
    }
    ag->ring_len = ag->ev_len;
    // between windows the consumed history is recycled (inside a window its tail still feeds the top-level learner)
    if (ag->win_len == 0) ag->ev_len = ag->ring_len = 0;
    return 0;
}

// ---- the top-level learner's window update --------------------------------------------------------------------------
// Mirrors oracle/option.py OptionSet.top_update.  The step kernel left, for every env-step at which an option terminated
// (event byte), a record (s0, delta_top, option) in win_top.  k_top folds them into the top-level slots of dW:
//     dW[K + o / 5][o % 5][f] += delta_top * phi_f(s0)          and  cnt[K ..] += number of events.
// A CTA walks a contiguous chunk of the event bytes in rounds of TOP_LIST bytes: it scans a round's bytes into a shared
// list of event indices, then processes those events TOP_EB at a time: a few threads build the phasor powers
// exp(i pi c s0_j) of the batch (one sincospi each), then every thread forms its features as products of four table
// entries and accumulates into the CTA's shared-memory copy of the top-level rows, which carries over between rounds;
// one atomicAdd per touched element at the end.  The list bounds the shared memory whatever B * win_len is; a chunk of
// up to TOP_LIST bytes (B * win_len up to about 1.2 M) is one round.
#define TOP_NT 256
#define TOP_EB 8
#define TOP_CTAS 148
#define TOP_LIST 8192

template <int N1>
__global__ void __launch_bounds__(TOP_NT) k_top(int n, int K, int top_slots, const uint8_t *__restrict__ ev,
                                                const float4 *__restrict__ top, float *dW, int *cnt) {
    constexpr int F = N1 * N1 * N1 * N1;
    constexpr int FPT = (F + TOP_NT - 1) / TOP_NT;              // features per thread
    extern __shared__ __align__(16) unsigned char smem_raw[];
    float *acc = reinterpret_cast<float *>(smem_raw);           // [K][F]: row j = option j (slot K + j / 5, row j % 5)
    float2 *tab = reinterpret_cast<float2 *>(acc + (((size_t)K * F + 3) & ~(size_t)3));   // [TOP_EB][4][N1], 16-byte aligned
    float *dl = reinterpret_cast<float *>(tab + TOP_EB * 4 * N1);           // [TOP_EB] delta_top
    int *oo = reinterpret_cast<int *>(dl + TOP_EB);                         // [TOP_EB] option
    int *list = oo + TOP_EB;                                 // [min(chunk, TOP_LIST)] flat indices of a round's events
    __shared__ int n_ev;                                     // events of this CTA so far (all rounds)
    const int tid = threadIdx.x;
    const int chunk = (n + gridDim.x - 1) / gridDim.x;
    const int beg = min(n, (int)blockIdx.x * chunk), end = min(n, beg + chunk);
    for (int i = tid; i < K * F; i += TOP_NT) acc[i] = 0.f;
    if (tid == 0) n_ev = 0;
    __syncthreads();
    // per-thread constants: digits of the owned features, packed 4 x 4 bits
    uint32_t dig[FPT];
#pragma unroll
    for (int k = 0; k < FPT; ++k) {
        int f = tid + k * TOP_NT;
        if (f >= F) f = F - 1;
        const int c3 = f % N1, c2 = (f / N1) % N1, c1 = (f / (N1 * N1)) % N1, c0 = f / (N1 * N1 * N1);
        dig[k] = (uint32_t)c0 | ((uint32_t)c1 << 4) | ((uint32_t)c2 << 8) | ((uint32_t)c3 << 12);
    }
    int seen = 0;                                            // events of the earlier rounds
    for (int r0 = 0; r0 < end - beg; r0 += TOP_LIST) {
        // (after the first round: every thread has read n_ev, and the last batch's barrier has released the list)
        if (r0 > 0) __syncthreads();
        const int rend = beg + min(end - beg, r0 + TOP_LIST);
        for (int i = beg + r0 + tid; i < rend; i += TOP_NT)
            if (ev[i] & SCG_EV_TERM) list[atomicAdd(&n_ev, 1) - seen] = i;
        __syncthreads();
        const int ne = n_ev - seen;
        seen += ne;
        for (int e0 = 0; e0 < ne; e0 += TOP_EB) {
            const int nb = min(TOP_EB, ne - e0);
            if (tid < nb * 4 * N1) {                             // table entry (event, dimension j, power c)
                const int e = tid / (4 * N1), r = tid - e * 4 * N1, j = r / N1, c = r - j * N1;
                const float4 s0 = __ldg(top + (size_t)list[e0 + e] * 2);
                const float raw = j == 0 ? s0.x : (j == 1 ? s0.y : (j == 2 ? s0.z : s0.w));
                const float sh = j < 2 ? raw : __fmul_rn(__fadd_rn(raw, 2.0f), 0.25f);
                float sn, cs;
                sincospif((float)c * sh, &sn, &cs);
                tab[tid] = make_float2(cs, sn);
            }
            if (tid < nb) {
                const float4 r1 = __ldg(top + (size_t)list[e0 + tid] * 2 + 1);
                dl[tid] = r1.x;
                oo[tid] = min(max(__float_as_int(r1.y), 0), K - 1);
            }
            __syncthreads();
            for (int e = 0; e < nb; ++e) {
                const float2 *t = tab + e * 4 * N1;
                const float d = dl[e];
                float *row = acc + (size_t)oo[e] * F;
#pragma unroll
                for (int k = 0; k < FPT; ++k) {
                    const int f = tid + k * TOP_NT;
                    if (f < F) {
                        const float2 p = scg_cmul(scg_cmul(t[dig[k] & 15], t[N1 + ((dig[k] >> 4) & 15)]),
                                                  scg_cmul(t[2 * N1 + ((dig[k] >> 8) & 15)], t[3 * N1 + (dig[k] >> 12)]));
                        row[f] = fmaf(d, p.x, row[f]);
                    }
                }
            }
            __syncthreads();
        }
    }
    if (seen == 0) return;
    for (int i = tid; i < K * F; i += TOP_NT) {
        const float v = acc[i];
        if (v != 0.f) {
            const int j = i / F, f = i - j * F;
            atomicAdd(dW + ((size_t)(K + j / SCG_A) * SCG_A + (j % SCG_A)) * F + f, v);
        }
    }
    if (tid < top_slots) atomicAdd(cnt + K + tid, seen);
}

template <int N1>
static int launch_top(const scg_agent_t *ag, int n, int grid, size_t smem, cudaStream_t st) {
    static ScgKernelCfg cfgc = {};
    int per_sm = 0;
    int rc = scg_configure(cfgc, k_top<N1>, TOP_NT, smem, &per_sm);
    if (rc) return rc;
    k_top<N1><<<grid, TOP_NT, smem, st>>>(n, ag->K, ag->top_slots, ag->ev_hist + (size_t)(ag->ev_len - ag->win_len) * ag->B,
                                          reinterpret_cast<const float4 *>(ag->win_top), ag->dW, ag->cnt);
    SCG_LAUNCH_CHECK();
    return 0;
}

// fold the open window's top-level update records (slabs 0 .. win_len-1) into dW / cnt
int scg_launch_top(scg_ctx *ctx, const scg_agent_t *ag, cudaStream_t st) {
    if (ag->top_slots <= 0 || ag->win_len <= 0 || ag->B <= 0) return 0;
    if (!ag->win_top || !ag->ev_hist || ag->ev_len < ag->win_len) return SCG_EINVAL;
    const long long n = (long long)ag->win_len * ag->B;
    if (n > 0x7fffffffll) return SCG_ELIMIT;
    const int grid = (int)std::max<long long>(1, std::min<long long>(TOP_CTAS, (n + 4095) / 4096));
    const int chunk = (int)((n + grid - 1) / grid);
    const size_t smem = ((((size_t)ag->K * ctx->F + 3) & ~(size_t)3)) * sizeof(float) + (size_t)TOP_EB * 4 * (ctx->order + 1) * sizeof(float2) +
                        TOP_EB * (sizeof(float) + sizeof(int)) + (size_t)std::min(chunk, TOP_LIST) * sizeof(int);
    int rc = 0;
    DISPATCH_ORDER(ctx->order, rc = launch_top<N1>(ag, (int)n, grid, smem, st));
    return rc;
}

// ---- the promote-and-fit kernel ---------------------------------------------------------------------------------
#define MANAGE_NT 1024

struct ManageArgs {
    scg_agent_t ag;
    scg_mirror *mirror;              // host-mapped copy of ctl, written last
    uint32_t mirror_seq;             // the even sequence word the mirror holds after this write
    int world, rank;
    unsigned char *peer[XCHG_MAX_WORLD];
    size_t m_off;
    uint32_t *status;
    long long timeout_cycles;
};

// Sum `nval` (<= XCHG_M_WORDS) per-rank values over the ranks through the peer-memory block: publish, signal every peer,
// wait for every peer, add in rank order (identical on every rank).  vals: shared memory, in/out.  One flag round;
// `seq` is the round counter every rank advances in step.  Returns false (and raises the sticky flag) if a peer never came.
__device__ __forceinline__ bool manage_exchange(const ManageArgs &a, float *vals, int nval, uint32_t &seq, int *s_abort) {
    const int tid = threadIdx.x;
    unsigned char *mine = a.peer[a.rank] + a.m_off;
    seq += 1;
    float *mb = reinterpret_cast<float *>(mine + XCHG_M_BUF) + (seq & 1u) * XCHG_M_WORDS;
    if (tid < nval) mb[tid] = vals[tid];
    __syncthreads();
    if (tid < a.world && tid != a.rank &&
        !xchg_signal_wait(reinterpret_cast<uint32_t *>(a.peer[tid] + a.m_off + XCHG_M_FLAG) + a.rank,
                          reinterpret_cast<const uint32_t *>(mine + XCHG_M_FLAG) + tid, seq, a.status, a.timeout_cycles))
        *s_abort = 1;
    __syncthreads();
    if (tid < nval && !*s_abort) {
        float v = 0.f;
        for (int r = 0; r < a.world; ++r) {
            const float *pb = reinterpret_cast<const float *>(a.peer[r] + a.m_off + XCHG_M_BUF) + (seq & 1u) * XCHG_M_WORDS;
            v += (r == a.rank) ? mb[tid] : ld_sys_f32(pb + tid);
        }
        vals[tid] = v;
    }
    __syncthreads();
    return !*s_abort;
}

__global__ void __launch_bounds__(MANAGE_NT) k_manage(const __grid_constant__ ManageArgs a) {
    __shared__ float sm[33 * SCG_N_PSI];
    __shared__ float xv[XCHG_M_WORDS];           // values summed over ranks: a fit step's (6 sums, N) / the merge counts
    __shared__ int s_go, s_abort;
    const scg_agent_t &g = a.ag;
    scg_ctl_t *ctl = g.ctl;
    const int tid = threadIdx.x, lane = tid & 31;
    const int K = g.K;
    if (tid == 0) {
        const int gi = ctl->n_active;
        int go = 0;
        if (gi < K - 1) {
            // one rank: the live counter; several: the sum over ranks the last exchange left on every GPU
            const long long ns = a.world > 1 ? (long long)g.n_success_global[gi] : (long long)(unsigned int)g.n_success[gi];
            go = ns >= (long long)g.gestation_successes;
        }
        s_go = go;
        s_abort = 0;
    }
    __syncthreads();
    if (s_go) {
        const int gi = ctl->n_active;
        const long long have = g.ex_count[gi];
        const int N = (int)(have < (long long)g.example_capacity ? have : (long long)g.example_capacity);
        const float *X = g.ex_xy + (size_t)gi * g.example_capacity * 2;
        const uint8_t *Y = g.ex_label + (size_t)gi * g.example_capacity;
        ClfCache cache;
        clf_load(N, X, Y, cache);
        float th[SCG_N_PSI] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
        unsigned char *mine = a.world > 1 ? a.peer[a.rank] + a.m_off : nullptr;
        uint32_t seq = (a.world > 1) ? *reinterpret_cast<uint32_t *>(mine + XCHG_M_SEQ) : 0u;
        for (int it = 0; it < g.clf_steps && !s_abort; ++it) {
            float gs[SCG_N_PSI];
            clf_grad_sum(N, X, Y, cache, th, gs, sm);
            float ntot = (float)N;
            if (a.world > 1) {     // the step of one fit on the union of all ranks' rings
                if (tid == 0) {
#pragma unroll
                    for (int j = 0; j < SCG_N_PSI; ++j) xv[j] = gs[j];
                    xv[6] = ntot;
                }
                __syncthreads();
                manage_exchange(a, xv, 7, seq, &s_abort);
#pragma unroll
                for (int j = 0; j < SCG_N_PSI; ++j) gs[j] = xv[j];
                ntot = xv[6];
            }
            // no examples anywhere: theta stays 0 (initiation set = everywhere), as in the oracle
            if (ntot > 0.f) clf_step(th, g.clf_lr, gs, ntot);
        }
        if (!s_abort && tid < SCG_N_PSI) g.theta[gi * SCG_N_PSI + tid] = th[tid];
        __syncthreads();
        // the next gestating slot's targets.  chain: {g}.  graph: {g}, every older option whose initiation set holds at
        // least merge_overlap of g's positive examples, and the goal if it lies inside I_g or merge_overlap is 0
        // (oracle/agent.py merged_parents; merge_overlap = 0: all of them)
        uint32_t pm = 1u << gi;
        if (g.graph && !s_abort) {
            if (tid < XCHG_M_WORDS) xv[tid] = 0.f;
            __syncthreads();
            if (g.merge_overlap > 0.f) {
                // inside-counts of the positive examples, per older option
                for (int j = 0; j < gi; ++j) {
                    float c = 0.f, np = 0.f;
                    for (int i = tid; i < N; i += MANAGE_NT) {
                        if (Y[i]) {
                            const float x = X[2 * i], y = X[2 * i + 1];
                            np += 1.f;
                            if (scg_init_logit(g.theta + j * SCG_N_PSI, x, y, __fmul_rn(x, x), __fmul_rn(x, y), __fmul_rn(y, y)) >= 0.f)
                                c += 1.f;
                        }
                    }
                    c = scg_warp_sum(c);
                    np = scg_warp_sum(np);
                    if (lane == 0) { atomicAdd(&xv[j], c); if (j == 0) atomicAdd(&xv[SCG_MAX_OPTIONS], np); }
                }
                __syncthreads();
                if (a.world > 1) manage_exchange(a, xv, SCG_MAX_OPTIONS + 1, seq, &s_abort);
                const float npos = xv[SCG_MAX_OPTIONS];
                for (int j = 0; j < gi; ++j) {
                    const float frac = npos > 0.f ? __fdiv_rn(xv[j], npos) : 0.f;
                    if (frac >= g.merge_overlap) pm |= 1u << j;
                }
                const float gx = g.goal_x, gy = g.goal_y;
                // theta_gi from the registers that hold the fit (this kernel wrote it: not for the read-only path)
                const float zg = scg_init_logit_of([&](int j) { return th[j]; }, gx, gy, __fmul_rn(gx, gx), __fmul_rn(gx, gy),
                                                   __fmul_rn(gy, gy));
                if (zg >= 0.f) pm |= SCG_GOAL_BIT;
            } else {
                pm = ((1u << (gi + 1)) - 1u) | SCG_GOAL_BIT;
            }
        }
        if (a.world > 1 && tid == 0) *reinterpret_cast<uint32_t *>(mine + XCHG_M_SEQ) = seq;
        if (!s_abort && tid == 0) {
            const int n = gi + 1;
            ctl->parents[n] = pm;
            ctl->active_mask |= (1u << gi);
            ctl->n_promotions += 1;
            ctl->last_promotion_step = g.step;
            __threadfence();
            ctl->n_active = n;
        }
    }
    __syncthreads();
    // host mirror (a seqlock, read by scg_agent_poll): odd sequence word, the block, even sequence word
    volatile uint32_t *seq = &a.mirror->seq;
    if (tid == 0) {
        ctl->manage_calls += 1;
        *seq = a.mirror_seq - 1u;
        __threadfence_system();
    }
    __syncthreads();
    constexpr int NW = (int)(sizeof(scg_ctl_t) / 4);
    const uint32_t *src = reinterpret_cast<const uint32_t *>(ctl);
    volatile uint32_t *dst = reinterpret_cast<volatile uint32_t *>(&a.mirror->ctl);
    if (tid < NW) dst[tid] = src[tid];
    __threadfence_system();
    __syncthreads();
    if (tid == 0) *seq = a.mirror_seq;
}

// guards scg_ctx::ctl_snap: scg_agent_poll may be called from several host threads at once
static std::mutex ctl_snap_mutex;

static int ensure_mirror(scg_ctx *ctx) {
    if (ctx->h_mirror) return 0;
    SCG_CUDA_OK(cudaHostAlloc((void **)&ctx->h_mirror, sizeof(scg_mirror), cudaHostAllocMapped));
    memset(ctx->h_mirror, 0, sizeof(scg_mirror));
    SCG_CUDA_OK(cudaHostGetDevicePointer((void **)&ctx->d_mirror, (void *)ctx->h_mirror, 0));
    return 0;
}

extern "C" int scg_agent_manage(scg_ctx_t *ctx, scg_agent_t *ag, scg_xchg_t *xchg, void *stream) {
    if (!ctx || !ag || !ag->ctl || !ag->theta || !ag->n_success) return SCG_EINVAL;
    if (ag->K + ag->top_slots != ctx->K || ag->K < 1 || ctx->K > SCG_MAX_OPTIONS || ag->clf_steps < 0) return SCG_EINVAL;
    if (xchg && (!ag->n_success_global || xchg->K != ctx->K)) return SCG_EINVAL;
    if (xchg && *xchg->h_status) return SCG_EPEER;
    int rc;
    if ((rc = ensure_mirror(ctx))) return rc;
    if ((rc = scg_agent_ring(ctx, ag, stream))) return rc;    // the rings must hold every example up to this step
    ManageArgs a;
    memset(&a, 0, sizeof(a));
    a.ag = *ag;
    a.mirror = ctx->d_mirror;
    a.mirror_seq = ctx->mirror_seq += 2;
    a.world = xchg ? xchg->world : 1;
    a.rank = xchg ? xchg->rank : 0;
    if (xchg) {
        for (int r = 0; r < xchg->world; ++r) {
            if (!xchg->d_peer[r]) return SCG_EINVAL;
            a.peer[r] = xchg->d_peer[r];
        }
        a.m_off = xchg->m_off;
        a.status = xchg->d_status;
        a.timeout_cycles = xchg->timeout_cycles;
    }
    if ((rc = scg_prof_push(ctx, 5, (cudaStream_t)stream, false))) return rc;
    k_manage<<<1, MANAGE_NT, 0, (cudaStream_t)stream>>>(a);
    SCG_LAUNCH_CHECK();
    if ((rc = scg_prof_push(ctx, 5, (cudaStream_t)stream, true))) return rc;
    if (ctx->deterministic) {   // reproducible runs: the host sizes the next launches with exact knowledge
        SCG_CUDA_OK(cudaStreamSynchronize((cudaStream_t)stream));
        ag->n_active = std::max(ag->n_active, (int)ctx->h_mirror->ctl.n_active);
    }
    return 0;
}

extern "C" int scg_agent_poll(scg_ctx_t *ctx, scg_ctl_t *out) {
    if (!ctx || !out) return SCG_EINVAL;
    int rc = ensure_mirror(ctx);
    if (rc) return rc;
    const volatile uint32_t *seq = &ctx->h_mirror->seq;
    const volatile uint32_t *src = reinterpret_cast<const volatile uint32_t *>(&ctx->h_mirror->ctl);
    // a copy taken while the sequence word stayed the same even value is consistent.  A writer holds the word odd for
    // a few microseconds: retry for up to 1 ms, then fall back to the last consistent copy (a stale copy is a valid
    // lower bound, and a device that stopped in the middle of a write cannot hang the host)
    const auto t_end = std::chrono::steady_clock::now() + std::chrono::milliseconds(1);
    do {
        const uint32_t s0 = *seq;
        if (s0 & 1u) continue;
        std::atomic_thread_fence(std::memory_order_acquire);
        scg_ctl_t c;
        uint32_t *dst = reinterpret_cast<uint32_t *>(&c);
        for (size_t i = 0; i < sizeof(scg_ctl_t) / 4; ++i) dst[i] = src[i];
        std::atomic_thread_fence(std::memory_order_acquire);
        if (*seq == s0) {
            *out = c;
            std::lock_guard<std::mutex> lk(ctl_snap_mutex);
            ctx->ctl_snap = c;
            return 0;
        }
    } while (std::chrono::steady_clock::now() < t_end);
    std::lock_guard<std::mutex> lk(ctl_snap_mutex);
    *out = ctx->ctl_snap;
    return 0;
}

extern "C" int scg_agent_set_ctl(scg_ctx_t *ctx, scg_agent_t *ag, const scg_ctl_t *in, void *stream) {
    if (!ctx || !ag || !ag->ctl || !in) return SCG_EINVAL;
    if (in->n_active < 0 || in->n_active > ag->K - 1 || (in->active_mask >> ag->K) != 0) return SCG_EINVAL;
    int rc = ensure_mirror(ctx);
    if (rc) return rc;
    // staged through the mirror (pinned): the copy is asynchronous and ordered on the stream
    SCG_CUDA_OK(cudaStreamSynchronize((cudaStream_t)stream));   // a manage kernel in flight may still write the mirror
    volatile uint32_t *seq = &ctx->h_mirror->seq;
    *seq = ctx->mirror_seq + 1u;
    std::atomic_thread_fence(std::memory_order_release);
    memcpy(&ctx->h_mirror->ctl, in, sizeof(scg_ctl_t));
    std::atomic_thread_fence(std::memory_order_release);
    *seq = ctx->mirror_seq += 2;
    {
        std::lock_guard<std::mutex> lk(ctl_snap_mutex);
        ctx->ctl_snap = *in;
    }
    SCG_CUDA_OK(cudaMemcpyAsync(ag->ctl, &ctx->h_mirror->ctl, sizeof(scg_ctl_t), cudaMemcpyHostToDevice, (cudaStream_t)stream));
    SCG_CUDA_OK(cudaStreamSynchronize((cudaStream_t)stream));
    ag->n_active = in->n_active;
    return 0;
}
