// scg_sarsa.cu - K3, the Sarsa(lambda) eligibility traces and weight deltas (sm_100a).
//
// Mirrors oracle/option.py OptionSet.flush, OptionSet.update (trace part) and OptionSet.apply.  Three kernels:
//   k_window  the forward-view sweep over a window of T recorded steps: every env's dense trace (A*F fp32, HBM-bound) is
//             read and written once per window, and each CTA accumulates its envs' dW contribution in shared memory
//   k_reduce  folds the per-CTA dW slabs into dW
//   k_apply   W += scaled dW, refreshes the packed copy Wt, zeroes dW and cnt
// The agent pipeline sweeps the windows its step kernel recorded.  The dense per-step operator scg_sarsa_update is the
// same sweep over a window of one step (k_make_rec writes that step's records): with T = 1 the forward view is
//     e_b <- gamma*lambda e_b ;  e_b[a] += phi(s_b) ;  dW[o] += delta_b e_b ;  e_b <- 0 if done_b
#include <stdlib.h>

#include <algorithm>

#include <type_traits>

#include "scg_common.cuh"

template <int VEC> struct VecT;
template <> struct VecT<4> { using type = float4; };
template <> struct VecT<1> { using type = float; };

__device__ __forceinline__ float4 vscale(float4 v, float s) { return make_float4(v.x * s, v.y * s, v.z * s, v.w * s); }
__device__ __forceinline__ float vscale(float v, float s) { return v * s; }
__device__ __forceinline__ float4 vfma(float s, float4 a, float4 c) {
    return make_float4(fmaf(s, a.x, c.x), fmaf(s, a.y, c.y), fmaf(s, a.z, c.z), fmaf(s, a.w, c.w));
}
__device__ __forceinline__ float vfma(float s, float a, float c) { return fmaf(s, a, c); }
__device__ __forceinline__ float4 vzero4() { return make_float4(0.f, 0.f, 0.f, 0.f); }

// ---- windowed (forward-view) sweep: the agent pipeline's K3 --------------------------------------
// Mirrors oracle/option.py OptionSet.flush.  The fused step kernel left, for each of the T steps of the
// window, a 32-byte record per env (state, delta, action / option / termination bits).  One CTA sweeps
// one env at a time; thread t owns the same VEC features of all A rows of every env's trace (registers)
// and of the CTA's dW accumulator (shared memory, [K][A*F], plain read-modify-write: ownership is
// exclusive).  Work items are (env, block of 8 steps); per item:
//   build  the pair tables P01[t][c0][c1] = exp(i pi (c0 s0 + c1 s1)) and P23[t][c2][c3] = exp(i pi (c2 s2 + c3 s3))
//          of the NEXT item, one SFU sincos per entry; for an env's first block a scan warp also runs the backward
//          recursion G_t = delta_t + (done_t ? 0 : gl G_{t+1}), the trace coefficients c_t and (windows of <= 8
//          steps) sorts the contributing steps by (segment, action) into a list
//   main   phi_f = Re(P01[f / N1^2] P23[f % N1^2]);  d[a_t][f] += G_t phi_f;  e[a_t][f] += c_t phi_f
//          with d (the env's dW contribution, seeded with the carry-in gl G_0 e_start) and e in registers;
//          d is added to the shared accumulator once per env (or when the option changes)
// The tables are double-buffered and the records of the following items are prefetched into registers, so there is one
// barrier per item and no phase waits on a load it has just issued.  The next trace is prefetched either into L2 by one
// bulk-prefetch instruction (L2PF: order 3, where the 20 registers it frees buy two more CTAs per SM) or into registers
// (order 5: one CTA per SM, nothing else would cover an L2 hit).  With two warps per env (order 3, SPLIT) warp 0 runs
// the scan and warp 1 builds all the table entries, so neither waits for the other at the barrier; with many warps per
// env (orders 4, 5) an extra warp does nothing but the scan (CTRL).  A feature costs two 8-byte shared loads and two
// FP32 ops to form, and the dense trace crosses HBM once per window: 8*A*F/T + 32 algorithmic bytes per env-step.
#define SCG_WIN_TB 8   // steps per table block

struct WinItem {   // a work item of the sweep: block `blk` of 8 steps of env `b`
    int b, blk;
};

// per-env control block written by the scan warp, read by every thread in the main phase (double-buffered)
template <int NS>                      // NS: steps a window can have (8 for the single-block sweep, SCG_WIN_MAX otherwise)
struct WinCtlT {
    float2 gc[NS];                     // (G_t, c_t) per step
    uint32_t mask[NS][8];              // [segment][action]: steps of that segment taken with that action (5 used)
    uint32_t seg_o[NS];                // option of each segment (an env changes option only after a termination)
    float scale, carry;                // e <- scale * e_start;  d <- carry * e_start
    int nseg, pad;
};

// Single-block sweep (T <= 8): the scan warp sorts the window's steps by (segment, action) into a list, so that the main
// phase walks plain index ranges with static register rows - one broadcast 16-byte load per step carries G_t, c_t and
// the byte offset of the step's tables, and there is no bit-mask bookkeeping in the loop.
struct WinCtlList {
    float4 ent[SCG_WIN_TB + 1];        // (G_t, c_t, byte offset of step t's pair tables, -) in (segment, action, t) order
    uint8_t rng[SCG_WIN_TB][8];        // [segment][action]: first list index of that action's steps; [5] = end
    uint32_t seg_o[SCG_WIN_TB];
    float scale, carry;
    int nseg, pad;
};

// One sweep configuration per order: only what is chosen.  NT work threads; CTRL: one extra warp only runs the per-env
// scan (worth it when a CTA has many work warps: orders 4 and 5); LIST: step lists instead of bit-mask loops; L2PF: the
// next trace is prefetched into L2 instead of registers; SPLIT: two warps per env, one scans, one builds the tables;
// MINB: minimum CTAs per SM (the register budget).  Step lists and split warps are single-block mechanisms: the
// multi-block sweep (T > 8) runs without them.
struct WinCfgBase {
    static constexpr bool CTRL = false, LIST = true, L2PF = false, SPLIT = false;
    static constexpr int MINB = 1;
};
template <int N1_> struct WinCfg;
template <> struct WinCfg<2> : WinCfgBase { static constexpr int N1 = 2, NT = 32; };
template <> struct WinCfg<3> : WinCfgBase { static constexpr int N1 = 3, NT = 96; };
template <> struct WinCfg<5> : WinCfgBase { static constexpr int N1 = 5, NT = 640; };
// Order 3: two warps per env.  With the next trace prefetched into L2 instead of registers the sweep needs 140 registers
// (7 CTAs per SM) and loses nothing when squeezed to 128 (8 CTAs, while 8 accumulators fit: WinCfgO3Split).  With more
// option slots in use (larger accumulators) it runs without the split warps or the squeeze (WinCfg<4>).
struct WinCfgO3Split : WinCfgBase {
    static constexpr int N1 = 4, NT = 64, MINB = 8;
    static constexpr bool L2PF = true, SPLIT = true;
};
template <> struct WinCfg<4> : WinCfgBase {
    static constexpr int N1 = 4, NT = 64;
    static constexpr bool L2PF = true;
};
// Order 5: one CTA per SM, 11 work warps + a scan warp; next trace prefetched in registers (L2 prefetch: 1.98 vs 1.75 ms -
// one CTA cannot cover the L2 latency); bit-mask loop (step lists: 1.74 vs 1.70 ms).
template <> struct WinCfg<6> : WinCfgBase {
    static constexpr int N1 = 6, NT = 352;
    static constexpr bool CTRL = true, LIST = false;
};

// What follows from a configuration: the feature chunking and the sweep's shared memory, in bytes from the start of
// the dynamic block: the accumulator [k_used][A*F] (rounded up to 16 bytes), the two table buffers, the two control
// blocks and glpow[36] (gl^n).  The kernel carves its pointers from it and the host sizes the launch with it.
template <class Cfg, bool MULTI>
struct WinLayout {
    static constexpr int N1 = Cfg::N1, NN = N1 * N1, F = NN * NN, AF = SCG_A * F;
    static constexpr int VEC = N1 % 2 == 0 ? 4 : 1;       // floats per chunk
    static constexpr bool LIST = Cfg::LIST && !MULTI, SPLIT = Cfg::SPLIT && !MULTI;
    using Ctl = std::conditional_t<LIST, WinCtlList, WinCtlT<MULTI ? SCG_WIN_MAX : SCG_WIN_TB>>;
    // Storage of one step's tables, in float2: P01 (NN entries) then P23 in two halves of 16-byte groups (entries
    // (4g, 4g+1) of every group g of four, then entries (4g+2, 4g+3)).  DUP9 (order 5): the 9 groups of a half cannot
    // sit in 8 distinct bank quads, and a quarter-warp reads 8 consecutive groups (mod 9) with one 16-byte load: 7 of 9
    // quarters hit groups 0 and 8 together - two wavefronts (6.4 per load measured).  So a half is 16 slots: groups 0..7,
    // then eight copies of group 8, copy m in the bank quad of group m; the thread that needs group 8 reads the copy in
    // the quad its quarter leaves free.
    static constexpr bool DUP9 = VEC == 4 && NN / 4 == 9;
    static constexpr int HS = DUP9 ? 32 : NN / 2;                 // float2 per half of P23
    static constexpr int TSZ = VEC == 4 ? NN + 2 * HS : 2 * NN;   // float2 per step
    static constexpr int TABS = SCG_WIN_TB * TSZ;                 // float2 per table buffer
    static constexpr int N_TAB = 2 * TABS, N_CTL = 2, N_GLPOW = 36;   // float2, Ctl, float
    __host__ __device__ static constexpr size_t acc_floats(int k_used) { return ((size_t)k_used * AF + 3) & ~(size_t)3; }
    __host__ __device__ static constexpr size_t bytes(int k_used) {
        return acc_floats(k_used) * sizeof(float) + N_TAB * sizeof(float2) + N_CTL * sizeof(Ctl) + N_GLPOW * sizeof(float);
    }
    // option slots whose accumulator stays in shared memory: the most for which the layout fits a CTA's 227 KiB.  Only
    // order 5 holds fewer than SCG_MAX_OPTIONS (8); its spill sweep accumulates the slots beyond in global memory.
    static constexpr int K_SM = [] {
        int k = SCG_MAX_OPTIONS;
        while (k > 1 && bytes(k) > 227 * 1024) --k;
        return k;
    }();
};

// SPILL: more option slots are in use (K) than the shared accumulator holds (L::K_SM).  Slots K_SM .. K-1 accumulate in
// this CTA's own slab rows in global memory, which the reduction reads anyway: the thread that owns a chunk zeroes it,
// adds to it and leaves it there, so each element still has one writer and a fixed order of additions.
template <class Cfg, bool MULTI, bool SPILL>
__global__ void __launch_bounds__(Cfg::NT + (Cfg::CTRL ? 32 : 0), Cfg::MINB)
k_window(int B, int K, int T, const float4 *__restrict__ rec, float *trace, float *__restrict__ partial, float gl,
         float *dW, int K_all) {
    using L = WinLayout<Cfg, MULTI>;
    constexpr int N1 = Cfg::N1, NT = Cfg::NT, VEC = L::VEC, NN = L::NN, F = L::F, AF = L::AF;
    constexpr int HS = L::HS, TSZ = L::TSZ, TABS = L::TABS;
    constexpr bool CTRL = Cfg::CTRL, L2PF = Cfg::L2PF, LIST = L::LIST, SPLIT = L::SPLIT, DUP9 = L::DUP9;
    using V = typename VecT<VEC>::type;
    using WinCtl = typename L::Ctl;
    constexpr int NCHR = F / VEC;          // chunks per action row
    constexpr int TABN = SCG_WIN_TB * 2 * NN;             // entries of one table buffer
    // SPLIT (two warps per env): warp 0 runs the per-env scan, warp 1 builds all the table entries - the two jobs take
    // about as long, so neither warp waits for the other at the per-item barrier.  The 16 state pairs the entries need
    // (8 steps x positions / velocities) are loaded by 16 lanes, one each, and handed round with shuffles.
    static_assert(!Cfg::SPLIT || (!CTRL && NT == 64 && 2 * NN == 32), "split warps: one scan warp and one builder warp");
    constexpr int BT = SPLIT ? 32 : NT;                   // threads that build table entries
    constexpr int EPT = (TABN + BT - 1) / BT;             // table entries built per builder thread
    constexpr int TSTRIDE = TSZ * (int)sizeof(float2);    // bytes between the tables of consecutive steps
    static_assert(F % VEC == 0 && NT >= NCHR && NT >= 32 && SCG_WIN_MAX <= 32, "layout");
    static_assert(VEC == 1 || NN % VEC == 0, "a chunk shares its (c0, c1) digits");
    static_assert(!SPILL || L::K_SM < SCG_MAX_OPTIONS, "a spill sweep only where the slots do not all fit on chip");
    const int KS = SPILL ? L::K_SM : K;                  // option slots accumulated in shared memory
    extern __shared__ __align__(128) unsigned char smem_raw[];
    float *acc = reinterpret_cast<float *>(smem_raw);                                      // [KS][AF]
    float2 *tab = reinterpret_cast<float2 *>(acc + L::acc_floats(KS));                     // [2][TABS]
    WinCtl *ctl = reinterpret_cast<WinCtl *>(tab + L::N_TAB);                              // [2]
    float *glpow = reinterpret_cast<float *>(ctl + L::N_CTL);                              // [N_GLPOW]: gl^n

    const int tid = threadIdx.x;
    // CTRL: the scan warp is threads NT .. NT+31, so that no work warp is slower than the others at the per-env barrier
    constexpr int NTT = NT + (CTRL ? 32 : 0);
    const bool scan_warp = CTRL ? (tid >= NT) : (tid < 32);
    const bool worker = tid < NT;
    const bool builder = SPLIT ? tid >= 32 : worker;
    const int bt = SPLIT ? tid - 32 : tid;                // builder index (SPLIT: lane = half * NN + ij)
    // thread t owns chunk t of every action row (a coalesced access across the CTA)
    const bool own = tid < NCHR;
    const int NBLK = MULTI ? (T + SCG_WIN_TB - 1) / SCG_WIN_TB : 1;
    // per-thread constants: table offsets (bytes) of the owned features' (c0, c1) and (c2, c3) entries ...
    const int f0 = (own ? tid : 0) * VEC;
    const int off01 = (f0 / NN) * (int)sizeof(float2);
    // P23: scalar form one float2 per (c2, c3); vector form: the 16-byte slot of the chunk's group in the first half
    // (the second half is HS float2 further on); DUP9: group 8 is read from the copy in the bank quad that the other
    // seven lanes of this quarter-warp leave free
    int off23;
    if constexpr (VEC == 4) {
        const int c = own ? tid : 0;
        int slot = c % (NN / 4);
        if (DUP9 && slot == 8) slot = 8 + (8 * (c / 8) + 8) % 9;
        off23 = NN * (int)sizeof(float2) + slot * 16;
    } else {
        off23 = (NN + f0 % NN) * (int)sizeof(float2);
    }
    // ... and, for the EPT table entries this thread builds: step within the block, which state pair, digits,
    // the affine map of the raw state pair to [0, 1] (positions: identity; velocities: (v + 2) / 4) folded into the
    // digit coefficients (x = ca s0 + cb s1 + cc on the raw pair), and where the entry goes.
    // REG: the threads of a CTA tile the steps' tables exactly (NT a multiple of the 2 NN entries of a step), so all of
    // this is the same for every entry a thread builds, up to a constant step stride - scalars instead of arrays.
    constexpr bool REG = BT % (2 * NN) == 0 && TABN % BT == 0 && !DUP9;
    constexpr int EN = REG ? 1 : EPT;
    int e_tt[EN], e_half[EN], e_at[EN];
    bool e_dup[EN];                                      // DUP9: an entry of group 8 - stored eight times
    float e_ca[EN], e_cb[EN], e_cc[EN];
#pragma unroll
    for (int k = 0; k < EN; ++k) {
        int idx = (builder ? bt : 0) + k * BT;
        if (idx >= TABN) idx = TABN - 1;                 // duplicate work on the last entry, never out of range
        const int tt = idx / (2 * NN), rem = idx - tt * 2 * NN, half = rem / NN, ij = rem - half * NN;
        e_tt[k] = tt; e_half[k] = half;
        const float mul = half ? 0.25f : 1.f, add = half ? 0.5f : 0.f;
        e_ca[k] = (float)(ij / N1) * mul; e_cb[k] = (float)(ij % N1) * mul;
        e_cc[k] = (float)(ij / N1 + ij % N1) * add;
        int at = tt * TSZ + rem;
        if (VEC == 4 && half) {
            const int g = ij >> 2, kk = ij & 3;
            at = tt * TSZ + NN + (kk >> 1) * HS + 2 * g + (kk & 1);
        }
        e_at[k] = at;
        e_dup[k] = DUP9 && half && (ij >> 2) == 8;
    }
    auto ent_tt = [&](int k) { return REG ? e_tt[0] + k * (BT / (2 * NN)) : e_tt[REG ? 0 : k]; };
    auto ent_at = [&](int k) { return REG ? e_at[0] + k * BT : e_at[REG ? 0 : k]; };
    for (int i = tid; i < KS * AF; i += NTT) acc[i] = 0.f;
    if constexpr (SPILL) {
        if (own) {
            V *sp = reinterpret_cast<V *>(partial + ((size_t)blockIdx.x * K + KS) * AF);
            for (int o = KS; o < K; ++o, sp += SCG_A * NCHR) {
#pragma unroll
                for (int r = 0; r < SCG_A; ++r) {
                    if constexpr (VEC == 4) sp[r * NCHR + tid] = vzero4(); else sp[r * NCHR + tid] = 0.f;
                }
            }
        }
    }
    if (tid == 0) {
        float p = 1.f;
        for (int n = 0; n < L::N_GLPOW; ++n) { glpow[n] = p; p *= gl; }
    }

    const int stride = gridDim.x;
    auto advance = [&](WinItem it) {
        if constexpr (MULTI) {
            if (++it.blk == NBLK) { it.blk = 0; it.b += stride; }
        } else {
            it.b += stride;
        }
        return it;
    };

    // prefetch registers
    float2 r_sv[SPLIT ? 1 : EPT];                        // state pair of the steps this thread builds entries for
    float2 r_dm = make_float2(0.f, 0.f);                 // (delta, meta) of step tid (first block of an env only)
    V e[SCG_A], d[SCG_A];
    V e_nx[L2PF ? 1 : SCG_A];                            // register prefetch of the next env's trace (!L2PF)
    uint32_t o_cur = 0;
#pragma unroll
    for (int r = 0; r < SCG_A; ++r) {
        if constexpr (VEC == 4) { e[r] = vzero4(); d[r] = vzero4(); }
        else { e[r] = 0.f; d[r] = 0.f; }
    }

    auto load_rec = [&](WinItem it) {                    // records of a work item -> registers
        if constexpr (SPLIT) {
            if (tid >= 32 && tid < 32 + 2 * SCG_WIN_TB) {                 // lane l: step l / 2, pair l & 1
                const int t = min((tid - 32) >> 1, T - 1);
                r_sv[0] = __ldg(reinterpret_cast<const float2 *>(rec + ((size_t)t * B + it.b) * 2) + (tid & 1));
            }
        } else if (worker) {
#pragma unroll
            for (int k = 0; k < EPT; ++k) {
                const int t = min(it.blk * SCG_WIN_TB + ent_tt(k), T - 1);
                r_sv[k] = __ldg(reinterpret_cast<const float2 *>(rec + ((size_t)t * B + it.b) * 2) + e_half[REG ? 0 : k]);
            }
        }
        if (it.blk == 0 && scan_warp && (tid & 31) < T)
            r_dm = __ldg(reinterpret_cast<const float2 *>(rec + ((size_t)(tid & 31) * B + it.b) * 2 + 1));
    };
    // The trace of an env is pulled into L2 two items ahead by one bulk-prefetch instruction (no registers, no shared
    // memory); the item itself then loads it straight into the trace registers, an L2 hit whose latency the table build
    // covers.  (Holding the next trace in registers instead cost 20 registers per thread - one CTA per SM at order 3.)
    auto prefetch_trace = [&](int b) {
        constexpr int BYTES = AF * (int)sizeof(float);
        if constexpr (BYTES % 16 == 0) {
            if (tid == NT - 1)
                asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(trace + (size_t)b * AF), "n"(BYTES)
                             : "memory");
        } else {                                         // odd N1: the env's trace is only 4-byte aligned - line by line
            const char *base = reinterpret_cast<const char *>(trace + (size_t)b * AF);
            for (int ofs = tid * 128; ofs < BYTES; ofs += NT * 128)
                asm volatile("prefetch.global.L2 [%0];" ::"l"(base + ofs) : "memory");
        }
    };
    auto load_trace = [&](int b) {
        const V *tp = reinterpret_cast<const V *>(trace + (size_t)b * AF);
        if (own) {
#pragma unroll
            for (int r = 0; r < SCG_A; ++r) {
                if constexpr (L2PF) e[r] = tp[r * NCHR + tid];
                else e_nx[r] = tp[r * NCHR + tid];
            }
        }
    };
    // registers -> pair tables (buffer `par`) and, for an env's first block, its control block (buffer `epar`)
    auto build = [&](WinItem it, int par, int epar) {
        float2 *tb = tab + par * TABS;
        if (builder) {
#pragma unroll
            for (int k = 0; k < EPT; ++k) {
                // exp(i pi x): exact reduction of x to [-1, 1], then the SFU (abs error ~4e-7)
                const int kc = REG ? 0 : k;
                float2 sv;
                if constexpr (SPLIT) {                   // entry k of this lane is step k: its pair sits in lane 2k + half
                    sv.x = __shfl_sync(0xffffffffu, r_sv[0].x, 2 * k + e_half[0]);
                    sv.y = __shfl_sync(0xffffffffu, r_sv[0].y, 2 * k + e_half[0]);
                } else {
                    sv = r_sv[k];
                }
                const float x = fmaf(e_ca[kc], sv.x, fmaf(e_cb[kc], sv.y, e_cc[kc]));
                const float xr = 3.14159265358979f * fmaf(-2.f, rintf(0.5f * x), x);
                if (REG || bt + k * BT < TABN) {
                    const float2 v = make_float2(__cosf(xr), __sinf(xr));
                    tb[ent_at(k)] = v;
                    if constexpr (DUP9) {
                        if (e_dup[kc]) {
#pragma unroll
                            for (int mq = 1; mq < 8; ++mq) tb[ent_at(k) + 2 * mq] = v;
                        }
                    }
                }
            }
        }
        if (it.blk == 0 && scan_warp) {
            // warp 0, lane = step: backward recursion G_t = delta_t + m_t G_{t+1} as a suffix scan over (m, delta)
            // pairs, m_t = 0 after a termination, gl otherwise (1 for a step the env sat out)
            WinCtl &cb = ctl[epar];
            const unsigned FULL = 0xffffffffu;
            const int t = tid & 31;
            const uint32_t meta = (t < T) ? __float_as_uint(r_dm.y) : 0u;
            const bool act = (meta & SCG_META_ACTIVE) != 0;
            const bool dn = act && (meta & SCG_META_ZERO_AFTER);
            const uint32_t a = meta & 7u, o = (meta >> 8) & 0xFFu;
            float D = act ? r_dm.x : 0.f, M = !act ? 1.f : (dn ? 0.f : gl);
#pragma unroll
            for (int off = 1; off < (MULTI ? 32 : SCG_WIN_TB); off <<= 1) {   // T <= 8 steps without MULTI: 3 rounds
                const float D2 = __shfl_down_sync(FULL, D, off), M2 = __shfl_down_sync(FULL, M, off);
                if (t + off < 32) { D = fmaf(M, D2, D); M *= M2; }
            }
            const unsigned am = __ballot_sync(FULL, act), dm = __ballot_sync(FULL, dn);
            const bool dead = (dm >> t) != 0;                     // a termination at this step or later in the window
            const float cf = (act && !dead) ? glpow[__popc((am >> t) >> 1)] : 0.f;
            const float G = act ? D : 0.f;
            // segments: maximal runs of steps under the same option
            const unsigned before = am & ((1u << t) - 1u);
            const int prev = before ? 31 - __clz(before) : t;
            const uint32_t o_prev = __shfl_sync(FULL, o, prev);
            const unsigned chg = __ballot_sync(FULL, act && before && o != o_prev);
            const int seg = __popc(chg & ((2u << t) - 1u));
            const int nseg = am ? __popc(chg) + 1 : 0;
            const bool nz = act && (G != 0.f || cf != 0.f);
            if constexpr (!LIST) {
                if (t < T) cb.gc[t] = make_float2(G, cf);
                for (int sgm = 0; sgm < nseg; ++sgm) {
                    const unsigned in_seg = __ballot_sync(FULL, act && seg == sgm);
                    const uint32_t os = __shfl_sync(FULL, o, __ffs(in_seg) - 1);
                    unsigned mine = 0;
#pragma unroll
                    for (int r = 0; r < SCG_A; ++r) {
                        const unsigned mr = __ballot_sync(FULL, nz && seg == sgm && a == (uint32_t)r);
                        if (t == r) mine = mr;
                    }
                    if (t < SCG_A) cb.mask[sgm][t] = mine;
                    if (t == 0) cb.seg_o[sgm] = os;
                }
            } else {
                // counting sort of the contributing steps by (segment, action, t): segments are runs in time
                uint32_t m[SCG_A], nzm = 0;
#pragma unroll
                for (int r = 0; r < SCG_A; ++r) { m[r] = __ballot_sync(FULL, nz && a == (uint32_t)r); nzm |= m[r]; }
                const unsigned below = (1u << t) - 1u;
                for (int sgm = 0; sgm < nseg; ++sgm) {
                    const unsigned in_seg = __ballot_sync(FULL, act && seg == sgm);
                    const int first = __ffs(in_seg) - 1;
                    const uint32_t os = __shfl_sync(FULL, o, first);
                    const int base = __popc(nzm & ((1u << first) - 1u));
                    int c_lane = base, c_own = base;          // list index where action `t` / this step's action starts
                    uint32_t m_own = 0;
#pragma unroll
                    for (int r = 0; r < SCG_A; ++r) {
                        const int pc = __popc(m[r] & in_seg);
                        if (r < t) c_lane += pc;
                        if ((uint32_t)r < a) c_own += pc;
                        if ((uint32_t)r == a) m_own = m[r];
                    }
                    if (t <= SCG_A) cb.rng[sgm][t] = (uint8_t)c_lane;
                    if (nz && seg == sgm)
                        cb.ent[c_own + __popc(m_own & in_seg & below)] =
                            make_float4(G, cf, __int_as_float(par * TABS * (int)sizeof(float2) + t * TSTRIDE), 0.f);
                    if (t == 0) cb.seg_o[sgm] = os;
                }
            }
            if (t == 0) {
                cb.scale = dm ? 0.f : glpow[__popc(am)];
                cb.carry = am ? gl * D : 0.f;
                cb.nseg = nseg;
            }
        }
    };
    auto flush_d = [&]() {
        if (o_cur >= (uint32_t)K) {
            // an option promoted after the host sized this launch (the accumulator covers options 0 .. K-1 only): its
            // contribution goes straight to dW with atomics (rare and transient; ids beyond K_all are ignored)
            if (o_cur < (uint32_t)K_all) {
                float *gp = dW + (size_t)o_cur * AF;
                if (own) {
#pragma unroll
                    for (int r = 0; r < SCG_A; ++r) {
                        float *q = gp + (size_t)(r * NCHR + tid) * VEC;
                        if constexpr (VEC == 4) {
                            atomicAdd(q, d[r].x); atomicAdd(q + 1, d[r].y);
                            atomicAdd(q + 2, d[r].z); atomicAdd(q + 3, d[r].w);
                        } else {
                            atomicAdd(q, d[r]);
                        }
                    }
                }
            }
            return;
        }
        auto add_d = [&](V *ap) {
            if (own) {
#pragma unroll
                for (int r = 0; r < SCG_A; ++r) {
                    V cur = ap[r * NCHR + tid];
                    if constexpr (VEC == 4) cur = make_float4(cur.x + d[r].x, cur.y + d[r].y, cur.z + d[r].z, cur.w + d[r].w);
                    else cur = cur + d[r];
                    ap[r * NCHR + tid] = cur;
                }
            }
        };
        if constexpr (SPILL) {
            if (o_cur >= (uint32_t)KS) {                 // a slot beyond the shared accumulator: this CTA's slab row
                add_d(reinterpret_cast<V *>(partial + ((size_t)blockIdx.x * K + o_cur) * AF));
                return;
            }
        }
        add_d(reinterpret_cast<V *>(acc + (size_t)o_cur * AF));
    };

    WinItem cur = {(int)blockIdx.x, 0};
    if (cur.b < B) {
        load_rec(cur);
        if constexpr (!L2PF) load_trace(cur.b);
    }
    __syncthreads();                                     // accumulator zeroed, glpow ready
    WinItem nxt = advance(cur);
    if (L2PF && nxt.b < B) prefetch_trace(nxt.b);
    if (cur.b < B) build(cur, 0, 0);
    if (nxt.b < B) load_rec(nxt);
    __syncthreads();

    int par = 0, epar = 0;
    while (cur.b < B) {
        const WinItem nx2 = advance(nxt);
        if constexpr (L2PF) {
            if (cur.blk == 0) load_trace(cur.b);
            if (nx2.blk == 0 && nx2.b < B) prefetch_trace(nx2.b);
        } else if (cur.blk == 0) {
#pragma unroll
            for (int r = 0; r < SCG_A; ++r) e[r] = e_nx[r];
        }
        // next item's tables (into the other buffer), then the loads for the items after it
        if (nxt.b < B) build(nxt, par ^ 1, nxt.blk == 0 ? epar ^ 1 : epar);
        if (nx2.b < B) load_rec(nx2);
        if constexpr (!L2PF) {
            if (nxt.blk == 0 && nxt.b < B) load_trace(nxt.b);
        }
        // ---- main ----
        const WinCtl &cb = ctl[epar];
        const char *tb0 = reinterpret_cast<const char *>(tab + par * TABS);
        [[maybe_unused]] const float2 *gc = nullptr;
        if constexpr (!LIST) gc = cb.gc + cur.blk * SCG_WIN_TB;
        if (cur.blk == 0) {
            const float carry = cb.carry, scale = cb.scale;
            o_cur = cb.seg_o[0];
#pragma unroll
            for (int r = 0; r < SCG_A; ++r) {
                d[r] = vscale(e[r], carry);              // carry-in: gl G_0 e_start
                e[r] = vscale(e[r], scale);
            }
        }
        const int nseg = cb.nseg;
        auto change_option = [&](uint32_t so) {          // the env changed option inside the window (after a termination)
            flush_d();
#pragma unroll
            for (int r = 0; r < SCG_A; ++r) {
                if constexpr (VEC == 4) d[r] = vzero4(); else d[r] = 0.f;
            }
            o_cur = so;
        };
        // one step's contribution to row r of the owned chunk; tb: the step's pair tables
        auto step_row = [&](const char *tb, float G, float c, int r) {
            const float2 p = *reinterpret_cast<const float2 *>(tb + off01);
            V ph;
            if constexpr (VEC == 4) {
                const float4 q01 = *reinterpret_cast<const float4 *>(tb + off23);
                const float4 q23 = *reinterpret_cast<const float4 *>(tb + off23 + HS * (int)sizeof(float2));
                ph = make_float4(fmaf(p.x, q01.x, -p.y * q01.y), fmaf(p.x, q01.z, -p.y * q01.w),
                                 fmaf(p.x, q23.x, -p.y * q23.y), fmaf(p.x, q23.z, -p.y * q23.w));
            } else {
                const float2 q = *reinterpret_cast<const float2 *>(tb + off23);
                ph = fmaf(p.x, q.x, -p.y * q.y);
            }
            d[r] = vfma(G, ph, d[r]);
            e[r] = vfma(c, ph, e[r]);
        };
        if constexpr (LIST) {
            const char *tbase = reinterpret_cast<const char *>(tab);
            for (int sgm = 0; sgm < nseg; ++sgm) {
                const uint2 rr = *reinterpret_cast<const uint2 *>(cb.rng[sgm]);
                int lo = rr.x & 0xFF;
                if (lo == (int)((rr.y >> 8) & 0xFF)) continue;         // no contributing step in this segment
                const uint32_t so = cb.seg_o[sgm];
                if (so != o_cur) change_option(so);
                float4 en = cb.ent[lo];                  // the list is contiguous across the actions: always one ahead
#pragma unroll
                for (int r = 0; r < SCG_A; ++r) {        // static register rows: no dynamic indexing, no switch
                    const int hi = r < 3 ? (rr.x >> (8 * (r + 1))) & 0xFF : (rr.y >> (8 * (r - 3))) & 0xFF;
#pragma unroll 1
                    for (int i = lo; i < hi; ++i) {      // (two steps per trip, to spare the copy: measured equal)
                        const float4 nx = cb.ent[i + 1];
                        step_row(tbase + __float_as_int(en.z), en.x, en.y, r);
                        en = nx;
                    }
                    lo = hi;
                }
            }
        } else {
        for (int sgm = 0; sgm < nseg; ++sgm) {
            // this segment's steps inside this block, one bit mask per action
            uint32_t mk[SCG_A];
            {
                const uint4 m4 = *reinterpret_cast<const uint4 *>(cb.mask[sgm]);
                mk[0] = m4.x; mk[1] = m4.y; mk[2] = m4.z; mk[3] = m4.w; mk[4] = cb.mask[sgm][4];
            }
            uint32_t any = 0;
#pragma unroll
            for (int r = 0; r < SCG_A; ++r) {
                if constexpr (MULTI) mk[r] = (mk[r] >> (cur.blk * SCG_WIN_TB)) & ((1u << SCG_WIN_TB) - 1u);
                any |= mk[r];
            }
            if (!any) continue;
            const uint32_t so = cb.seg_o[sgm];
            if (so != o_cur) change_option(so);
#pragma unroll
            for (int r = 0; r < SCG_A; ++r) {
                uint32_t mm = mk[r];
                while (mm) {
                    const int tt = __ffs(mm) - 1;
                    mm &= mm - 1;
                    const float2 g2 = gc[tt];
                    step_row(tb0 + tt * TSTRIDE, g2.x, g2.y, r);
                }
            }
        }
        }
        if (cur.blk == NBLK - 1) {
            flush_d();
            V *tp = reinterpret_cast<V *>(trace + (size_t)cur.b * AF);
            if (own) {
#pragma unroll
                for (int r = 0; r < SCG_A; ++r) tp[r * NCHR + tid] = e[r];
            }
        }
        __syncthreads();   // the tables just built become readable, the ones just read become writable
        if (nxt.blk == 0) epar ^= 1;
        par ^= 1;
        cur = nxt;
        nxt = nx2;
    }
    float *out = partial + (size_t)blockIdx.x * K * AF;
    for (int i = tid; i < KS * AF; i += NTT) out[i] = acc[i];   // (SPILL: rows KS .. K-1 are already there)
}

// dW[j] += sum over the per-CTA slabs.  Block (x, y) sums every SCG_RED_SLICES-th slab, four loads in flight per thread
// (the slabs were just written and mostly sit in L2).  Fast mode (default): one atomicAdd per address per slice, so the
// order of the last additions is not fixed and weights agree run-to-run to rounding.  Deterministic mode
// (scg_ctx_set_deterministic; 1.3 -> 2.2 us per step at configs[1]): the slice sums go to a small scratch and the last
// block of column x to finish - an integer ticket per column - adds them in a fixed order: same inputs, same bits.
#define SCG_RED_SLICES 96
__global__ void __launch_bounds__(256) k_reduce(int n_partials, int n, const float *__restrict__ partial, float *red,
                                                unsigned int *tickets, float *__restrict__ dW) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    const int gy = gridDim.y;
    float mine = 0.f;
    if (j < n) {
        float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
        int p = blockIdx.y;
        for (; p + 3 * gy < n_partials; p += 4 * gy) {
            s0 += partial[(size_t)p * n + j];
            s1 += partial[(size_t)(p + gy) * n + j];
            s2 += partial[(size_t)(p + 2 * gy) * n + j];
            s3 += partial[(size_t)(p + 3 * gy) * n + j];
        }
        for (; p < n_partials; p += gy) s0 += partial[(size_t)p * n + j];
        mine = (s0 + s1) + (s2 + s3);
    }
    if (!tickets) {                              // fast mode: one atomic per address per slice (order not fixed)
        if (j < n) atomicAdd(dW + j, mine);
        return;                                  // (the whole grid returns here: no CTA is left waiting on a ticket)
    }
    if (j < n) red[(size_t)blockIdx.y * n + j] = mine;
    // the last of the gy CTAs of column x adds the slice sums; the fence orders its reads after the ticket
    if (scg_last_block(tickets + blockIdx.x, gy) && j < n) {
        __threadfence();
        float t0 = 0.f, t1 = 0.f, t2 = 0.f, t3 = 0.f;     // fixed association: four interleaved chains, then a fixed tree
        int y = 0;
        for (; y + 3 < gy; y += 4) {
            t0 += __ldcg(red + (size_t)y * n + j);
            t1 += __ldcg(red + (size_t)(y + 1) * n + j);
            t2 += __ldcg(red + (size_t)(y + 2) * n + j);
            t3 += __ldcg(red + (size_t)(y + 3) * n + j);
        }
        for (; y < gy; ++y) t0 += __ldcg(red + (size_t)y * n + j);
        dW[j] += (t0 + t1) + (t2 + t3);
    }
}

// slabs -> dW on stream st
static int reduce_slabs(scg_ctx *ctx, int n_slabs, int n, float *dW, cudaStream_t st) {
    const int nx_max = (ctx->K * SCG_A * ctx->F + 255) / 256;
    if (ctx->deterministic && !ctx->d_red) {
        SCG_CUDA_OK(cudaMalloc((void **)&ctx->d_red, (size_t)SCG_RED_SLICES * ctx->K * SCG_A * ctx->F * sizeof(float)));
        SCG_CUDA_OK(cudaMalloc((void **)&ctx->d_tickets, (size_t)nx_max * sizeof(unsigned int)));
        SCG_CUDA_OK(cudaMemsetAsync(ctx->d_tickets, 0, (size_t)nx_max * sizeof(unsigned int), st));
    }
    dim3 g((n + 255) / 256, std::min(n_slabs, SCG_RED_SLICES));
    k_reduce<<<g, 256, 0, st>>>(n_slabs, n, ctx->d_partial, ctx->d_red, ctx->deterministic ? ctx->d_tickets : nullptr, dW);
    SCG_LAUNCH_CHECK();
    return 0;
}

// the window records ([1][B][2] float4) of one step of the dense operator scg_sarsa_update, and its cnt increments
__global__ void k_make_rec(int B, const float *__restrict__ x, const float *__restrict__ y,
                           const float *__restrict__ vx, const float *__restrict__ vy, const int *__restrict__ a,
                           const int *__restrict__ option, const float *__restrict__ delta,
                           const uint8_t *__restrict__ done, const uint8_t *__restrict__ mask, int K,
                           float4 *__restrict__ rec, int *__restrict__ cnt) {
    for (int b = blockIdx.x * blockDim.x + threadIdx.x; b < B; b += gridDim.x * blockDim.x) {
        bool act = !mask || mask[b];
        int o = min(max(option[b], 0), K - 1);
        uint32_t meta = (uint32_t)(a[b] & 7) | ((uint32_t)o << 8) | (done[b] ? SCG_META_ZERO_AFTER : 0u) |
                        (act ? SCG_META_ACTIVE : 0u);
        rec[(size_t)b * 2 + 0] = make_float4(x[b], y[b], vx[b], vy[b]);
        rec[(size_t)b * 2 + 1] = make_float4(delta[b], __uint_as_float(meta), 0.f, 0.f);
        if (act) atomicAdd(cnt + o, 1);
    }
}

// W += (alpha * alpha_scale_f) * (dW * (steps / cnt_k));  refresh the packed copy;  dW <- 0  (scg_apply_elem)
template <int N1>
__global__ void k_apply(int K, int K_opt, float *__restrict__ W, float *__restrict__ Wt, float *__restrict__ dW,
                        int *cnt, float alpha, float alpha_top, float steps, unsigned int *ticket) {
    constexpr int F = N1 * N1 * N1 * N1;
    int n = K * SCG_A * F;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x)
        scg_apply_elem<N1>(i, cnt[i / (SCG_A * F)], K_opt, alpha, alpha_top, steps, dW[i], W, Wt, dW);
    // the last block to finish zeroes cnt for the next window (every block has read it by then): no extra launch
    if (scg_last_block(ticket, gridDim.x) && threadIdx.x < K) cnt[threadIdx.x] = 0;
}

// ---- launch plumbing ----------------------------------------------------------------------------
static int ensure_partials(scg_ctx *ctx, int n) {
    if (n <= ctx->n_partials && ctx->d_partial) return 0;
    if (ctx->d_partial) cudaFree(ctx->d_partial);
    ctx->d_partial = nullptr;
    ctx->n_partials = 0;
    size_t slab = (size_t)ctx->K * SCG_A * ctx->F * sizeof(float);
    SCG_CUDA_OK(cudaMalloc((void **)&ctx->d_partial, slab * n));
    ctx->n_partials = n;
    return 0;
}

// bytes of dynamic shared memory the sweep takes (multi: the multi-block sweep of a window longer than 8 steps)
template <class Cfg>
static size_t window_smem(int k_used, bool multi) {
    return multi ? WinLayout<Cfg, true>::bytes(k_used) : WinLayout<Cfg, false>::bytes(k_used);
}

// k_used: options that can appear in the window's records (ids 0 .. k_used-1): the CTA accumulator, the slabs and
// the reduction only cover those, which is what lets two CTAs share an SM at order 5 while the chain is short.  When
// k_used slots do not fit the shared accumulator (order 5, more than 8 slots) the spill sweep keeps the first K_SM on
// chip; the spill variant only exists where SCG_MAX_OPTIONS slots do not fit.
template <class Cfg>
static int launch_window(scg_ctx *ctx, int B, int T, int k_used, const float4 *rec, float *trace, float gl, float *dW,
                         cudaStream_t st) {
    const bool multi = T > SCG_WIN_TB;
    constexpr int KS1 = WinLayout<Cfg, false>::K_SM, KSM = WinLayout<Cfg, true>::K_SM;
    const int k_sm = multi ? KSM : KS1;
    const bool spill = k_used > k_sm;
    const size_t smem = window_smem<Cfg>(std::min(k_used, k_sm), multi);
    auto kern = multi ? (spill ? k_window<Cfg, true, (KSM < SCG_MAX_OPTIONS)> : k_window<Cfg, true, false>)
                      : (spill ? k_window<Cfg, false, (KS1 < SCG_MAX_OPTIONS)> : k_window<Cfg, false, false>);
    constexpr int NTT = Cfg::NT + (Cfg::CTRL ? 32 : 0);
    static ScgKernelCfg cfgc[2][2] = {};
    int per_sm = 0;
    int rcc = scg_configure(cfgc[multi][spill], kern, NTT, smem, &per_sm);
    if (rcc) return rcc;
    if (per_sm < 1) return SCG_ELIMIT;
    int grid = scg_grid(B, 1, per_sm);
    int rc = ensure_partials(ctx, grid);
    if (rc) return rc;
    kern<<<grid, NTT, smem, st>>>(B, k_used, T, rec, trace, ctx->d_partial, gl, dW, ctx->K);
    SCG_LAUNCH_CHECK();
    return grid;
}

int scg_prof_push(scg_ctx *ctx, int kind, cudaStream_t st, bool end);

// fold the T recorded steps of the window into the traces and the per-CTA dW slabs; returns the number of slabs (> 0)
// or an error (<= 0); scg_reduce_window then folds the slabs into dW
int scg_launch_window(scg_ctx *ctx, int B, int T, int k_used, const float *rec, float *trace, float gl, float *dW,
                      cudaStream_t st) {
    if (T < 1 || T > SCG_WIN_MAX || k_used < 1 || k_used > ctx->K) return SCG_EINVAL;
    const float4 *r4 = reinterpret_cast<const float4 *>(rec);
    int grid = 0, rc;
    if ((rc = scg_prof_push(ctx, 1, st, false))) return rc;
    // order 3: the split, squeezed sweep while the shared memory of 8 CTAs (and the 1 KB each reserves) fits an SM
    const bool o3_split = 8 * (window_smem<WinCfgO3Split>(k_used, T > SCG_WIN_TB) + 1024) <= 227 * 1024;
    DISPATCH_ORDER(ctx->order, grid = N1 == 4 && o3_split
                                          ? launch_window<WinCfgO3Split>(ctx, B, T, k_used, r4, trace, gl, dW, st)
                                          : launch_window<WinCfg<N1>>(ctx, B, T, k_used, r4, trace, gl, dW, st));
    if (grid <= 0) return grid == 0 ? SCG_EINVAL : grid;
    if ((rc = scg_prof_push(ctx, 1, st, true))) return rc < 0 ? rc : -rc;
    return grid;
}

int scg_reduce_window(scg_ctx *ctx, int n_slabs, int k_used, float *dW, cudaStream_t st) {
    int rc;
    if ((rc = scg_prof_push(ctx, 2, st, false))) return rc;
    if ((rc = reduce_slabs(ctx, n_slabs, k_used * SCG_A * ctx->F, dW, st))) return rc;
    return scg_prof_push(ctx, 2, st, true);
}

extern "C" int scg_ctx_create(int order, int K, scg_ctx_t **out) {
    if (!out) return SCG_EINVAL;
    if (order < 1 || order > SCG_MAX_ORDER || K < 1 || K > SCG_MAX_OPTIONS) return SCG_ELIMIT;
    scg_ctx *c = (scg_ctx *)calloc(1, sizeof(scg_ctx));
    if (!c) return SCG_ENOMEM;
    c->order = order; c->K = K; c->F = scg_pow4(order + 1);
    // (the dense per-step operator scg_sarsa_update sweeps all K slots, the agent pipeline's sweep only the slots in
    // use; where they do not all fit a CTA's shared accumulator - order 5, more than 8 - the rest accumulate in global
    // memory, so every K <= SCG_MAX_OPTIONS runs at every order)
    *out = c;   // the per-CTA dW slabs are allocated by the first sweep (ensure_partials)
    return 0;
}

extern "C" int scg_ctx_set_deterministic(scg_ctx_t *c, int on) {
    if (!c) return SCG_EINVAL;
    c->deterministic = on ? 1 : 0;
    return 0;
}

extern "C" int scg_ctx_destroy(scg_ctx_t *c) {
    if (!c) return 0;
    if (c->d_partial) cudaFree(c->d_partial);
    if (c->d_rec) cudaFree(c->d_rec);
    if (c->d_red) cudaFree(c->d_red);
    if (c->d_tickets) cudaFree(c->d_tickets);
    if (c->d_apply_ticket) cudaFree(c->d_apply_ticket);
    if (c->host_ev) cudaEventDestroy(c->host_ev);
    for (int i = 0; i < 2; ++i) if (c->host_st[i]) cudaStreamDestroy(c->host_st[i]);
    for (int i = 0; i < 2 * SCG_HOST_PARTS_MAX + 1; ++i) if (c->host_evs[i]) cudaEventDestroy(c->host_evs[i]);
    if (c->h_mirror) cudaFreeHost(c->h_mirror);
    if (c->d_ring) cudaFree(c->d_ring);
    for (int i = 0; i < 2 * c->prof_cap; ++i) cudaEventDestroy(c->prof_ev[i]);
    free(c->prof_ev);
    free(c->prof_kind);
    free(c);
    return 0;
}

extern "C" int scg_sarsa_update(scg_ctx_t *ctx, int B, const float *x, const float *y, const float *vx,
                                const float *vy, const int *a, const int *option, const float *delta,
                                const uint8_t *done, const uint8_t *mask, float gamma_lambda, float *trace, float *dW,
                                int *cnt, void *stream) {
    if (!ctx || B < 0) return SCG_EINVAL;
    if (B == 0) return 0;
    if (!x || !y || !vx || !vy || !a || !option || !delta || !done || !trace || !dW || !cnt) return SCG_EINVAL;
    cudaStream_t st = (cudaStream_t)stream;
    if (B > ctx->rec_capacity) {
        if (ctx->d_rec) cudaFree(ctx->d_rec);
        ctx->d_rec = nullptr; ctx->rec_capacity = 0;
        SCG_CUDA_OK(cudaMalloc((void **)&ctx->d_rec, (size_t)B * SCG_WREC_FLOATS * sizeof(float)));
        ctx->rec_capacity = B;
    }
    k_make_rec<<<scg_grid(B, 256, 8), 256, 0, st>>>(B, x, y, vx, vy, a, option, delta, done, mask, ctx->K,
                                     reinterpret_cast<float4 *>(ctx->d_rec), cnt);
    SCG_LAUNCH_CHECK();
    // the dense update is the forward-view sweep over a window of one step
    const int n = scg_launch_window(ctx, B, 1, ctx->K, ctx->d_rec, trace, gamma_lambda, dW, st);
    if (n <= 0) return n == 0 ? SCG_EINVAL : n;
    return scg_reduce_window(ctx, n, ctx->K, dW, st);
}

extern "C" int scg_apply(scg_ctx_t *ctx, int K_opt, float *W, float *Wt, float *dW, int *cnt, float alpha,
                         float alpha_top, int window_steps, void *stream) {
    if (!ctx || !W || !Wt || !dW || !cnt || K_opt < 0 || K_opt > ctx->K) return SCG_EINVAL;
    cudaStream_t st = (cudaStream_t)stream;
    float steps = (float)std::max(window_steps, 1);
    int grid = scg_grid(ctx->K * SCG_A * ctx->F, 256, 8);
    // the "blocks done" counter: atomicInc wraps it back to 0, so it serves every (stream-ordered) apply on this context
    if (!ctx->d_apply_ticket) {
        SCG_CUDA_OK(cudaMalloc((void **)&ctx->d_apply_ticket, sizeof(unsigned int)));
        SCG_CUDA_OK(cudaMemsetAsync(ctx->d_apply_ticket, 0, sizeof(unsigned int), st));
    }
    DISPATCH_ORDER(ctx->order, k_apply<N1><<<grid, 256, 0, st>>>(ctx->K, K_opt, W, Wt, dW, cnt, alpha, alpha_top, steps,
                                                                 ctx->d_apply_ticket));
    SCG_LAUNCH_CHECK();
    return 0;
}
