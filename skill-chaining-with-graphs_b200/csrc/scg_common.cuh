// scg_common.cuh - shared device/host helpers for the sm_100a Pinball / skill-chaining kernels.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/scg_b200.h"

#define SCG_A SCG_N_ACTIONS
#define SCG_WREC_FLOATS 8

// window step record (agent pipeline and scg_sarsa_update), 32 bytes per env-step:
//   [0..3]  x, y, vx, vy of the state the update is for     [4] delta     [5] meta bits     [6],[7] unused
// meta bits: action (bits 0-2), option (bits 8-15), ZERO_AFTER (trace reset after the update), ACTIVE
#define SCG_META_ACTIVE (1u << 31)
#define SCG_META_ZERO_AFTER (1u << 16)
// window records also carry, in floats [6], [7], the position where the executing option started (the example an option
// termination appends to that option's ring); the event byte of a step (win_ev) says whether it terminated:
#define SCG_EV_TERM 0x80u   // the option terminated at this step
#define SCG_EV_HIT 0x40u    // ... by reaching one of its targets (label 1), else label 0
#define SCG_EV_OPT 0x0Fu    // option id
// episode or trajectory log on (scg_agent_t::ev_ep or traj_log set): an episode ended at this step (always also TERM);
// GOAL: it ended at the goal, else it timed out.  With the episode log on its return and length are in the ev_ep plane
#define SCG_EV_EPEND 0x20u
#define SCG_EV_GOAL 0x10u
// option log on (scg_agent_t::ev_opt set): outcome bits of word 2 of a record (option id in bits 0-3), include/scg_b200.h
#define SCG_OL_HIT 0x100u
#define SCG_OL_LABEL 0x200u
#define SCG_OL_ENV_DONE 0x400u
#define SCG_OL_OPTION_TIMEOUT 0x800u
#define SCG_OL_LEFT 0x1000u
#define SCG_OL_EPISODE_TIMEOUT 0x2000u
// trajectory log on (scg_agent_t::traj_log set): flag bits of word 6 of a record (action in bits 0-2, option << 8)
#define SCG_TL_TERM 0x10000u
#define SCG_TL_LABEL 0x20000u
#define SCG_TL_EPEND 0x40000u
#define SCG_TL_GOAL 0x80000u

extern uint64_t g_scg_launches;  // host-side launch counter (scg_api.cu)

#define SCG_CUDA_OK(expr)                      \
    do {                                       \
        cudaError_t _e = (expr);               \
        if (_e != cudaSuccess) return (int)_e; \
    } while (0)

#define SCG_LAUNCH_CHECK()                     \
    do {                                       \
        ++g_scg_launches;                      \
        cudaError_t _e = cudaGetLastError();   \
        if (_e != cudaSuccess) return (int)_e; \
    } while (0)

// run `...` with `constexpr int N1 = order + 1` for the supported orders
#define DISPATCH_ORDER(order, ...)                              \
    switch (order) {                                            \
        case 1: { constexpr int N1 = 2; __VA_ARGS__; } break;   \
        case 2: { constexpr int N1 = 3; __VA_ARGS__; } break;   \
        case 3: { constexpr int N1 = 4; __VA_ARGS__; } break;   \
        case 4: { constexpr int N1 = 5; __VA_ARGS__; } break;   \
        case 5: { constexpr int N1 = 6; __VA_ARGS__; } break;   \
        default: return SCG_ELIMIT;                             \
    }

static inline int scg_pow4(int n1) { return n1 * n1 * n1 * n1; }

#define SCG_MAX_DEVICES 32

// SMs of the current device, read once per device (scg_api.cu); 0 if it cannot be read, and a launch sized from that
// fails its launch check
int scg_num_sms();

// blocks for n items at `threads` per block, at most blocks_per_sm_cap per SM (at least one)
static inline int scg_grid(int n, int threads, int blocks_per_sm_cap) {
    const int blocks = (n + threads - 1) / threads, cap = scg_num_sms() * blocks_per_sm_cap;
    if (cap < 1) return 0;
    return blocks < 1 ? 1 : (blocks < cap ? blocks : cap);
}

// Per-device cache of a kernel's dynamic shared-memory opt-in and occupancy (cudaFuncSetAttribute is per device,
// and one process may drive several devices).
struct ScgKernelCfg {
    size_t configured[SCG_MAX_DEVICES];
    int per_sm[SCG_MAX_DEVICES];
};
template <typename Kern>
static inline int scg_configure(ScgKernelCfg &c, Kern kern, int threads, size_t smem, int *per_sm_out) {
    int dev = 0;
    SCG_CUDA_OK(cudaGetDevice(&dev));
    if (dev < 0 || dev >= SCG_MAX_DEVICES) return SCG_ELIMIT;
    if (smem != c.configured[dev] || c.per_sm[dev] == 0) {
        SCG_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        SCG_CUDA_OK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&c.per_sm[dev], kern, threads, smem));
        c.configured[dev] = smem;
    }
    *per_sm_out = c.per_sm[dev];
    return 0;
}

// ---- map blob ------------------------------------------------------------------------------
// One contiguous, 16-byte aligned block in global memory, bulk-copied into shared memory by the
// step kernel.  Sections (byte offsets in the header):
//   edges_a: float4[E]  (x1, y1, dx, dy)
//   edges_b: float4[E]  (inv_len2, nx, ny, bits(obstacle << 8 | local))
//   cells:   uint32[G*G] (start << 8 | count) into cand
//   cand:    uint16[n_cand] edge indices, ascending within a cell
//   starts:  float2[n_starts]
struct ScgMapHeader {
    int32_t n_edges, grid_n, n_cand, n_starts;
    float ball_r, h, r2, tx;
    float ty, tr2, grid_f, pad0;
    int32_t off_edges_a, off_edges_b, off_cells, off_cand;
    int32_t off_starts, blob_bytes, pad1, pad2;
};
static_assert(sizeof(ScgMapHeader) == 80, "header layout");

struct scg_map {
    ScgMapHeader hdr;
    unsigned char *h_blob;  // host copy
    unsigned char *d_blob;  // device copy
    float *h_edges;         // [E][8] oracle-format table
    int *h_obst, *h_local;  // [E]
    int *h_cell_start;      // [G*G+1]
    int *h_cand;            // [n_cand]
    float *d_stage;         // device staging of scg_step_host (state, action, reward, flags), grown on demand
    size_t stage_cap;
};

// host-mapped mirror of the device controller state (scg_agent_poll): the block and a sequence word that is odd while
// a writer (k_manage's tail, scg_agent_set_ctl) stores the block
struct scg_mirror {
    scg_ctl_t ctl;
    uint32_t seq;
};

#define SCG_HOST_PARTS_MAX 2
struct scg_ctx {
    int order, K, F;
    int n_partials;      // CTAs of the window sweep
    float *d_partial;    // [n_partials][K][A*F]
    float *d_red;        // [SCG_RED_SLICES][K][A*F] second-stage scratch of the slab reduction
    unsigned int *d_tickets;   // one "blocks done" counter per 256-element column of the reduction
    int deterministic;         // 1: fixed-order slab reduction (scg_ctx_set_deterministic)
    unsigned int *d_apply_ticket;   // "blocks done" counter of k_apply, allocated by the first apply
    float *d_rec;        // records for the standalone scg_sarsa_update, grown on demand
    int rec_capacity;
    cudaEvent_t host_ev; // "results copied" marker of scg_agent_step_host
    // scg_agent_step_host pipelines a step over parts of the batch: copies in on host_st[0], copies out on host_st[1]
    cudaStream_t host_st[2];
    cudaEvent_t host_evs[2 * SCG_HOST_PARTS_MAX + 1];   // [part] copied in, [MAX + part] stepped, [2 MAX] entry marker
    // controller (scg_ctl.cu)
    scg_mirror *h_mirror;      // host-mapped mirror of the device controller state, allocated on first use
    scg_mirror *d_mirror;      // its device alias
    uint32_t mirror_seq;       // the even sequence word the last queued write of the mirror leaves behind
    scg_ctl_t ctl_snap;        // the last consistent copy of the mirror scg_agent_poll read
    unsigned int *d_ring;      // scratch of the example-ring pass: per-CTA option counts and the "done" ticket
    // optional per-kernel timing of the agent pipeline (scg_profile_begin / scg_profile_end)
    cudaEvent_t *prof_ev;  // [prof_cap][2] start/stop pairs
    int *prof_kind;        // [prof_cap]
    int prof_cap, prof_n, prof_on, prof_open, prof_mask;
};

#ifdef __CUDACC__
// ---- Philox4x32-10 (matches oracle/philox.py) -------------------------------------------------
__device__ __forceinline__ uint4 scg_philox(uint4 c, uint2 k) {
#pragma unroll
    for (int i = 0; i < 10; ++i) {
        uint32_t hi0 = __umulhi(0xD2511F53u, c.x), lo0 = 0xD2511F53u * c.x;
        uint32_t hi1 = __umulhi(0xCD9E8D57u, c.z), lo1 = 0xCD9E8D57u * c.z;
        c = make_uint4(hi1 ^ c.y ^ k.x, lo1, hi0 ^ c.w ^ k.y, lo0);
        k.x += 0x9E3779B9u;
        k.y += 0xBB67AE85u;
    }
    return c;
}
__device__ __forceinline__ float scg_u01(uint32_t v) { return (float)(v >> 8) * 5.9604644775390625e-08f; }
__device__ __forceinline__ uint4 scg_draw(uint64_t seed, uint32_t env, uint32_t step, uint32_t stream) {
    return scg_philox(make_uint4(env, step, stream, 0u), make_uint2((uint32_t)seed, (uint32_t)(seed >> 32)));
}

// epsilon-greedy (oracle/option.py epsilon_greedy): explore iff u0 < eps, then min(int(u1*5), 4);
// otherwise the first maximal action.
__device__ __forceinline__ int scg_eps_greedy(const float q[SCG_A], float eps, uint4 rnd) {
    int best = 0;
    float bq = q[0];
#pragma unroll
    for (int a = 1; a < SCG_A; ++a)
        if (q[a] > bq) { bq = q[a]; best = a; }
    float u0 = scg_u01(rnd.x), u1 = scg_u01(rnd.y);
    int ra = min((int)__fmul_rn(u1, (float)SCG_A), SCG_A - 1);
    return (u0 < eps) ? ra : best;
}

// ---- packed fp32 pairs ---------------------------------------------------------------------------
// sm_100a has two-wide fp32 instructions (fma / mul / add .f32x2 -> SASS FFMA2 / FMUL2 / FADD2) on 64-bit register
// pairs.  Measured on B200 (tools/probes/ffma2_probe.cu): 117 FMA/clk/SM packed against 73 scalar, and - what matters
// for the issue-bound kernels here - half the instructions for the same arithmetic.  Each half is an ordinary IEEE
// round-to-nearest fp32 operation, so results are bit-identical to the scalar form.
typedef unsigned long long f2_t;   // two fp32: low word = first element
__device__ __forceinline__ f2_t f2_pack(float x, float y) { f2_t r; asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(x), "f"(y)); return r; }
__device__ __forceinline__ f2_t f2_dup(float x) { return f2_pack(x, x); }
__device__ __forceinline__ float f2_x(f2_t v) { return __uint_as_float((uint32_t)v); }
__device__ __forceinline__ float f2_y(f2_t v) { return __uint_as_float((uint32_t)(v >> 32)); }
__device__ __forceinline__ f2_t f2_fma(f2_t a, f2_t b, f2_t c) { f2_t d; asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c)); return d; }
__device__ __forceinline__ f2_t f2_mul(f2_t a, f2_t b) { f2_t d; asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b)); return d; }
__device__ __forceinline__ f2_t f2_add(f2_t a, f2_t b) { f2_t d; asm("add.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b)); return d; }
__device__ __forceinline__ f2_t f2_neg(f2_t a) { return a ^ 0x8000000080000000ull; }

// ---- complex helpers ----------------------------------------------------------------------------
__device__ __forceinline__ float2 scg_cmul(float2 a, float2 b) {
    return make_float2(fmaf(a.x, b.x, -a.y * b.y), fmaf(a.x, b.y, a.y * b.x));
}

// normalised state (oracle/fourier.py FourierBasis.normalise)
__device__ __forceinline__ void scg_normalise(float x, float y, float vx, float vy, float s[4]) {
    s[0] = x;
    s[1] = y;
    s[2] = __fmul_rn(__fadd_rn(vx, 2.0f), 0.25f);
    s[3] = __fmul_rn(__fadd_rn(vy, 2.0f), 0.25f);
}

// z_j = exp(i pi s_hat_j), j = 0..3
__device__ __forceinline__ void scg_phasors(float x, float y, float vx, float vy, float2 z[4]) {
    float s[4];
    scg_normalise(x, y, vx, vy, s);
#pragma unroll
    for (int j = 0; j < 4; ++j) sincospif(s[j], &z[j].y, &z[j].x);
}

// ---- packed weights ------------------------------------------------------------------------------
// Packed weights "Wt": [slot][pair][12] fp32.  A pair is two features that differ only in the last multi-index digit
// (c3 = 2j, 2j + 1; an odd N1 pairs its last feature with a phantom whose weights are 0): 48 bytes
//     (w0a w1a w2a w3a | w0b w1b w2b w3b | w4a w4b 0 0)
// = three 16-byte loads that deliver the register pairs (w0, w1), (w2, w3) of both features and the pair (w4a, w4b) -
// exactly the operands of the two-wide FMAs - 1.5 loads per feature.  Pairs of a slot are contiguous, so every address is
// the slot base plus a constant (no per-feature address arithmetic), a slot is one bulk copy into shared memory, and the
// slot stride is padded to 16 bytes mod 128 so that lanes of a warp on different slots hit different banks.
template <int N1>
struct WtLayout {
    static constexpr int NP = (N1 + 1) / 2;                 // pairs per (c0, c1, c2) row
    static constexpr int P = N1 * N1 * N1 * NP;             // pairs per slot
    static constexpr int RAW = P * 48;
    static constexpr int SLOT_BYTES = RAW + ((16 - RAW % 128) + 128) % 128;
    static constexpr int SLOT_FLOATS = SLOT_BYTES / 4;
    // float offset inside a slot of weight (action a, feature f)
    __host__ __device__ static inline int index(int a, int f) {
        const int row = f / N1, c3 = f - row * N1;
        const int pi = row * NP + (c3 >> 1), h = c3 & 1;
        return pi * 12 + (a < 4 ? h * 4 + a : 8 + h);
    }
};
static inline int scg_wt_slot_floats(int order) {
    switch (order) {
        case 1: return WtLayout<2>::SLOT_FLOATS;
        case 2: return WtLayout<3>::SLOT_FLOATS;
        case 3: return WtLayout<4>::SLOT_FLOATS;
        case 4: return WtLayout<5>::SLOT_FLOATS;
        case 5: return WtLayout<6>::SLOT_FLOATS;
        default: return 0;
    }
}
__device__ __forceinline__ uint32_t scg_smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

// WCur walks one slot of the table, from global memory (read-only path) or from a shared-memory copy.
// load_pair(pi): (w0a, w1a), (w2a, w3a), (w0b, w1b), (w2b, w3b), (w4a, w4b) of pair pi.
template <bool SMEM> struct WCur;
template <> struct WCur<false> {
    const ulonglong2 *p;
    __device__ __forceinline__ WCur(const float *Wt, int slot_floats, int slot)
        : p(reinterpret_cast<const ulonglong2 *>(Wt + (size_t)slot * slot_floats)) {}
    __device__ __forceinline__ void load_pair(int pi, f2_t &a01, f2_t &a23, f2_t &b01, f2_t &b23, f2_t &w4) const {
        const ulonglong2 *q = p + 3 * pi;
        const ulonglong2 u = __ldg(q), v = __ldg(q + 1), w = __ldg(q + 2);
        a01 = u.x; a23 = u.y; b01 = v.x; b23 = v.y; w4 = w.x;
    }
};
template <> struct WCur<true> {
    uint32_t addr;  // bytes
    __device__ __forceinline__ WCur(const float *Wt_smem, int slot_floats, int slot)
        : addr(scg_smem_u32(Wt_smem) + 4u * (uint32_t)slot_floats * (uint32_t)slot) {}
    __device__ __forceinline__ void load_pair(int pi, f2_t &a01, f2_t &a23, f2_t &b01, f2_t &b23, f2_t &w4) const {
        const uint32_t q = addr + 48u * (uint32_t)pi;
        asm("ld.shared.v2.b64 {%0, %1}, [%2];" : "=l"(a01), "=l"(a23) : "r"(q));
        asm("ld.shared.v2.b64 {%0, %1}, [%2+16];" : "=l"(b01), "=l"(b23) : "r"(q));
        asm("ld.shared.b64 %0, [%1+32];" : "=l"(w4) : "r"(q));
    }
};

// ---- Q evaluation on the two-wide fp32 instructions ---------------------------------------------------------
// The step kernel is bound by instruction issue, and most of its Q evaluation is FMAs.  Two features are formed per
// instruction pair (phi = cos01 * cos23 - sin01 * sin23 on packed (c2, c3) table entries, the (c0, c1) phasor as the
// broadcast scalar operand), and the pair's weights are consumed by four FFMA2 with phi_a / phi_b as the broadcast
// operand plus one FFMA2 on (w4a, w4b) x (phi_a, phi_b): 5 issue slots per feature (3 loads, 2 to form phi, 5 FMAs per
// pair) instead of 9 in scalar form.  Accumulators: q01 = (Q0, Q1), q23 = (Q2, Q3), q4 = (even, odd) partial sums of Q4.
struct QAcc {
    f2_t q01, q23, q4;
};
__device__ __forceinline__ void qacc_zero(QAcc &q) { q.q01 = 0ull; q.q23 = 0ull; q.q4 = 0ull; }
__device__ __forceinline__ void qacc_out(const QAcc &q, float out[SCG_A]) {
    out[0] = f2_x(q.q01); out[1] = f2_y(q.q01); out[2] = f2_x(q.q23); out[3] = f2_y(q.q23);
    out[4] = f2_x(q.q4) + f2_y(q.q4);
}
template <bool SMEM>
__device__ __forceinline__ void qacc_pair(const WCur<SMEM> &w, int pi, f2_t ph, QAcc &q) {
    f2_t a01, a23, b01, b23, w4;
    w.load_pair(pi, a01, a23, b01, b23, w4);
    const f2_t pa = f2_dup(f2_x(ph)), pb = f2_dup(f2_y(ph));     // fold into the broadcast-scalar operand form of FFMA2
    q.q01 = f2_fma(a01, pa, q.q01);
    q.q23 = f2_fma(a23, pa, q.q23);
    q.q01 = f2_fma(b01, pb, q.q01);
    q.q23 = f2_fma(b23, pb, q.q23);
    q.q4 = f2_fma(w4, ph, q.q4);
}
// z^c for c = 0 .. N1-1 as packed pairs: xs[i] = (Re z^(2i), Re z^(2i+1)), ys likewise (an odd N1 pads with z^N1)
template <int N1>
__device__ __forceinline__ void pow_pairs(float2 z, f2_t xs[(N1 + 1) / 2], f2_t ys[(N1 + 1) / 2]) {
    float2 p = make_float2(1.f, 0.f);
#pragma unroll
    for (int i = 0; i < (N1 + 1) / 2; ++i) {
        const float2 p1 = scg_cmul(p, z);
        xs[i] = f2_pack(p.x, p1.x);
        ys[i] = f2_pack(p.y, p1.y);
        p = scg_cmul(p1, z);
    }
}
// (phi_a, phi_b) = Re(u * t_a), Re(u * t_b) for the packed table entries (tx, ty) and the phasor u
__device__ __forceinline__ f2_t phi_pair(float2 u, f2_t tx, f2_t ty) {
    return f2_fma(f2_dup(u.x), tx, f2_mul(f2_dup(-u.y), ty));
}

// Q_o(s, .) for one env: nested loops over the multi-index with running phasor products
// (cos(pi c.s) = Re prod_j z_j^{c_j}); the two innermost dimensions are unrolled and use a register
// table of z_3 powers.  Each feature pair is consumed the moment it is formed.
template <int N1, bool SMEM>
__device__ __forceinline__ void scg_q_one(const float2 z[4], const WCur<SMEM> &w, float q[SCG_A]) {
    constexpr int NP = WtLayout<N1>::NP;
    QAcc acc;
    qacc_zero(acc);
    if constexpr (N1 == 2 || N1 == 4) {
        // small even orders: the N1^2 products z_2^c2 z_3^c3 fit in registers (as packed pairs over c3), so a feature
        // pair is one packed multiply-add with the (c0, c1) phasor
        f2_t px[N1 * NP], py[N1 * NP];
        {
            float2 p2 = make_float2(1.f, 0.f);
#pragma unroll
            for (int c2 = 0; c2 < N1; ++c2) {
                float2 v = p2;
#pragma unroll
                for (int j = 0; j < NP; ++j) {
                    const float2 v1 = scg_cmul(v, z[3]);
                    px[c2 * NP + j] = f2_pack(v.x, v1.x);
                    py[c2 * NP + j] = f2_pack(v.y, v1.y);
                    v = scg_cmul(v1, z[3]);
                }
                p2 = scg_cmul(p2, z[2]);
            }
        }
        float2 z0 = make_float2(1.f, 0.f);
        int pi = 0;
#pragma unroll 1
        for (int c0 = 0; c0 < N1; ++c0) {
            float2 z01 = z0;
#pragma unroll 1
            for (int c1 = 0; c1 < N1; ++c1) {
#pragma unroll
                for (int j = 0; j < N1 * NP; ++j) qacc_pair(w, pi + j, phi_pair(z01, px[j], py[j]), acc);
                pi += N1 * NP;
                z01 = scg_cmul(z01, z[1]);
            }
            z0 = scg_cmul(z0, z[0]);
        }
        qacc_out(acc, q);
        return;
    }
    f2_t p3x[NP], p3y[NP];
    pow_pairs<N1>(z[3], p3x, p3y);
    float2 z0 = make_float2(1.f, 0.f);
    int pi = 0;
#pragma unroll 1
    for (int c0 = 0; c0 < N1; ++c0) {
        float2 z01 = z0;
#pragma unroll 1
        for (int c1 = 0; c1 < N1; ++c1) {
            float2 z012 = z01;
#pragma unroll
            for (int c2 = 0; c2 < N1; ++c2) {
#pragma unroll
                for (int j = 0; j < NP; ++j) qacc_pair(w, pi + c2 * NP + j, phi_pair(z012, p3x[j], p3y[j]), acc);
                z012 = scg_cmul(z012, z[2]);
            }
            pi += N1 * NP;
            z01 = scg_cmul(z01, z[1]);
        }
        z0 = scg_cmul(z0, z[0]);
    }
    qacc_out(acc, q);
}

// The slice of Q_o(s, .) whose features have leading multi-index digit c0 (N1^3 features): N1 lanes
// that share one env each take one digit and add their partial sums (option re-selection).
template <int N1, bool SMEM>
__device__ __forceinline__ void scg_q_c0(int c0, const float2 z[4], const WCur<SMEM> &w, float q[SCG_A]) {
    constexpr int NP = WtLayout<N1>::NP;
    f2_t p3x[NP], p3y[NP];
    pow_pairs<N1>(z[3], p3x, p3y);
    QAcc acc;
    qacc_zero(acc);
    float2 z01 = make_float2(1.f, 0.f);
    for (int i = 0; i < c0; ++i) z01 = scg_cmul(z01, z[0]);
    int pi = c0 * N1 * N1 * NP;
#pragma unroll 1
    for (int c1 = 0; c1 < N1; ++c1) {
        float2 z012 = z01;
#pragma unroll
        for (int c2 = 0; c2 < N1; ++c2) {
#pragma unroll
            for (int j = 0; j < NP; ++j) qacc_pair(w, pi + c2 * NP + j, phi_pair(z012, p3x[j], p3y[j]), acc);
            z012 = scg_cmul(z012, z[2]);
        }
        pi += N1 * NP;
        z01 = scg_cmul(z01, z[1]);
    }
    qacc_out(acc, q);
}

// Same for two states sharing the weight loads: qa = Q_o(sa, .), qb = Q_o(sb, .)
template <int N1, bool SMEM>
__device__ __forceinline__ void scg_q_pair(const float2 za[4], const float2 zb[4], const WCur<SMEM> &w,
                                           float qa[SCG_A], float qb[SCG_A]) {
    constexpr int NP = WtLayout<N1>::NP;
    f2_t pax[NP], pay[NP], pbx[NP], pby[NP];
    pow_pairs<N1>(za[3], pax, pay);
    pow_pairs<N1>(zb[3], pbx, pby);
    QAcc A, Bq;
    qacc_zero(A);
    qacc_zero(Bq);
    float2 a0 = make_float2(1.f, 0.f), b0 = a0;
    int pi = 0;
#pragma unroll 1
    for (int c0 = 0; c0 < N1; ++c0) {
        float2 a01 = a0, b01 = b0;
#pragma unroll 1
        for (int c1 = 0; c1 < N1; ++c1) {
            float2 a012 = a01, b012 = b01;
#pragma unroll 1
            for (int c2 = 0; c2 < N1; ++c2) {
#pragma unroll
                for (int j = 0; j < NP; ++j) {
                    const f2_t pa = phi_pair(a012, pax[j], pay[j]);
                    const f2_t pb = phi_pair(b012, pbx[j], pby[j]);
                    f2_t a01w, a23w, b01w, b23w, w4;
                    w.load_pair(pi + j, a01w, a23w, b01w, b23w, w4);
                    const f2_t paa = f2_dup(f2_x(pa)), pab = f2_dup(f2_y(pa));
                    const f2_t pba = f2_dup(f2_x(pb)), pbb = f2_dup(f2_y(pb));
                    A.q01 = f2_fma(a01w, paa, A.q01);
                    A.q23 = f2_fma(a23w, paa, A.q23);
                    A.q01 = f2_fma(b01w, pab, A.q01);
                    A.q23 = f2_fma(b23w, pab, A.q23);
                    A.q4 = f2_fma(w4, pa, A.q4);
                    Bq.q01 = f2_fma(a01w, pba, Bq.q01);
                    Bq.q23 = f2_fma(a23w, pba, Bq.q23);
                    Bq.q01 = f2_fma(b01w, pbb, Bq.q01);
                    Bq.q23 = f2_fma(b23w, pbb, Bq.q23);
                    Bq.q4 = f2_fma(w4, pb, Bq.q4);
                }
                pi += NP;
                a012 = scg_cmul(a012, za[2]);
                b012 = scg_cmul(b012, zb[2]);
            }
            a01 = scg_cmul(a01, za[1]);
            b01 = scg_cmul(b01, zb[1]);
        }
        a0 = scg_cmul(a0, za[0]);
        b0 = scg_cmul(b0, zb[0]);
    }
    qacc_out(A, qa);
    qacc_out(Bq, qb);
}

// initiation bits (oracle/agent.py initiation_bits): bit k iff active and z_k >= 0 (sigmoid(z) >= 0.5  <=>  z >= 0), with
// z_k = theta_k . psi(x, y) formed exactly as oracle/option.py initiation_logit does - fp32, one rounding per operation,
// the same order - so that the decision is bit-identical to the oracle's, also for states on a classifier's boundary.
// th(j) yields theta_j; it is called where theta_j is used, so a loading th interleaves its loads with the arithmetic.
template <typename Th>
__device__ __forceinline__ float scg_init_logit_of(Th th, float x, float y, float xx, float xy, float yy) {
    float z = __fadd_rn(th(0), __fmul_rn(th(1), x));
    z = __fadd_rn(z, __fmul_rn(th(2), y));
    z = __fadd_rn(z, __fmul_rn(th(3), xx));
    z = __fadd_rn(z, __fmul_rn(th(4), xy));
    z = __fadd_rn(z, __fmul_rn(th(5), yy));
    return z;
}
// the same for a classifier in global memory that no thread of the kernel writes (read-only path)
__device__ __forceinline__ float scg_init_logit(const float *__restrict__ t, float x, float y, float xx, float xy, float yy) {
    return scg_init_logit_of([t](int j) { return __ldg(t + j); }, x, y, xx, xy, yy);
}
__device__ __forceinline__ uint32_t scg_init_bits(const float *__restrict__ theta, int K, uint32_t active_mask,
                                                  float x, float y) {
    uint32_t bits = 0;
    const float xx = __fmul_rn(x, x), xy = __fmul_rn(x, y), yy = __fmul_rn(y, y);
    for (int k = 0; k < K; ++k) {
        if (!((active_mask >> k) & 1u)) continue;
        if (scg_init_logit(theta + k * SCG_N_PSI, x, y, xx, xy, yy) >= 0.f) bits |= (1u << k);
    }
    return bits;
}

__device__ __forceinline__ float scg_warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// ---- logistic initiation classifier fit (k_clf_grad / k_clf_fit in scg_q.cu, k_manage in scg_ctl.cu) --------------
// one example's term of the logistic loss gradient: g += (sigmoid(theta . psi) - label) * psi
__device__ __forceinline__ void scg_clf_accum(float px, float py, float lab, const float th[SCG_N_PSI], float g[SCG_N_PSI]) {
    const float psi[SCG_N_PSI] = {1.f, px, py, px * px, px * py, py * py};
    float z = 0.f;
#pragma unroll
    for (int j = 0; j < SCG_N_PSI; ++j) z = fmaf(th[j], psi[j], z);
    const float d = 1.0f / (1.0f + expf(-z)) - lab;
#pragma unroll
    for (int j = 0; j < SCG_N_PSI; ++j) g[j] = fmaf(d, psi[j], g[j]);
}

// The fits run in one CTA.  Each thread keeps up to CLF_CACHE of its examples in registers, so the gradient-descent loop
// touches global memory only for the examples beyond blockDim.x * CLF_CACHE.
#define CLF_CACHE 8
struct ClfCache {
    float x[CLF_CACHE], y[CLF_CACHE], lab[CLF_CACHE];
};
__device__ __forceinline__ void clf_load(int N, const float *__restrict__ X, const uint8_t *__restrict__ y, ClfCache &c) {
#pragma unroll
    for (int k = 0; k < CLF_CACHE; ++k) {
        const int i = threadIdx.x + k * blockDim.x;
        const bool in = i < N;
        c.x[k] = in ? X[2 * i] : 0.f;
        c.y[k] = in ? X[2 * i + 1] : 0.f;
        c.lab[k] = in ? (float)y[i] : 0.f;
    }
}
// sum_i (p_i - y_i) psi_i over the N examples -> g_sum on every thread: per-thread partial sums, warp shuffles, then warp 0
// folds the per-warp sums in warp order.  sm: 33 * SCG_N_PSI floats of shared memory.
__device__ __forceinline__ void clf_grad_sum(int N, const float *__restrict__ X, const uint8_t *__restrict__ y,
                                             const ClfCache &c, const float th[SCG_N_PSI], float g_sum[SCG_N_PSI],
                                             float *sm) {
    float g[SCG_N_PSI] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
#pragma unroll
    for (int k = 0; k < CLF_CACHE; ++k)
        if ((int)(threadIdx.x + k * blockDim.x) < N) scg_clf_accum(c.x[k], c.y[k], c.lab[k], th, g);
    for (int i = threadIdx.x + CLF_CACHE * blockDim.x; i < N; i += blockDim.x)
        scg_clf_accum(X[2 * i], X[2 * i + 1], (float)y[i], th, g);
    int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
#pragma unroll
    for (int j = 0; j < SCG_N_PSI; ++j) {
        float v = scg_warp_sum(g[j]);
        if (lane == 0) sm[warp * SCG_N_PSI + j] = v;
    }
    __syncthreads();
    if (threadIdx.x < 32) {   // warp 0 folds the per-warp sums: lane (w % 32) holds warp w's value of component j
#pragma unroll
        for (int j = 0; j < SCG_N_PSI; ++j) {
            float v = (lane < nw) ? sm[lane * SCG_N_PSI + j] : 0.f;
            v = scg_warp_sum(v);
            if (lane == 0) sm[32 * SCG_N_PSI + j] = v;
        }
    }
    __syncthreads();
#pragma unroll
    for (int j = 0; j < SCG_N_PSI; ++j) g_sum[j] = sm[32 * SCG_N_PSI + j];
    __syncthreads();
}
// one gradient-descent step on the mean gradient g_sum / n
__device__ __forceinline__ void clf_step(float th[SCG_N_PSI], float lr, const float g_sum[SCG_N_PSI], float n) {
#pragma unroll
    for (int j = 0; j < SCG_N_PSI; ++j) th[j] = __fsub_rn(th[j], __fmul_rn(lr, __fdiv_rn(g_sum[j], n)));
}

// ---- weight apply (k_apply in scg_sarsa.cu, k_sync in scg_xchg.cu) -------------------------------------------------
// Element i of W [K][5][F]:  W += (alpha * alpha_scale_f) * (delta * (steps / c))  when its slot's count c > 0;  refresh
// the packed copy Wt;  dW <- 0.  delta is this element of the window's dW (summed over ranks by k_sync).  Slots
// k >= K_opt hold the top-level learner (oracle/option.py): step size alpha_top, mean over the window's events.
template <int N1>
__device__ __forceinline__ void scg_apply_elem(int i, int c, int K_opt, float alpha, float alpha_top, float steps, float delta,
                                               float *W, float *Wt, float *dW) {
    constexpr int F = N1 * N1 * N1 * N1;
    const int f = i % F, ka = i / F, a = ka % SCG_A, k = ka / SCG_A;
    float w = W[i];
    if (c > 0) {
        int d = f, ss = 0;
#pragma unroll
        for (int j = 0; j < 4; ++j) { int q = d % N1; ss += q * q; d /= N1; }
        const float as = (ss == 0) ? 1.0f : (float)(1.0 / sqrt((double)ss));
        const bool top = k >= K_opt;
        const float scale = __fdiv_rn(top ? 1.0f : steps, (float)c);
        w = __fadd_rn(w, __fmul_rn(__fmul_rn(top ? alpha_top : alpha, as), __fmul_rn(delta, scale)));
        W[i] = w;
    }
    Wt[(size_t)k * WtLayout<N1>::SLOT_FLOATS + WtLayout<N1>::index(a, f)] = w;
    dW[i] = 0.f;
}

// True on every thread of the last of the n CTAs sharing `ticket` to get here; every thread of the CTA must call it.
// The CTA's earlier writes are visible grid-wide before the ticket moves.  atomicInc wraps the ticket back to 0 on the
// last CTA, so the same ticket serves the next launch on the same stream.
__device__ __forceinline__ bool scg_last_block(unsigned int *ticket, unsigned int n) {
    __shared__ bool last;
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence();
        last = atomicInc(ticket, n - 1) == n - 1;
    }
    __syncthreads();
    return last;
}
#endif  // __CUDACC__

// the episode log's fields: all off (NULL / 0), or the event plane, the log ring, its count and a capacity all set
static inline bool scg_episode_log_ok(const scg_agent_t *ag) {
    if (!ag->ev_ep && !ag->ep_log) return true;
    return ag->ev_ep && ag->ep_log && ag->ep_log_count && ag->episode_capacity > 0;
}

// the option log's fields: all off (NULL / 0), or the event plane, the log ring, its count and a capacity all set
static inline bool scg_option_log_ok(const scg_agent_t *ag) {
    if (!ag->ev_opt && !ag->opt_log && !ag->opt_log_count && ag->option_capacity == 0) return true;
    return ag->ev_opt && ag->opt_log && ag->opt_log_count && ag->option_capacity > 0;
}

// the trajectory log's fields: all off (NULL / 0), or the tracked envs (1 .. B of them), the log ring, its count and a
// capacity all set; traj_len counts gathered steps of the open window
static inline bool scg_traj_log_ok(const scg_agent_t *ag) {
    if (!ag->traj_env && !ag->traj_log && !ag->traj_log_count && ag->traj_n == 0 && ag->traj_capacity == 0)
        return ag->traj_len == 0;
    return ag->traj_env && ag->traj_log && ag->traj_log_count && ag->traj_n >= 1 && ag->traj_n <= (uint32_t)ag->B &&
           ag->B > 0 && ag->traj_capacity > 0 && ag->traj_len >= 0 && ag->traj_len <= ag->win_len;
}

// the occupancy grid's fields: off (occ_grid = 0, occ_counts NULL), or a power of two <= SCG_OCC_GRID_MAX cells per
// side with the counts set; occ_len counts the open window's steps already added
#define SCG_OCC_GRID_MAX 128u
static inline bool scg_occupancy_ok(const scg_agent_t *ag) {
    if (ag->occ_grid == 0) return !ag->occ_counts && ag->occ_len == 0;
    return ag->occ_counts && ag->occ_grid <= SCG_OCC_GRID_MAX && (ag->occ_grid & (ag->occ_grid - 1)) == 0 &&
           ag->occ_len >= 0 && ag->occ_len <= ag->win_len;
}
