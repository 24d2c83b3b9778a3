// scg_step.cuh - device side of the Pinball step, shared by the standalone K1 kernel (scg_step.cu)
// and the fused agent-step kernel (scg_agent.cu).
//
// Semantics follow oracle/pinball.py step_scalar operation for operation: every fp32 +,-,* is an
// explicit round-to-nearest intrinsic so that nvcc cannot contract a*b+c into an FMA and the collision
// decisions, terminal flags and next states are bit-identical to the oracle (SURVEY.md section 7.2-2).
#pragma once
#include "scg_common.cuh"

// ---------------------------------------------------------------------------------------------
// device: TMA bulk staging of the map blob (and of the agent step's weight slots)
// ---------------------------------------------------------------------------------------------
// bulk-TMA staging of up to three global blocks into shared memory behind one mbarrier (blocks 1 and 2 may be empty)
__device__ __forceinline__ void stage3(unsigned char *dst0, const void *src0, int bytes0, unsigned char *dst1,
                                       const void *src1, int bytes1, unsigned char *dst2, const void *src2, int bytes2,
                                       unsigned long long *bar) {
    uint32_t bar_a = scg_smem_u32(bar);
    if (threadIdx.x == 0) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(bar_a));
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar_a),
                     "r"(bytes0 + bytes1 + bytes2)
                     : "memory");
        asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                         scg_smem_u32(dst0)),
                     "l"(src0), "r"(bytes0), "r"(bar_a)
                     : "memory");
        if (bytes1 > 0)
            asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                             scg_smem_u32(dst1)),
                         "l"(src1), "r"(bytes1), "r"(bar_a)
                         : "memory");
        if (bytes2 > 0)
            asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                             scg_smem_u32(dst2)),
                         "l"(src2), "r"(bytes2), "r"(bar_a)
                         : "memory");
    }
    uint32_t ok = 0;
    while (!ok) {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], 0;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(ok)
            : "r"(bar_a)
            : "memory");
    }
}

// ---------------------------------------------------------------------------------------------
// device: the step, shared by scg_step and the fused agent step
// ---------------------------------------------------------------------------------------------
struct StepMap {
    const float4 *ea, *eb;
    const uint32_t *cells;
    const uint16_t *cand;
    int n_edges, G;
    float gf, h, r2, tx, ty, tr2;
};

__device__ __forceinline__ StepMap make_step_map(const unsigned char *blob) {
    const ScgMapHeader *h = reinterpret_cast<const ScgMapHeader *>(blob);
    StepMap m;
    m.ea = reinterpret_cast<const float4 *>(blob + h->off_edges_a);
    m.eb = reinterpret_cast<const float4 *>(blob + h->off_edges_b);
    m.cells = reinterpret_cast<const uint32_t *>(blob + h->off_cells);
    m.cand = reinterpret_cast<const uint16_t *>(blob + h->off_cand);
    m.n_edges = h->n_edges; m.G = h->grid_n; m.gf = h->grid_f;
    m.h = h->h; m.r2 = h->r2; m.tx = h->tx; m.ty = h->ty; m.tr2 = h->tr2;
    return m;
}

__device__ __forceinline__ bool edge_hit(float4 ea, float inv, float x, float y, float vx, float vy, float r2) {
    float rx = __fsub_rn(x, ea.x), ry = __fsub_rn(y, ea.y);
    float t = __fmul_rn(__fadd_rn(__fmul_rn(rx, ea.z), __fmul_rn(ry, ea.w)), inv);
    t = fminf(fmaxf(t, 0.f), 1.f);
    float cx = __fadd_rn(ea.x, __fmul_rn(t, ea.z)), cy = __fadd_rn(ea.y, __fmul_rn(t, ea.w));
    float ex = __fsub_rn(cx, x), ey = __fsub_rn(cy, y);
    float d2 = __fadd_rn(__fmul_rn(ex, ex), __fmul_rn(ey, ey));
    float dot = __fadd_rn(__fmul_rn(ex, vx), __fmul_rn(ey, vy));
    return (d2 <= r2) && (dot > 0.f);
}

__device__ __forceinline__ bool goal_hit(const StepMap &m, float x, float y) {
    float gx = __fsub_rn(x, m.tx), gy = __fsub_rn(y, m.ty);
    return __fadd_rn(__fmul_rn(gx, gx), __fmul_rn(gy, gy)) < m.tr2;
}

// Substeps tested per walk of a cell's candidate list (DESIGN.md section 3, K1: chosen by measurement).
constexpr int kStepChunk = 4;

// The 20 substeps run in chunks.  A chunk takes the next kStepChunk positions as the sequential loop would compute
// them while the velocity stays as it is (x += vx h, one rounding each), keeps the leading ones that lie in the first
// one's broad-phase cell (all of them, almost always: a ball moves at most 0.07 r per substep), loads that cell and
// walks its candidate list once, testing every candidate edge at all of those positions - independent dependency
// chains instead of one per substep.  The substeps before the first one with a hit or a goal are committed as they
// are; that substep then runs the sequential loop's collision response and goal test in the same order, and the
// next chunk starts after it with the new velocity.  So every committed substep sees exactly the position, velocity,
// edge set and goal bit the one-substep-at-a-time loop saw, and the result is the same bit for bit.
template <bool kCull>
__device__ __forceinline__ void pinball_step(const StepMap &m, float &x, float &y, float &vx, float &vy, int a,
                                             float &reward, int &flags) {
    constexpr int C = kStepChunk;
    const float kImpulse = 0.2f;  // fp32(1)/fp32(5)
    if (a == 0) vx = fminf(fmaxf(__fadd_rn(vx, kImpulse), -1.f), 1.f);
    else if (a == 1) vy = fminf(fmaxf(__fadd_rn(vy, kImpulse), -1.f), 1.f);
    else if (a == 2) vx = fminf(fmaxf(__fsub_rn(vx, kImpulse), -1.f), 1.f);
    else if (a == 3) vy = fminf(fmaxf(__fsub_rn(vy, kImpulse), -1.f), 1.f);
    int kind = 0, ids = 0;
    bool done = false;
#pragma unroll 1
    for (int i = 0; i < 20;) {
        const float hx = __fmul_rn(vx, m.h), hy = __fmul_rn(vy, m.h);
        float px[C], py[C];
        int key[C];   // cell of each position, -1 outside the grid (or without culling: every edge is tested)
#pragma unroll
        for (int k = 0; k < C; ++k) {
            px[k] = __fadd_rn(k ? px[k - 1] : x, hx);
            py[k] = __fadd_rn(k ? py[k - 1] : y, hy);
            // floor(x G) is exact (G is a power of two), and 0 <= x < 1 is 0 <= floor(x G) < G
            const int ci = __float2int_rd(px[k] * m.gf), cj = __float2int_rd(py[k] * m.gf);
            key[k] = (kCull && (unsigned)ci < (unsigned)m.G && (unsigned)cj < (unsigned)m.G) ? ci * m.G + cj : -1;
        }
        int n = 1;   // substeps of this chunk: the leading positions in position 0's cell, within the 20 substeps
#pragma unroll
        for (int k = 1; k < C; ++k) n += (n == k && i + k < 20 && key[k] == key[0]) ? 1 : 0;
        const bool in_grid = key[0] >= 0;
        bool goal_near = true;
        int cnt = m.n_edges, start = 0;
        if (in_grid) {
            const uint32_t cell = m.cells[key[0]];
            goal_near = (cell >> 31) != 0u;      // set by scg_map_create where the goal test can succeed
            cnt = cell & 0xFF;
            start = (cell >> 8) & 0x7FFFFF;
        }
        const unsigned live = (1u << n) - 1u;
        // bit k of hit: substep k hits an edge; of multi: it hits two or more.  first: the first edge (lists ascend)
        // that the earliest substep with a hit hits - the only substep whose hits are used.
        unsigned hit = 0u, multi = 0u;
        int first = -1;
#pragma unroll 1   // lists are short (0-4 edges)
        for (int j = 0; j < cnt; ++j) {
            const int e = in_grid ? (int)m.cand[start + j] : j;
            const float4 ea = m.ea[e];
            const float inv = m.eb[e].x;
            unsigned hm = 0u;
#pragma unroll
            for (int k = 0; k < C; ++k) hm |= edge_hit(ea, inv, px[k], py[k], vx, vy, m.r2) ? 1u << k : 0u;
            hm &= live;
            if (hm & ((hit & (0u - hit)) - 1u)) first = e;   // hits a substep before every earlier hit (or is the first)
            multi |= hm & hit;
            hit |= hm;
        }
        unsigned goal = 0u;
        if (goal_near) {
#pragma unroll
            for (int k = 0; k < C; ++k) goal |= goal_hit(m, px[k], py[k]) ? 1u << k : 0u;
            goal &= live;
        }
        // commit up to the first substep with an event, or the whole chunk
        const unsigned ev = hit | goal;
        const int j = ev ? __ffs(ev) - 1 : n - 1;
#pragma unroll
        for (int k = 0; k < C; ++k)
            if (k == j) { x = px[k]; y = py[k]; }
        const int sub = i + j;
        i = sub + 1;
        if (!ev) continue;
        // substep `sub` as the sequential loop runs it: collision response, then the goal test on the new position
        const int nhit = ((hit >> j) & 1u) ? (((multi >> j) & 1u) ? 2 : 1) : 0;
        if (nhit == 1) {
            float4 eb = m.eb[first];
            float k = __fmul_rn(2.0f, __fadd_rn(__fmul_rn(vx, eb.y), __fmul_rn(vy, eb.z)));
            vx = __fsub_rn(vx, __fmul_rn(k, eb.y));
            vy = __fsub_rn(vy, __fmul_rn(k, eb.z));
            kind = 1;
            ids = __float_as_int(eb.w);
            if (sub == 19) {
                x = __fadd_rn(x, __fmul_rn(vx, m.h));
                y = __fadd_rn(y, __fmul_rn(vy, m.h));
            }
        } else if (nhit >= 2) {
            vx = -vx;
            vy = -vy;
            kind = 2;
            ids = __float_as_int(m.eb[first].w);
        }
        if (goal_near && goal_hit(m, x, y)) {
            done = true;
            break;
        }
    }
    if (done) {
        reward = 10000.0f;
    } else {
        vx = __fmul_rn(vx, 0.995f);
        vy = __fmul_rn(vy, 0.995f);
        if (x > 1.f) x = 0.95f;
        if (x < 0.f) x = 0.05f;
        if (y > 1.f) y = 0.95f;
        if (y < 0.f) y = 0.05f;
        reward = (a == 4) ? -1.0f : -5.0f;
    }
    flags = (done ? 1 : 0) | (kind << SCG_FLAG_KIND_SHIFT) | (kind ? (ids << SCG_FLAG_EDGE_SHIFT) : 0);
}

