// scg_step.cu - map preprocessing (host) and K1, the batched Pinball step kernel (sm_100a).
//
// Semantics follow oracle/pinball.py step_scalar operation for operation: every fp32 +,-,* below
// is an explicit round-to-nearest intrinsic so that nvcc cannot contract a*b+c into an FMA and the
// collision decisions, terminal flags and next states are bit-identical to the oracle
// (SURVEY.md section 7.2-2).  The reference itself has no code (/root/reference/README.md:1-2).
//
// Design: one thread per env, SoA state read/written as coalesced 128-byte warp transactions.
// The whole map (edge table + broad-phase grid) is one blob that each CTA pulls into shared
// memory with a single TMA bulk copy (cp.async.bulk + mbarrier).  The broad phase is a G x G
// uniform grid: each cell lists, in ascending edge order, the edges within ball_r (+ margin) of
// the cell, so a ball only tests the few edges near it; cells in open space test nothing.  The
// lists are conservative, so results equal the oracle's all-edges loop bit for bit.
// Roofline: HBM, 44 algorithmic bytes per env-step (16 in, 16 out, 4 action, 4 reward, 4 flags).
#include <math.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <vector>

#include "scg_common.cuh"
#include "scg_step.cuh"

// ---------------------------------------------------------------------------------------------
// host: map build
// ---------------------------------------------------------------------------------------------
static double seg_point_d(double px, double py, double x1, double y1, double x2, double y2) {
    double dx = x2 - x1, dy = y2 - y1;
    double t = ((px - x1) * dx + (py - y1) * dy) / (dx * dx + dy * dy);
    t = std::min(1.0, std::max(0.0, t));
    return hypot(x1 + t * dx - px, y1 + t * dy - py);
}
static bool seg_seg_intersect(double ax, double ay, double bx, double by, double cx, double cy, double dx,
                              double dy) {
    auto orient = [](double px, double py, double qx, double qy, double rx, double ry) {
        return (qx - px) * (ry - py) - (qy - py) * (rx - px);
    };
    double o1 = orient(ax, ay, bx, by, cx, cy), o2 = orient(ax, ay, bx, by, dx, dy);
    double o3 = orient(cx, cy, dx, dy, ax, ay), o4 = orient(cx, cy, dx, dy, bx, by);
    return ((o1 > 0) != (o2 > 0)) && ((o3 > 0) != (o4 > 0));
}
// distance between a segment and an axis-aligned rectangle (0 when they touch)
static double seg_rect_d(double x1, double y1, double x2, double y2, double rx0, double ry0, double rx1,
                         double ry1) {
    auto inside = [&](double px, double py) { return px >= rx0 && px <= rx1 && py >= ry0 && py <= ry1; };
    if (inside(x1, y1) || inside(x2, y2)) return 0.0;
    const double cx[4] = {rx0, rx1, rx1, rx0}, cy[4] = {ry0, ry0, ry1, ry1};
    double d = 1e30;
    for (int i = 0; i < 4; ++i) {
        int j = (i + 1) & 3;
        if (seg_seg_intersect(x1, y1, x2, y2, cx[i], cy[i], cx[j], cy[j])) return 0.0;
        d = std::min(d, seg_point_d(cx[i], cy[i], x1, y1, x2, y2));
        d = std::min(d, seg_point_d(x1, y1, cx[i], cy[i], cx[j], cy[j]));
        d = std::min(d, seg_point_d(x2, y2, cx[i], cy[i], cx[j], cy[j]));
    }
    return d;
}

static int align16(int v) { return (v + 15) & ~15; }

extern "C" int scg_map_create(const float *verts, const int *poly_start, int n_poly, float ball_r, float tx,
                              float ty, float tr, const float *starts, int n_starts, int grid_n,
                              scg_map_t **out) {
    if (!verts || !poly_start || !out || n_poly <= 0 || n_starts <= 0 || !starts) return SCG_EINVAL;
    if (!(ball_r > 0.f) || !(tr > 0.f)) return SCG_EINVAL;
    if (grid_n == 0) grid_n = 64;
    if (grid_n < 1 || grid_n > 128 || (grid_n & (grid_n - 1))) return SCG_EINVAL;
    if (n_poly > 4095) return SCG_ELIMIT;
    int E = 0;
    for (int p = 0; p < n_poly; ++p) {
        int n = poly_start[p + 1] - poly_start[p];
        if (n < 3) return SCG_EINVAL;
        if (n > 255) return SCG_ELIMIT;
        E += n;
    }
    if (E > 4096) return SCG_ELIMIT;

    scg_map *m = (scg_map *)calloc(1, sizeof(scg_map));
    if (!m) return SCG_ENOMEM;
    m->h_edges = (float *)calloc((size_t)E * 8, sizeof(float));
    m->h_obst = (int *)calloc(E, sizeof(int));
    m->h_local = (int *)calloc(E, sizeof(int));
    // edge table: same fp32 operations, same order as oracle/pinball.py PinballMap.__init__
    int e = 0;
    for (int p = 0; p < n_poly; ++p) {
        int s = poly_start[p], n = poly_start[p + 1] - s;
        for (int j = 0; j < n; ++j, ++e) {
            float x1 = verts[2 * (s + j)], y1 = verts[2 * (s + j) + 1];
            float x2 = verts[2 * (s + (j + 1) % n)], y2 = verts[2 * (s + (j + 1) % n) + 1];
            volatile float dx = x2 - x1, dy = y2 - y1;
            volatile float dxx = dx * dx, dyy = dy * dy;
            volatile float len2 = dxx + dyy;
            if (!(len2 > 0.f)) {
                scg_map_destroy(m);
                return SCG_EINVAL;
            }
            volatile float inv = 1.0f / len2;
            volatile float ln = sqrtf(len2);
            volatile float nx = dy / ln;
            volatile float ndx = 0.0f - dx;
            volatile float ny = ndx / ln;
            float *row = m->h_edges + 8 * e;
            row[0] = x1; row[1] = y1; row[2] = dx; row[3] = dy;
            row[4] = inv; row[5] = nx; row[6] = ny; row[7] = 0.f;
            m->h_obst[e] = p;
            m->h_local[e] = j;
        }
    }
    // broad-phase grid (fp64 geometry; conservative by `margin`)
    const int G = grid_n;
    const double reach = (double)ball_r * 1.02 + 1e-5;
    std::vector<std::vector<int>> lists((size_t)G * G);
    for (int ed = 0; ed < E; ++ed) {
        const float *row = m->h_edges + 8 * ed;
        double x1 = row[0], y1 = row[1], x2 = (double)row[0] + (double)row[2], y2 = (double)row[1] + (double)row[3];
        // vertices as the kernel sees them are x1 + t*dx in fp32; cover both the fp32 and exact end points
        int i0 = std::max(0, (int)floor((std::min(x1, x2) - reach) * G) - 1);
        int i1 = std::min(G - 1, (int)floor((std::max(x1, x2) + reach) * G) + 1);
        int j0 = std::max(0, (int)floor((std::min(y1, y2) - reach) * G) - 1);
        int j1 = std::min(G - 1, (int)floor((std::max(y1, y2) + reach) * G) + 1);
        for (int i = i0; i <= i1; ++i)
            for (int j = j0; j <= j1; ++j) {
                double d = seg_rect_d(x1, y1, x2, y2, (double)i / G, (double)j / G, (double)(i + 1) / G,
                                      (double)(j + 1) / G);
                if (d <= reach) lists[(size_t)i * G + j].push_back(ed);
            }
    }
    int n_cand = 0;
    for (auto &l : lists) {
        if (l.size() > 255) {
            scg_map_destroy(m);
            return SCG_ELIMIT;
        }
        n_cand += (int)l.size();
    }
    if (n_cand >= (1 << 23)) {
        scg_map_destroy(m);
        return SCG_ELIMIT;
    }
    m->h_cell_start = (int *)calloc((size_t)G * G + 1, sizeof(int));
    m->h_cand = (int *)calloc(std::max(n_cand, 1), sizeof(int));

    ScgMapHeader &h = m->hdr;
    h.n_edges = E; h.grid_n = G; h.n_cand = n_cand; h.n_starts = n_starts;
    h.ball_r = ball_r;
    {
        volatile float hh = ball_r / 20.0f, r2 = ball_r * ball_r, tr2 = tr * tr;
        h.h = hh; h.r2 = r2; h.tr2 = tr2;
    }
    h.tx = tx; h.ty = ty; h.grid_f = (float)G;
    int off = align16((int)sizeof(ScgMapHeader));
    h.off_edges_a = off; off = align16(off + E * 16);
    h.off_edges_b = off; off = align16(off + E * 16);
    h.off_cells = off;   off = align16(off + G * G * 4);
    h.off_cand = off;    off = align16(off + n_cand * 2);
    h.off_starts = off;  off = align16(off + n_starts * 8);
    h.blob_bytes = off;
    m->h_blob = (unsigned char *)calloc(1, off);
    if (!m->h_blob) {
        scg_map_destroy(m);
        return SCG_ENOMEM;
    }
    memcpy(m->h_blob, &h, sizeof(h));
    float *ea = (float *)(m->h_blob + h.off_edges_a), *eb = (float *)(m->h_blob + h.off_edges_b);
    for (int ed = 0; ed < E; ++ed) {
        const float *row = m->h_edges + 8 * ed;
        memcpy(ea + 4 * ed, row, 16);
        eb[4 * ed + 0] = row[4]; eb[4 * ed + 1] = row[5]; eb[4 * ed + 2] = row[6];
        int ids = (m->h_obst[ed] << 8) | m->h_local[ed];
        memcpy(eb + 4 * ed + 3, &ids, 4);
    }
    uint32_t *cells = (uint32_t *)(m->h_blob + h.off_cells);
    uint16_t *cand = (uint16_t *)(m->h_blob + h.off_cand);
    int pos = 0;
    for (int c = 0; c < G * G; ++c) {
        m->h_cell_start[c] = pos;
        // bit 31: the goal test can succeed for a ball in this cell (the cell, grown by 0.003 for the extra move after a
        // bounce on the last substep, reaches the target disc): elsewhere the kernel skips the test (same result)
        const int ci = c / G, cj = c % G;
        const double mg = 0.003;
        const double ddx = std::max(std::max((double)ci / G - mg - (double)tx, (double)tx - ((double)(ci + 1) / G + mg)), 0.0);
        const double ddy = std::max(std::max((double)cj / G - mg - (double)ty, (double)ty - ((double)(cj + 1) / G + mg)), 0.0);
        const bool goal_near = ddx * ddx + ddy * ddy <= (double)tr * (double)tr * 1.0001 + 1e-9;
        cells[c] = (goal_near ? 0x80000000u : 0u) | ((uint32_t)pos << 8) | (uint32_t)lists[c].size();
        for (int ed : lists[c]) {
            m->h_cand[pos] = ed;
            cand[pos++] = (uint16_t)ed;
        }
    }
    m->h_cell_start[G * G] = pos;
    memcpy(m->h_blob + h.off_starts, starts, (size_t)n_starts * 8);

    cudaError_t ce = cudaMalloc((void **)&m->d_blob, h.blob_bytes);
    if (ce == cudaSuccess) ce = cudaMemcpy(m->d_blob, m->h_blob, h.blob_bytes, cudaMemcpyHostToDevice);
    if (ce != cudaSuccess) {
        scg_map_destroy(m);
        return (int)ce;
    }
    *out = m;
    return 0;
}

extern "C" int scg_map_destroy(scg_map_t *m) {
    if (!m) return 0;
    if (m->d_blob) cudaFree(m->d_blob);
    if (m->d_stage) cudaFree(m->d_stage);
    free(m->h_blob); free(m->h_edges); free(m->h_obst); free(m->h_local);
    free(m->h_cell_start); free(m->h_cand);
    free(m);
    return 0;
}
extern "C" int scg_map_num_edges(const scg_map_t *m) { return m ? m->hdr.n_edges : SCG_EINVAL; }
extern "C" int scg_map_num_candidates(const scg_map_t *m) { return m ? m->hdr.n_cand : SCG_EINVAL; }
extern "C" int scg_map_edge_table(const scg_map_t *m, float *edges_out, int *obst_out, int *local_out) {
    if (!m) return SCG_EINVAL;
    int E = m->hdr.n_edges;
    if (edges_out) memcpy(edges_out, m->h_edges, (size_t)E * 8 * sizeof(float));
    if (obst_out) memcpy(obst_out, m->h_obst, E * sizeof(int));
    if (local_out) memcpy(local_out, m->h_local, E * sizeof(int));
    return 0;
}
extern "C" int scg_map_grid(const scg_map_t *m, int *grid_n_out, int *cell_start_out, int *cand_out) {
    if (!m) return SCG_EINVAL;
    int G = m->hdr.grid_n;
    if (grid_n_out) *grid_n_out = G;
    if (cell_start_out) memcpy(cell_start_out, m->h_cell_start, ((size_t)G * G + 1) * sizeof(int));
    if (cand_out) memcpy(cand_out, m->h_cand, (size_t)m->hdr.n_cand * sizeof(int));
    return 0;
}

template <bool kCull>
__global__ void __launch_bounds__(256) k_step(const unsigned char *__restrict__ gblob, int blob_bytes, int B,
                                              const float *x, const float *y, const float *vx, const float *vy,
                                              const int *__restrict__ action, float *x2, float *y2, float *vx2,
                                              float *vy2, float *__restrict__ reward, int *__restrict__ flags) {
    extern __shared__ __align__(128) unsigned char smem[];
    __shared__ __align__(8) unsigned long long bar;
    stage3(smem, gblob, blob_bytes, nullptr, nullptr, 0, nullptr, nullptr, 0, &bar);
    const StepMap m = make_step_map(smem);
    for (int b = blockIdx.x * blockDim.x + threadIdx.x; b < B; b += gridDim.x * blockDim.x) {
        float px = x[b], py = y[b], pvx = vx[b], pvy = vy[b];
        int a = action[b];
        float r;
        int fl;
        pinball_step<kCull>(m, px, py, pvx, pvy, a, r, fl);
        x2[b] = px; y2[b] = py; vx2[b] = pvx; vy2[b] = pvy;
        reward[b] = r;
        flags[b] = fl;
    }
}

__global__ void k_reset(const unsigned char *__restrict__ gblob, int B, const uint8_t *__restrict__ mask, float *x,
                        float *y, float *vx, float *vy, uint64_t seed, uint32_t step, uint32_t env_offset) {
    const ScgMapHeader *h = reinterpret_cast<const ScgMapHeader *>(gblob);
    const float2 *starts = reinterpret_cast<const float2 *>(gblob + h->off_starts);
    int ns = h->n_starts;
    for (int b = blockIdx.x * blockDim.x + threadIdx.x; b < B; b += gridDim.x * blockDim.x) {
        if (mask && !mask[b]) continue;
        uint4 r = scg_draw(seed, env_offset + (uint32_t)b, step, SCG_STREAM_RESET);
        int pick = min((int)__fmul_rn(scg_u01(r.x), (float)ns), ns - 1);
        float2 s = starts[pick];
        x[b] = s.x; y[b] = s.y; vx[b] = 0.f; vy[b] = 0.f;
    }
}

int scg_launch_step(const scg_map_t *map, int B, const float *x, const float *y, const float *vx, const float *vy,
                    const int *action, float *x2, float *y2, float *vx2, float *vy2, float *reward, int *flags,
                    int cull, cudaStream_t st) {
    if (B == 0) return 0;
    const int threads = 256;
    int smem = map->hdr.blob_bytes;
    static ScgKernelCfg cfg_t = {}, cfg_f = {};
    int occ = 0, rcc;
    if ((rcc = scg_configure(cfg_t, k_step<true>, threads, (size_t)smem, &occ))) return rcc;
    if ((rcc = scg_configure(cfg_f, k_step<false>, threads, (size_t)smem, &occ))) return rcc;
    int grid = scg_grid(B, threads, 8);
    if (cull)
        k_step<true><<<grid, threads, smem, st>>>(map->d_blob, smem, B, x, y, vx, vy, action, x2, y2, vx2, vy2, reward, flags);
    else
        k_step<false><<<grid, threads, smem, st>>>(map->d_blob, smem, B, x, y, vx, vy, action, x2, y2, vx2, vy2, reward, flags);
    SCG_LAUNCH_CHECK();
    return 0;
}

extern "C" int scg_step(const scg_map_t *map, int B, const float *x, const float *y, const float *vx,
                        const float *vy, const int *action, float *x2, float *y2, float *vx2, float *vy2,
                        float *reward, int *flags, int cull, void *stream) {
    if (!map || B < 0 || (B > 0 && (!x || !y || !vx || !vy || !action || !x2 || !y2 || !vx2 || !vy2 || !reward || !flags)))
        return SCG_EINVAL;
    if (map->hdr.blob_bytes > 200 * 1024) return SCG_ELIMIT;
    return scg_launch_step(map, B, x, y, vx, vy, action, x2, y2, vx2, vy2, reward, flags, cull, (cudaStream_t)stream);
}

extern "C" int scg_reset(const scg_map_t *map, int B, const uint8_t *mask, float *x, float *y, float *vx, float *vy,
                         uint64_t seed, uint32_t step, uint32_t env_offset, void *stream) {
    if (!map || B < 0 || (B > 0 && (!x || !y || !vx || !vy))) return SCG_EINVAL;
    if (B == 0) return 0;
    k_reset<<<scg_grid(B, 256, 8), 256, 0, (cudaStream_t)stream>>>(map->d_blob, B, mask, x, y, vx, vy, seed, step, env_offset);
    SCG_LAUNCH_CHECK();
    return 0;
}

// HOST-buffer variant: the call a user of PinballEnv.step makes with NumPy arrays.
extern "C" int scg_step_host(scg_map_t *map, int B, float *state_soa, const int *action, float *reward,
                             int *flags, void *stream) {
    if (!map || B < 0 || (B > 0 && (!state_soa || !action || !reward || !flags))) return SCG_EINVAL;
    if (B == 0) return 0;
    cudaStream_t st = (cudaStream_t)stream;
    size_t need = (size_t)B * 7 * 4;  // 4 state + action + reward + flags
    if (need > map->stage_cap) {      // the staging block belongs to the map (freed by scg_map_destroy)
        if (map->d_stage) cudaFree(map->d_stage);
        map->d_stage = nullptr; map->stage_cap = 0;
        SCG_CUDA_OK(cudaMalloc((void **)&map->d_stage, need));
        map->stage_cap = need;
    }
    float *d_buf = map->d_stage;
    float *ds = d_buf;
    int *da = (int *)(d_buf + (size_t)4 * B);
    float *dr = d_buf + (size_t)5 * B;
    int *df = (int *)(d_buf + (size_t)6 * B);
    SCG_CUDA_OK(cudaMemcpyAsync(ds, state_soa, (size_t)B * 16, cudaMemcpyHostToDevice, st));
    SCG_CUDA_OK(cudaMemcpyAsync(da, action, (size_t)B * 4, cudaMemcpyHostToDevice, st));
    int rc = scg_launch_step(map, B, ds, ds + B, ds + 2 * (size_t)B, ds + 3 * (size_t)B, da, ds, ds + B,
                             ds + 2 * (size_t)B, ds + 3 * (size_t)B, dr, df, 1, st);
    if (rc) return rc;
    SCG_CUDA_OK(cudaMemcpyAsync(state_soa, ds, (size_t)B * 16, cudaMemcpyDeviceToHost, st));
    SCG_CUDA_OK(cudaMemcpyAsync(reward, dr, (size_t)B * 4, cudaMemcpyDeviceToHost, st));
    SCG_CUDA_OK(cudaMemcpyAsync(flags, df, (size_t)B * 4, cudaMemcpyDeviceToHost, st));
    SCG_CUDA_OK(cudaStreamSynchronize(st));
    return 0;
}
