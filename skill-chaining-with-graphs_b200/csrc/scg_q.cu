// scg_q.cu - K2 (Fourier features, per-option Q evaluation, epsilon-greedy selection, TD error)
// and K4 (initiation-classifier evaluation, gradient, fit) as stand-alone operators (sm_100a).
//
// Mirrors oracle/fourier.py FourierBasis.features and oracle/option.py OptionSet.q / act /
// td_error / initiation_prob / clf_grad / fit_initiation (the reference has no code:
// /root/reference/README.md:1-2).
//
// K2 design: one thread per env.  phi = cos(pi C s_hat) is never materialised: four sincospi
// calls give z_j = exp(i pi s_hat_j), the multi-index loops keep running complex products, and
// each pair of features is consumed by five two-wide FMAs the moment it is formed (scg_q_one / scg_q_pair
// in scg_common.cuh).  Weights are read from the packed pair layout (WtLayout: 48 bytes per feature pair,
// three 16-byte loads), warp-uniform when the warp's envs execute the same option.  The contraction is
// (B x F).(F x 5): far too skinny for tcgen05 tiles, so it stays on the FP32 pipe.
// Roofline: FP32, 18 F flop per (env, option).
#include "scg_common.cuh"

// ---- features (debug / parity operator; the hot path never writes phi to HBM) ------------------
template <int N1>
__global__ void k_features(int B, const float *__restrict__ x, const float *__restrict__ y,
                           const float *__restrict__ vx, const float *__restrict__ vy, float *__restrict__ phi) {
    constexpr int F = N1 * N1 * N1 * N1;
    for (int b = blockIdx.x * blockDim.x + threadIdx.x; b < B; b += gridDim.x * blockDim.x) {
        float2 z[4];
        scg_phasors(x[b], y[b], vx[b], vy[b], z);
        float2 p3[N1];
        p3[0] = make_float2(1.f, 0.f);
#pragma unroll
        for (int c = 1; c < N1; ++c) p3[c] = scg_cmul(p3[c - 1], z[3]);
        float *out = phi + (size_t)b * F;
        float2 z0 = make_float2(1.f, 0.f);
        for (int c0 = 0; c0 < N1; ++c0) {
            float2 z01 = z0;
            for (int c1 = 0; c1 < N1; ++c1) {
                float2 z012 = z01;
                for (int c2 = 0; c2 < N1; ++c2) {
#pragma unroll
                    for (int c3 = 0; c3 < N1; ++c3) *out++ = fmaf(z012.x, p3[c3].x, -z012.y * p3[c3].y);
                    z012 = scg_cmul(z012, z[2]);
                }
                z01 = scg_cmul(z01, z[1]);
            }
            z0 = scg_cmul(z0, z[0]);
        }
    }
}

// W [K][5][F] -> the packed pair layout (scg_common.cuh WtLayout): one thread per (slot, pair)
template <int N1>
__global__ void k_pack_weights(int K, const float *__restrict__ W, float *__restrict__ Wt) {
    using L = WtLayout<N1>;
    constexpr int F = N1 * N1 * N1 * N1;
    const int n = K * L::P;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const int k = i / L::P, pi = i - k * L::P;
        const int row = pi / L::NP, j = pi - row * L::NP;
        const int fa = row * N1 + 2 * j;
        const bool has_b = 2 * j + 1 < N1;          // an odd N1 pairs its last feature with a phantom of weight 0
        const float *w = W + (size_t)k * SCG_A * F;
        float *o = Wt + (size_t)k * L::SLOT_FLOATS + pi * 12;
#pragma unroll
        for (int a = 0; a < 4; ++a) {
            o[a] = w[(size_t)a * F + fa];
            o[4 + a] = has_b ? w[(size_t)a * F + fa + 1] : 0.f;
        }
        o[8] = w[(size_t)4 * F + fa];
        o[9] = has_b ? w[(size_t)4 * F + fa + 1] : 0.f;
        o[10] = o[11] = 0.f;
    }
}

template <int N1>
__global__ void __launch_bounds__(128) k_q_eval(int K, int B, const float *__restrict__ x, const float *__restrict__ y,
                                                const float *__restrict__ vx, const float *__restrict__ vy,
                                                const int *__restrict__ option, const float *__restrict__ Wt,
                                                float *__restrict__ Q) {
    for (int b = blockIdx.x * blockDim.x + threadIdx.x; b < B; b += gridDim.x * blockDim.x) {
        float2 z[4];
        scg_phasors(x[b], y[b], vx[b], vy[b], z);
        int o = min(max(option[b], 0), K - 1);
        float q[SCG_A];
        scg_q_one<N1, false>(z, WCur<false>(Wt, WtLayout<N1>::SLOT_FLOATS, o), q);
#pragma unroll
        for (int a = 0; a < SCG_A; ++a) Q[(size_t)b * SCG_A + a] = q[a];
    }
}

__global__ void k_select(int B, const float *__restrict__ Q, float eps, uint64_t seed, uint32_t step,
                         uint32_t stream_id, uint32_t env_offset, int *__restrict__ action) {
    for (int b = blockIdx.x * blockDim.x + threadIdx.x; b < B; b += gridDim.x * blockDim.x) {
        float q[SCG_A];
#pragma unroll
        for (int a = 0; a < SCG_A; ++a) q[a] = Q[(size_t)b * SCG_A + a];
        action[b] = scg_eps_greedy(q, eps, scg_draw(seed, env_offset + (uint32_t)b, step, stream_id));
    }
}

template <int N1>
__global__ void __launch_bounds__(128) k_td(int K, int B, const float *__restrict__ x, const float *__restrict__ y,
                                            const float *__restrict__ vx, const float *__restrict__ vy,
                                            const int *__restrict__ a, const float *__restrict__ r,
                                            const float *__restrict__ x2, const float *__restrict__ y2,
                                            const float *__restrict__ vx2, const float *__restrict__ vy2,
                                            const int *__restrict__ a2, const uint8_t *__restrict__ done,
                                            const int *__restrict__ option, const float *__restrict__ Wt, float gamma,
                                            float *__restrict__ delta) {
    for (int b = blockIdx.x * blockDim.x + threadIdx.x; b < B; b += gridDim.x * blockDim.x) {
        float2 za[4], zb[4];
        scg_phasors(x[b], y[b], vx[b], vy[b], za);
        scg_phasors(x2[b], y2[b], vx2[b], vy2[b], zb);
        int o = min(max(option[b], 0), K - 1);
        float qa[SCG_A], qb[SCG_A];
        scg_q_pair<N1, false>(za, zb, WCur<false>(Wt, WtLayout<N1>::SLOT_FLOATS, o), qa, qb);
        int ia = a[b], ib = a2[b];
        float qsa = 0.f, qs2 = 0.f;
#pragma unroll
        for (int i = 0; i < SCG_A; ++i) {
            qsa = (i == ia) ? qa[i] : qsa;
            qs2 = (i == ib) ? qb[i] : qs2;
        }
        float nd = done[b] ? 0.f : 1.f;
        delta[b] = __fsub_rn(__fadd_rn(r[b], __fmul_rn(__fmul_rn(gamma, nd), qs2)), qsa);
    }
}

// ---- K4 -----------------------------------------------------------------------------------------
__global__ void k_clf_eval(int B, const float *__restrict__ x, const float *__restrict__ y,
                           const float *__restrict__ theta, int K, float *__restrict__ p) {
    for (int b = blockIdx.x * blockDim.x + threadIdx.x; b < B; b += gridDim.x * blockDim.x) {
        float px = x[b], py = y[b];
        float xx = px * px, xy = px * py, yy = py * py;
        for (int k = 0; k < K; ++k) {
            const float *t = theta + k * SCG_N_PSI;
            float z = t[0];
            z = fmaf(t[1], px, z); z = fmaf(t[2], py, z); z = fmaf(t[3], xx, z);
            z = fmaf(t[4], xy, z); z = fmaf(t[5], yy, z);
            p[(size_t)b * K + k] = 1.0f / (1.0f + expf(-z));
        }
    }
}

// initiation decisions I_k(s) = (theta_k . psi >= 0) on the fp32 logit of scg_init_logit: bit-identical to the oracle
__global__ void k_clf_decide(int B, const float *__restrict__ x, const float *__restrict__ y,
                             const float *__restrict__ theta, int K, uint8_t *__restrict__ out) {
    for (int b = blockIdx.x * blockDim.x + threadIdx.x; b < B; b += gridDim.x * blockDim.x) {
        const uint32_t bits = scg_init_bits(theta, K, 0xffffffffu, x[b], y[b]);
        for (int k = 0; k < K; ++k) out[(size_t)b * K + k] = (bits >> k) & 1u;
    }
}

// mean_i (p_i - y_i) psi_i and the batch gradient-descent fit, each in a single CTA (clf_grad_sum, scg_common.cuh)
__global__ void __launch_bounds__(1024) k_clf_grad(int N, const float *__restrict__ X, const uint8_t *__restrict__ y,
                                                   const float *__restrict__ theta_k, float *__restrict__ grad) {
    __shared__ float sm[33 * SCG_N_PSI];
    float th[SCG_N_PSI], g[SCG_N_PSI];
#pragma unroll
    for (int j = 0; j < SCG_N_PSI; ++j) th[j] = theta_k[j];
    ClfCache c;
    clf_load(N, X, y, c);
    clf_grad_sum(N, X, y, c, th, g, sm);
    if (threadIdx.x < SCG_N_PSI) grad[threadIdx.x] = g[threadIdx.x] / (float)N;
}

__global__ void __launch_bounds__(1024) k_clf_fit(int N, const float *__restrict__ X, const uint8_t *__restrict__ y,
                                                  float *theta_k, int steps, float lr) {
    __shared__ float sm[33 * SCG_N_PSI];
    float th[SCG_N_PSI], g[SCG_N_PSI];
#pragma unroll
    for (int j = 0; j < SCG_N_PSI; ++j) th[j] = theta_k[j];
    ClfCache c;
    clf_load(N, X, y, c);
    for (int it = 0; it < steps; ++it) {
        clf_grad_sum(N, X, y, c, th, g, sm);
        clf_step(th, lr, g, (float)N);
    }
    if (threadIdx.x < SCG_N_PSI) theta_k[threadIdx.x] = th[threadIdx.x];
}

// ---- C ABI ------------------------------------------------------------------------------------

extern "C" int scg_features(int order, int B, const float *x, const float *y, const float *vx, const float *vy,
                            float *phi, void *stream) {
    if (B < 0 || (B > 0 && (!x || !y || !vx || !vy || !phi))) return SCG_EINVAL;
    if (B == 0) return 0;
    cudaStream_t st = (cudaStream_t)stream;
    DISPATCH_ORDER(order, k_features<N1><<<scg_grid(B, 128, 16), 128, 0, st>>>(B, x, y, vx, vy, phi));
    SCG_LAUNCH_CHECK();
    return 0;
}

extern "C" int scg_packed_slot_floats(int order) { return scg_wt_slot_floats(order); }

extern "C" int scg_pack_weights(int order, int K, const float *W, float *Wt, void *stream) {
    if (order < 1 || order > SCG_MAX_ORDER || K < 1 || K > SCG_MAX_OPTIONS) return SCG_ELIMIT;
    if (!W || !Wt) return SCG_EINVAL;
    int F = scg_pow4(order + 1);
    DISPATCH_ORDER(order, k_pack_weights<N1><<<scg_grid(K * WtLayout<N1>::P, 256, 16), 256, 0, (cudaStream_t)stream>>>(K, W, Wt));
    SCG_LAUNCH_CHECK();
    return 0;
}

extern "C" int scg_q_eval(int order, int K, int B, const float *x, const float *y, const float *vx, const float *vy,
                          const int *option, const float *Wt, float *Q, void *stream) {
    if (K < 1 || K > SCG_MAX_OPTIONS) return SCG_ELIMIT;
    if (B < 0 || (B > 0 && (!x || !y || !vx || !vy || !option || !Wt || !Q))) return SCG_EINVAL;
    if (B == 0) return 0;
    cudaStream_t st = (cudaStream_t)stream;
    DISPATCH_ORDER(order, k_q_eval<N1><<<scg_grid(B, 128, 16), 128, 0, st>>>(K, B, x, y, vx, vy, option, Wt, Q));
    SCG_LAUNCH_CHECK();
    return 0;
}

extern "C" int scg_select(int B, const float *Q, float epsilon, uint64_t seed, uint32_t step, uint32_t stream_id,
                          uint32_t env_offset, int *action, void *stream) {
    if (B < 0 || (B > 0 && (!Q || !action))) return SCG_EINVAL;
    if (B == 0) return 0;
    k_select<<<scg_grid(B, 256, 16), 256, 0, (cudaStream_t)stream>>>(B, Q, epsilon, seed, step, stream_id, env_offset, action);
    SCG_LAUNCH_CHECK();
    return 0;
}

extern "C" int scg_td_error(int order, int K, int B, const float *x, const float *y, const float *vx, const float *vy,
                            const int *a, const float *r, const float *x2, const float *y2, const float *vx2,
                            const float *vy2, const int *a2, const uint8_t *done, const int *option, const float *Wt,
                            float gamma, float *delta, void *stream) {
    if (K < 1 || K > SCG_MAX_OPTIONS) return SCG_ELIMIT;
    if (B < 0 || (B > 0 && (!x || !y || !vx || !vy || !a || !r || !x2 || !y2 || !vx2 || !vy2 || !a2 || !done ||
                            !option || !Wt || !delta)))
        return SCG_EINVAL;
    if (B == 0) return 0;
    cudaStream_t st = (cudaStream_t)stream;
    DISPATCH_ORDER(order, k_td<N1><<<scg_grid(B, 128, 16), 128, 0, st>>>(K, B, x, y, vx, vy, a, r, x2, y2, vx2, vy2, a2,
                                                                       done, option, Wt, gamma, delta));
    SCG_LAUNCH_CHECK();
    return 0;
}

extern "C" int scg_clf_eval(int B, const float *x, const float *y, const float *theta, int K, float *p, void *stream) {
    if (K < 1 || K > SCG_MAX_OPTIONS) return SCG_ELIMIT;
    if (B < 0 || (B > 0 && (!x || !y || !theta || !p))) return SCG_EINVAL;
    if (B == 0) return 0;
    k_clf_eval<<<scg_grid(B, 256, 16), 256, 0, (cudaStream_t)stream>>>(B, x, y, theta, K, p);
    SCG_LAUNCH_CHECK();
    return 0;
}

extern "C" int scg_clf_decide(int B, const float *x, const float *y, const float *theta, int K, uint8_t *inside, void *stream) {
    if (K < 1 || K > SCG_MAX_OPTIONS) return SCG_ELIMIT;
    if (B < 0 || (B > 0 && (!x || !y || !theta || !inside))) return SCG_EINVAL;
    if (B == 0) return 0;
    k_clf_decide<<<scg_grid(B, 256, 16), 256, 0, (cudaStream_t)stream>>>(B, x, y, theta, K, inside);
    SCG_LAUNCH_CHECK();
    return 0;
}

extern "C" int scg_clf_grad(int N, const float *X, const uint8_t *y, const float *theta_k, float *grad, void *stream) {
    if (N <= 0 || !X || !y || !theta_k || !grad) return SCG_EINVAL;
    k_clf_grad<<<1, 1024, 0, (cudaStream_t)stream>>>(N, X, y, theta_k, grad);
    SCG_LAUNCH_CHECK();
    return 0;
}

extern "C" int scg_clf_fit(int N, const float *X, const uint8_t *y, float *theta_k, int steps, float lr, void *stream) {
    if (N <= 0 || steps < 0 || !X || !y || !theta_k) return SCG_EINVAL;
    k_clf_fit<<<1, 1024, 0, (cudaStream_t)stream>>>(N, X, y, theta_k, steps, lr);
    SCG_LAUNCH_CHECK();
    return 0;
}
