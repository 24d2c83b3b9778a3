// scg_xchg.cu - S5, the cross-GPU weight-delta exchange, as ONE kernel over NVLink peer memory (sm_100a).
//
// Mirrors the multi-rank step of oracle/option.py OptionSet.apply ("dW and cnt are summed over ranks before
// apply()"; the reference has no code: /root/reference/README.md:1-2).  Every rank owns an env slice and a full
// replica of the option weights.  At a sync, k_sync on every GPU
//   1. publishes its slice of the window's dW (and its update counts) in its own exchange buffer,
//   2. raises a per-slice sequence flag in every peer's flag array (st.release.sys over NVLink),
//   3. waits for the same slice's flag from every peer (ld.acquire.sys on local memory),
//   4. reads that slice from every peer (NVLink P2P loads), sums in rank order - identical on every GPU, so the
//      replicas stay bit-identical - and applies  W += alpha * alpha_scale_f * dW_sum * (steps / cnt_sum),
//      refreshes the packed copy Wt and zeroes dW.
// One launch replaces two NCCL all-reduces and the apply kernel; the payload is 20 KiB .. 203 KiB, so the cost is
// a couple of NVLink round trips.  CTA c only ever waits for CTA c of the peers, which signals before it waits,
// so no grid-wide barrier (and no co-residency assumption beyond one CTA) is needed.  The exchange buffer is
// double-buffered by sequence parity: a rank can only be one sync ahead of the slowest reader.
// A peer that does not show up within the timeout (default 30 s, scg_xchg_set_timeout) is FATAL for the exchange: the
// waiting CTA raises a sticky flag in host-mapped memory and returns without applying or zeroing its slice; every later
// scg_xchg_sync / scg_agent_run on this handle returns SCG_EPEER (the host reads the flag without a device sync), so a
// stalled or dead rank can never silently de-synchronise the weight replicas.
// Peer buffers are mapped with CUDA IPC (one process per GPU) or passed as plain pointers (one process, several
// devices with peer access enabled - used by the two-device test).
#include <stdlib.h>
#include <string.h>

#include <algorithm>

#include "scg_common.cuh"

#include "scg_xchg.cuh"

struct SyncArgs {
    int n, K, K_opt, slices, rank, world;
    uint32_t seq;
    float alpha, alpha_top, steps;
    float *W, *Wt, *dW;
    int *cnt;
    const int *nsucc_local;   // [K] this rank's option success counters (may be NULL)
    int *nsucc_global;        // [K] out: their sum over ranks as of this sync (may be NULL)
    unsigned int *ticket;
    uint32_t *status;         // host-mapped sticky timeout flag
    long long timeout_cycles;
    size_t flag_bytes;
    unsigned char *peer[XCHG_MAX_WORLD];
};

template <int N1>
__global__ void __launch_bounds__(XCHG_SLICE, 8) k_sync(const __grid_constant__ SyncArgs a) {
    constexpr int F = N1 * N1 * N1 * N1;
    __shared__ int s_cnt[SCG_MAX_OPTIONS];
    __shared__ float s_hdr[XCHG_MAX_WORLD * XCHG_HDR];
    __shared__ int s_timeout;
    if (threadIdx.x == 0) s_timeout = 0;
    const int c = blockIdx.x, i = threadIdx.x, j = c * XCHG_SLICE + i;
    const int buf = a.seq & 1;
    unsigned char *mine = a.peer[a.rank];
    float *xrow = reinterpret_cast<float *>(mine + a.flag_bytes) + ((size_t)buf * a.slices + c) * XCHG_ROW;
    // 1. publish
    const float my = (j < a.n) ? a.dW[j] : 0.f;
    xrow[i] = my;
    if (i < a.K) {
        xrow[XCHG_SLICE + i] = __int_as_float(a.cnt[i]);
        xrow[XCHG_SLICE + 16 + i] = __int_as_float(a.nsucc_local ? a.nsucc_local[i] : 0);
    }
    __syncthreads();
    // 2. signal every peer, 3. wait for every peer (one thread per peer)
    if (i < a.world && i != a.rank &&
        !xchg_signal_wait(reinterpret_cast<uint32_t *>(a.peer[i]) + (size_t)a.rank * a.slices + c,
                          reinterpret_cast<const uint32_t *>(mine) + (size_t)i * a.slices + c, a.seq, a.status,
                          a.timeout_cycles))
        s_timeout = 1;                                // the peer never came: fatal for this exchange (see the header)
    __syncthreads();
    if (s_timeout) return;                            // no apply, dW of this slice kept (the whole CTA returns)
    // 4. sum in rank order, apply
    // every peer's copy of this slice: the NVLink loads of (up to) eight peers are issued before the first one is
    // consumed - one round trip per sync on an 8-GPU box, not one per peer - then added in rank order.  The 32-word
    // headers (update counts, success counters) are fetched by all threads together into shared memory.
    for (int h = i; h < a.world * XCHG_HDR; h += XCHG_SLICE) {
        const int r = h / XCHG_HDR, wd = h - r * XCHG_HDR;
        const float *prow = reinterpret_cast<const float *>(a.peer[r] + a.flag_bytes) + ((size_t)buf * a.slices + c) * XCHG_ROW;
        s_hdr[h] = (r == a.rank) ? xrow[XCHG_SLICE + wd] : ld_sys_f32(prow + XCHG_SLICE + wd);
    }
    float v = 0.f;
    for (int r0 = 0; r0 < a.world; r0 += 8) {
        float pv[8];
#pragma unroll
        for (int q = 0; q < 8; ++q) {
            const int r = r0 + q;
            pv[q] = 0.f;
            if (r < a.world && r != a.rank) {
                const float *prow = reinterpret_cast<const float *>(a.peer[r] + a.flag_bytes) + ((size_t)buf * a.slices + c) * XCHG_ROW;
                pv[q] = ld_sys_f32(prow + i);
            }
        }
#pragma unroll
        for (int q = 0; q < 8; ++q)
            if (r0 + q < a.world) v += (r0 + q == a.rank) ? my : pv[q];
    }
    __syncthreads();
    if (i < a.K) {
        int tot = 0;
        long long succ = 0;   // the counters are 32-bit and wrap: summed as unsigned
        for (int r = 0; r < a.world; ++r) {
            tot += __float_as_int(s_hdr[r * XCHG_HDR + i]);
            if (c == 0) succ += (unsigned int)__float_as_int(s_hdr[r * XCHG_HDR + 16 + i]);
        }
        s_cnt[i] = tot;
        // every rank publishes the same global success count, so the option-creation controller takes the same
        // decision everywhere without a collective of its own
        if (c == 0 && a.nsucc_global) a.nsucc_global[i] = (int)(succ > 0x7fffffffll ? 0x7fffffffll : succ);
    }
    __syncthreads();
    if (j < a.n)
        scg_apply_elem<N1>(j, s_cnt[j / (SCG_A * F)], a.K_opt, a.alpha, a.alpha_top, a.steps, v, a.W, a.Wt, a.dW);
    // the last CTA to finish zeroes cnt for the next window (every CTA read it when it published)
    if (scg_last_block(a.ticket, gridDim.x) && i < a.K) a.cnt[i] = 0;
}

// ---- host side ------------------------------------------------------------------------------------------
// the peer wait limit in SM clock cycles of the current device
static cudaError_t set_timeout_cycles(scg_xchg *x, double seconds) {
    int dev = 0, khz = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e == cudaSuccess) e = cudaDeviceGetAttribute(&khz, cudaDevAttrClockRate, dev);
    x->timeout_cycles = (long long)(seconds * 1000.0 * (double)(khz > 0 ? khz : 2000000));
    return e;
}

extern "C" int scg_xchg_create(scg_ctx_t *ctx, int rank, int world, scg_xchg_t **out) {
    if (!ctx || !out || world < 1 || world > XCHG_MAX_WORLD || rank < 0 || rank >= world) return SCG_EINVAL;
    if (ctx->K > 16) return SCG_ELIMIT;
    scg_xchg *x = (scg_xchg *)calloc(1, sizeof(scg_xchg));
    if (!x) return SCG_ENOMEM;
    x->rank = rank; x->world = world; x->order = ctx->order; x->K = ctx->K;
    x->n = ctx->K * SCG_A * ctx->F;
    x->slices = (x->n + XCHG_SLICE - 1) / XCHG_SLICE;
    x->flag_bytes = (((size_t)world * x->slices + 16) * sizeof(uint32_t) + 255) & ~(size_t)255;
    x->m_off = x->flag_bytes + (size_t)2 * x->slices * XCHG_ROW * sizeof(float);
    x->bytes = x->m_off + ((XCHG_M_BYTES + 255) & ~255);
    cudaError_t e = cudaMalloc((void **)&x->d_local, x->bytes);
    if (e == cudaSuccess) e = cudaMemset(x->d_local, 0, x->bytes);
    if (e == cudaSuccess) e = cudaMalloc((void **)&x->d_ticket, sizeof(unsigned int));
    if (e == cudaSuccess) e = cudaMemset(x->d_ticket, 0, sizeof(unsigned int));
    if (e == cudaSuccess) e = cudaHostAlloc((void **)&x->h_status, 64, cudaHostAllocMapped);
    if (e == cudaSuccess) {
        *x->h_status = 0u;
        e = cudaHostGetDevicePointer((void **)&x->d_status, (void *)x->h_status, 0);
    }
    if (e == cudaSuccess) e = set_timeout_cycles(x, 30.0);
    if (e == cudaSuccess) e = cudaDeviceSynchronize();
    if (e != cudaSuccess) {
        if (x->d_local) cudaFree(x->d_local);
        if (x->d_ticket) cudaFree(x->d_ticket);
        if (x->h_status) cudaFreeHost((void *)x->h_status);
        free(x);
        return (int)e;
    }
    x->d_peer[rank] = x->d_local;
    *out = x;
    return 0;
}

extern "C" int scg_xchg_destroy(scg_xchg_t *x) {
    if (!x) return 0;
    for (int r = 0; r < x->world; ++r)
        if (x->ipc_opened[r]) cudaIpcCloseMemHandle(x->d_peer[r]);
    if (x->d_local) cudaFree(x->d_local);
    if (x->d_ticket) cudaFree(x->d_ticket);
    if (x->h_status) cudaFreeHost((void *)x->h_status);
    free(x);
    return 0;
}

extern "C" int scg_xchg_set_timeout(scg_xchg_t *x, double seconds) {
    if (!x || !(seconds > 0.0)) return SCG_EINVAL;
    SCG_CUDA_OK(set_timeout_cycles(x, seconds));
    return 0;
}

extern "C" int scg_xchg_handle_bytes(void) { return (int)sizeof(cudaIpcMemHandle_t); }

extern "C" int scg_xchg_local_ptr(scg_xchg_t *x, void **ptr_out) {
    if (!x || !ptr_out) return SCG_EINVAL;
    *ptr_out = x->d_local;
    return 0;
}

extern "C" int scg_xchg_handle(scg_xchg_t *x, void *handle_out) {
    if (!x || !handle_out) return SCG_EINVAL;
    cudaIpcMemHandle_t h;
    SCG_CUDA_OK(cudaIpcGetMemHandle(&h, x->d_local));
    memcpy(handle_out, &h, sizeof(h));
    return 0;
}

extern "C" int scg_xchg_connect(scg_xchg_t *x, const void *all_handles) {
    if (!x || !all_handles) return SCG_EINVAL;
    const unsigned char *hs = (const unsigned char *)all_handles;
    for (int r = 0; r < x->world; ++r) {
        if (r == x->rank) continue;
        cudaIpcMemHandle_t h;
        memcpy(&h, hs + (size_t)r * sizeof(h), sizeof(h));
        void *p = nullptr;
        SCG_CUDA_OK(cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess));
        x->d_peer[r] = (unsigned char *)p;
        x->ipc_opened[r] = true;
    }
    return 0;
}

extern "C" int scg_xchg_connect_ptrs(scg_xchg_t *x, void *const *peer_ptrs) {
    if (!x || !peer_ptrs) return SCG_EINVAL;
    for (int r = 0; r < x->world; ++r) {
        if (r == x->rank) continue;
        if (!peer_ptrs[r]) return SCG_EINVAL;
        x->d_peer[r] = (unsigned char *)peer_ptrs[r];
    }
    return 0;
}

extern "C" int scg_xchg_status(scg_xchg_t *x, int *timed_out) {
    if (!x || !timed_out) return SCG_EINVAL;
    *timed_out = (int)*x->h_status;     // host-mapped: no device synchronisation (sticky once set)
    return 0;
}

// dW (already reduced over this rank's slabs) and cnt -> summed over ranks -> applied; dW and cnt zeroed
extern "C" int scg_xchg_sync(scg_xchg_t *x, int K_opt, float *W, float *Wt, float *dW, int *cnt, float alpha,
                             float alpha_top, int window_steps, const int *nsucc_local, int *nsucc_global, void *stream) {
    if (!x || !W || !Wt || !dW || !cnt || K_opt < 0 || K_opt > x->K) return SCG_EINVAL;
    for (int r = 0; r < x->world; ++r)
        if (!x->d_peer[r]) return SCG_EINVAL;   // not connected
    if (*x->h_status) return SCG_EPEER;         // an earlier exchange timed out: the replicas are no longer in step
    SyncArgs a;
    a.n = x->n; a.K = x->K; a.K_opt = K_opt; a.alpha_top = alpha_top; a.slices = x->slices; a.rank = x->rank; a.world = x->world;
    a.seq = ++x->seq;
    a.alpha = alpha; a.steps = (float)std::max(window_steps, 1);
    a.W = W; a.Wt = Wt; a.dW = dW; a.cnt = cnt; a.ticket = x->d_ticket;
    a.status = x->d_status; a.timeout_cycles = x->timeout_cycles;
    a.nsucc_local = nsucc_local; a.nsucc_global = nsucc_global;
    a.flag_bytes = x->flag_bytes;
    for (int r = 0; r < XCHG_MAX_WORLD; ++r) a.peer[r] = r < x->world ? x->d_peer[r] : nullptr;
    cudaStream_t st = (cudaStream_t)stream;
    DISPATCH_ORDER(x->order, k_sync<N1><<<x->slices, XCHG_SLICE, 0, st>>>(a));
    SCG_LAUNCH_CHECK();
    return 0;
}
