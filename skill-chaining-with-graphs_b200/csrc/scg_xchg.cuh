// scg_xchg.cuh - layout of a rank's peer-memory exchange block (scg_xchg.cu, scg_ctl.cu).
#pragma once
#include "scg_common.cuh"

#define XCHG_SLICE 256                 // elements per CTA
#define XCHG_HDR 32                    // per-slice header: update counts [0..15] and success counters [16..31] of the K options (int bits)
#define XCHG_ROW (XCHG_SLICE + XCHG_HDR)
#define XCHG_MAX_WORLD 16

struct scg_xchg {
    int rank, world, order, n, K, slices;
    uint32_t seq;
    size_t bytes, flag_bytes;
    // [flags: world*slices u32 | 16 spare u32 | xbuf: 2*slices*XCHG_ROW f32 | controller region, see XCHG_M_*]
    unsigned char *d_local;
    size_t m_off;                                // byte offset of the controller region
    unsigned char *d_peer[XCHG_MAX_WORLD];       // mapped bases of every rank's block (own entry = d_local)
    bool ipc_opened[XCHG_MAX_WORLD];
    unsigned int *d_ticket;                      // last-CTA-done counter
    volatile uint32_t *h_status;                 // host-mapped sticky "a peer timed out" flag (written by the kernel)
    uint32_t *d_status;                          // its device alias
    long long timeout_cycles;                    // peer wait limit in SM clock cycles
};


// controller region of the block (the classifier fit of scg_agent_manage exchanges per-step gradient sums through it):
//   u32 mflag[XCHG_MAX_WORLD]   round number last signalled by each peer
//   u32 mseq                    rounds completed so far (kept on the device: only the kernel knows whether it promoted)
//   f32 mbuf[2][32]             this rank's values of the current / previous round: (6 gradient sums, example count) of a
//                               fit step, or (inside-counts of up to 16 older options, positive count) of the merge detection
#define XCHG_M_FLAG 0
#define XCHG_M_SEQ (XCHG_MAX_WORLD * 4)
#define XCHG_M_BUF (XCHG_MAX_WORLD * 4 + 16)
#define XCHG_M_WORDS 32
#define XCHG_M_BYTES (XCHG_M_BUF + 2 * XCHG_M_WORDS * 4)

#ifdef __CUDACC__
__device__ __forceinline__ void st_release_sys(uint32_t *p, uint32_t v) {
    asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ uint32_t ld_acquire_sys(const uint32_t *p) {
    uint32_t v;
    asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ float ld_sys_f32(const float *p) {
    float v;
    asm volatile("ld.relaxed.sys.global.f32 %0, [%1];" : "=f"(v) : "l"(p) : "memory");
    return v;
}

// One peer's half of a flag round: publish round `seq` in the peer's flag for us (after this thread's earlier writes,
// system scope), then wait for the peer to raise our flag for it to `seq`.  A peer that does not come within
// timeout_cycles is fatal for the exchange: raise the sticky host-mapped status and return false.
__device__ __forceinline__ bool xchg_signal_wait(uint32_t *peer_flag, const uint32_t *own_flag, uint32_t seq, uint32_t *status,
                                                 long long timeout_cycles) {
    __threadfence_system();
    st_release_sys(peer_flag, seq);
    const long long t0 = clock64();
    while ((int32_t)(ld_acquire_sys(own_flag) - seq) < 0) {
        if (clock64() - t0 > timeout_cycles) {
            *reinterpret_cast<volatile uint32_t *>(status) = 1u;
            __threadfence_system();
            return false;
        }
    }
    return true;
}

#endif
