// scg_api.cu - error strings, version and the launch counter of the C ABI (include/scg_b200.h).
#include "scg_common.cuh"

uint64_t g_scg_launches = 0;

int scg_num_sms() {
    static int sms[SCG_MAX_DEVICES];
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= SCG_MAX_DEVICES) return 0;
    if (sms[dev] == 0 && cudaDeviceGetAttribute(&sms[dev], cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) sms[dev] = 0;
    return sms[dev];
}

extern "C" const char *scg_error_string(int code) {
    if (code == 0) return "ok";
    if (code == SCG_EINVAL) return "scg: invalid argument";
    if (code == SCG_ENOMEM) return "scg: host allocation failed";
    if (code == SCG_ELIMIT) return "scg: size exceeds a compiled-in limit (order 1..5, K <= 16 option slots including the top-level ones)";
    if (code == SCG_EPEER) return "scg: a peer rank did not arrive at a cross-GPU weight exchange within the timeout; the replicas are out of step";
    if (code > 0) return cudaGetErrorString((cudaError_t)code);
    return "scg: unknown error";
}

extern "C" int scg_version(void) { return 222; }

extern "C" uint64_t scg_launch_count(void) { return g_scg_launches; }
