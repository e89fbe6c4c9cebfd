// ABI bookkeeping: status strings, version, device check, launch counter.
#include "common.cuh"

namespace cpc {
std::atomic<uint64_t> g_launches{0};

int check_device() {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return CPC_ERR_CUDA;
    int major = 0;
    if (cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev) != cudaSuccess) return CPC_ERR_CUDA;
    return major == 10 ? CPC_OK : CPC_ERR_ARCH;
}
}  // namespace cpc

extern "C" const char* cpc_status_string(int status) {
    switch (status) {
        case CPC_OK: return "ok";
        case CPC_ERR_BAD_SHAPE: return "bad shape";
        case CPC_ERR_ALIGNMENT: return "bad alignment";
        case CPC_ERR_WORKSPACE: return "workspace missing or too small";
        case CPC_ERR_ARCH: return "device is not sm_100 (B200)";
        case CPC_ERR_CUDA: return "CUDA runtime error";
        case CPC_ERR_UNSUPPORTED: return "unsupported configuration";
        case CPC_ERR_NULL: return "null pointer";
        default: return "unknown status";
    }
}
extern "C" int cpc_abi_version(void) { return 7; }
extern "C" int cpc_runtime_check(void) { return cpc::check_device(); }
extern "C" uint64_t cpc_launch_count(void) { return cpc::g_launches.load(); }
extern "C" void cpc_launch_count_reset(void) { cpc::g_launches.store(0); }
