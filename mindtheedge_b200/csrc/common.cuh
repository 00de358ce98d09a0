// Shared device/host helpers for libmte (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdlib.h>

#include <mutex>
#include <utility>
#include <vector>

#include "../../include/mte.h"

#define MTE_FULL_MASK 0xffffffffu

#define MTE_RETURN_IF_CUDA_ERROR()                        \
    do {                                                  \
        cudaError_t e__ = cudaGetLastError();             \
        if (e__ != cudaSuccess) return (int)e__;          \
    } while (0)

namespace mte {

// ---- per-device hardware facts (read-only after the first query; no algorithmic state) ---------------------
// The library may be used on several devices of one process: everything that depends on the device (SM count,
// shared-memory opt-in limit, the per-function MaxDynamicSharedMemorySize attribute) is keyed by the CURRENT
// device's ordinal, never cached process-wide.
struct DevInfo {
    int sms;         // multiprocessor count (148 on B200: 2 dies x 74)
    int smemOptin;   // cudaDevAttrMaxSharedMemoryPerBlockOptin
};
inline int current_device() {
    int d = 0;
    cudaGetDevice(&d);
    return d;
}
inline DevInfo dev_info() {
    constexpr int kMaxDev = 64;
    static DevInfo cache[kMaxDev];
    static bool have[kMaxDev];
    static std::mutex mu;
    const int d = current_device();
    std::lock_guard<std::mutex> lock(mu);
    if (d >= 0 && d < kMaxDev && have[d]) return cache[d];
    DevInfo v{148, 232448};
    cudaDeviceGetAttribute(&v.sms, cudaDevAttrMultiProcessorCount, d);
    cudaDeviceGetAttribute(&v.smemOptin, cudaDevAttrMaxSharedMemoryPerBlockOptin, d);
    if (v.sms < 1) v.sms = 1;
    if (d >= 0 && d < kMaxDev) { cache[d] = v; have[d] = true; }
    return v;
}
inline int num_sms() { return dev_info().sms; }

// Raise a kernel's dynamic shared-memory limit ONCE PER (function, device): the attribute is per device, so a
// process-wide "done" flag would leave the second GPU of a process at the 48 KB default.
inline cudaError_t opt_in_smem(const void *func, int bytes) {
    static std::mutex mu;
    static std::vector<std::pair<const void *, long long>> done;  // (function, device << 32 | bytes)
    const int d = current_device();
    std::lock_guard<std::mutex> lock(mu);
    for (auto &e : done)
        if (e.first == func && (int)(e.second >> 32) == d) {
            if ((int)(e.second & 0xffffffffLL) >= bytes) return cudaSuccess;
            const cudaError_t r = cudaFuncSetAttribute(func, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
            if (r == cudaSuccess) e.second = ((long long)d << 32) | (unsigned)bytes;
            return r;
        }
    const cudaError_t r = cudaFuncSetAttribute(func, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
    if (r == cudaSuccess) done.emplace_back(func, ((long long)d << 32) | (unsigned)bytes);
    return r;
}

// Dynamic shared memory a kernel can use on the current device: the opt-in limit less its static shared memory and
// 1 KB, opted in; 0 if nothing is left or the opt-in fails.
template <typename Kernel>
inline int smem_budget(Kernel *kernel) {
    cudaFuncAttributes fa;
    cudaFuncGetAttributes(&fa, kernel);
    int budget = dev_info().smemOptin - (int)fa.sharedSizeBytes - 1024;
    if (budget <= 0 || opt_in_smem((const void *)kernel, budget) != cudaSuccess) budget = 0;
    cudaGetLastError();
    return budget;
}

// Tuning / diagnostic switches exist ONLY in builds made with -DMTE_DEBUG_KNOBS (scripts/ use them through
// MTE_NVCC_DEFS); the release library never reads the environment, so no call's result or algorithm can depend on
// process-global state.
#ifdef MTE_DEBUG_KNOBS
inline const char *debug_knob(const char *name) { return getenv(name); }
#else
inline const char *debug_knob(const char *) { return nullptr; }
#endif

// Start of every workspace: self-resetting tickets / flags (256 B), then, inside the zero-initialised 64 KB
// header, the per-image accumulators of the edge-loss forward at kWsAccumOffset.
struct WsHeader {
    unsigned int ticket[16];
    unsigned int flag[16];
    unsigned int pad[32];
};
static_assert(sizeof(WsHeader) == 256, "workspace header layout");
constexpr size_t kWsAccumOffset = 4096;
constexpr int kWsMaxLossImages = (MTE_WS_HEADER_BYTES - 4096) / 64;  // 960 images (all scales together)

__host__ __device__ inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }
__host__ __device__ inline int ceil_div(int a, int b) { return (a + b - 1) / b; }

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(MTE_FULL_MASK, v, o);
    return v;
}
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(MTE_FULL_MASK, v, o);
    return v;
}
__device__ __forceinline__ unsigned warp_or(unsigned v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v |= __shfl_xor_sync(MTE_FULL_MASK, v, o);
    return v;
}

// 128-bit streaming loads/stores (read-once planes: evict-first, no L1 allocation)
__device__ __forceinline__ float4 ld_stream4(const float *p) { return __ldcs(reinterpret_cast<const float4 *>(p)); }
__device__ __forceinline__ float4 ld_cached4(const float *p) { return __ldg(reinterpret_cast<const float4 *>(p)); }
__device__ __forceinline__ void st_stream4(float *p, float4 v) { __stcs(reinterpret_cast<float4 *>(p), v); }

inline bool aligned16(const void *p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

namespace canny {
// canny.cu: multi-level 8-connected hysteresis on (cl, E) level planes: afterwards E(p) = first level t >= cl(p)
// at which p is connected, through pixels with cl <= t, to a pixel whose initial E <= t.
int run_level_hysteresis(const unsigned char *cl, unsigned char *E, int N, int H, int W, int T, void *scratch,
                         cudaStream_t st);
size_t hysteresis_scratch_bytes(int N, int H, int W);
}  // namespace canny

}  // namespace mte
