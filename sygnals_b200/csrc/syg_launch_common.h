// helpers shared by the kernel translation units
#pragma once

#include <algorithm>
#include <mutex>
#include <string>

#include "syg_launch.h"

#ifndef SYG_EMU
#define SYG_OCCUPANCY(nb, kernel, threads, smem) cudaOccupancyMaxActiveBlocksPerMultiprocessor(&(nb), kernel, threads, smem)
#else
#define SYG_OCCUPANCY(nb, kernel, threads, smem) ((nb) = 2, cudaSuccess)
#endif

#define LCK(expr)                                                                          \
    do {                                                                                   \
        cudaError_t e_ = (expr);                                                           \
        if (e_ != cudaSuccess) { err = std::string(#expr) + ": " + cudaGetErrorString(e_); return -3; } \
    } while (0)

namespace syglaunch {
inline int ilog2i(long long v) { int l = 0; while ((1LL << l) < v) ++l; return l; }

// cudaFuncSetAttribute(MaxDynamicSharedMemorySize) and the occupancy result are PER DEVICE: one process may drive several GPUs
// (one syg_ctx each, possibly from several threads), so every kernel instantiation keeps one slot per device behind a mutex.
constexpr int kMaxDevices = 64;
struct KernelCache {
    std::mutex mu;
    size_t opted[kMaxDevices] = {};      // largest dynamic size opted in so far (the attribute only ever grows)
    size_t smem[kMaxDevices] = {};       // dynamic size the cached occupancy was measured for
    int blocks[kMaxDevices] = {};
};

// Makes `kfn` launchable with `smem` bytes of dynamic shared memory on the CURRENT device and returns the resident CTAs per SM
// for (threads, smem) in *blocks.  One cache per kernel FUNCTION (the attribute belongs to the function, not to a launch variant).
template <class K>
inline int prepare_kernel(K kfn, int threads, size_t smem, KernelCache& kc, int* blocks, std::string& err) {
    int dev = 0;
    LCK(cudaGetDevice(&dev));
    if (dev < 0 || dev >= kMaxDevices) { err = "device index out of range"; return -3; }
    std::lock_guard<std::mutex> lk(kc.mu);
    if (smem > kc.opted[dev] && smem > 48 * 1024) {
        // checked here rather than left to cudaFuncSetAttribute: its failure would also linger as the thread's last error and
        // fail the caller's next launch check
        int optin = 0;
        LCK(cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev));
        if (smem > (size_t)optin) {
            err = "the plan needs " + std::to_string(smem) + " bytes of shared memory per block, the device allows " + std::to_string(optin);
            return -5;                                               // SYG_E_UNSUPPORTED
        }
        LCK(cudaFuncSetAttribute(kfn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        kc.opted[dev] = smem;
    }
    if (kc.blocks[dev] == 0 || kc.smem[dev] != smem) {
        int nb = 0;
        LCK(SYG_OCCUPANCY(nb, kfn, threads, smem));
        if (nb < 1) { err = "kernel does not fit on an SM"; return -3; }
        kc.blocks[dev] = nb;
        kc.smem[dev] = smem;
    }
    *blocks = kc.blocks[dev];
    return 0;
}
}
