// sygnals_b200/csrc/syg_platform.h
//
// One source tree, two builds:
//   * nvcc  -gencode arch=compute_100a,code=sm_100a  -> sygnals_b200/libsygb200.so   (the product)
//   * g++   -DSYG_EMU                                -> tests/emu/libsygb200_emu.so   (TEST ONLY)
// The emulator build runs every kernel on the CPU with one fiber per CUDA thread (tests/emu/syg_emu.h) so
// the index arithmetic, barriers and host logic can be checked in the GPU-less build container before GPU
// time is spent.  The product package never loads the emulator library.
#pragma once

#include <cstddef>
#include <cstdint>

#ifdef SYG_EMU
#include "syg_emu.h"
#define SYG_LAUNCH(kernel, grid, block, smem, stream, ...) \
    ::sygemu::launch(dim3(grid), dim3(block), (size_t)(smem), [&]() { kernel(__VA_ARGS__); })
#define SYG_DYN_SMEM(name) unsigned char* name = ::sygemu::dyn_smem()
#define SYG_HD
#define SYG_DEVICE
#define SYG_INLINE inline
#define SYG_NOINLINE static inline
#define SYG_UNROLL
// separately rounded double multiply / add (never fused into one FMA); x86-64 g++ without -mfma has no FMA to fuse into
#define SYG_DMUL_RN(a, b) ((a) * (b))
#define SYG_DADD_RN(a, b) ((a) + (b))
#else
#include <cuda_runtime.h>
#define SYG_LAUNCH(kernel, grid, block, smem, stream, ...) \
    kernel<<<dim3(grid), dim3(block), (smem), (stream)>>>(__VA_ARGS__)
#define SYG_DYN_SMEM(name) extern __shared__ __align__(16) unsigned char name[]
#define SYG_HD __host__ __device__
#define SYG_DEVICE __device__
#define SYG_INLINE __forceinline__
#define SYG_NOINLINE static __noinline__
#define SYG_UNROLL _Pragma("unroll")
#define SYG_DMUL_RN(a, b) __dmul_rn((a), (b))
#define SYG_DADD_RN(a, b) __dadd_rn((a), (b))
#endif
