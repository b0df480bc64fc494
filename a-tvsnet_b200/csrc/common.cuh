// common.cuh - error plumbing shared by every translation unit of libatvs.so.
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <stdint.h>
#include <stdio.h>
#include <atomic>
#include "../../include/atvs.h"

void atvs_set_error(const char* fmt, ...);

#define ATVS_CHECK_ARG(cond, code, ...)                   \
    do {                                                  \
        if (!(cond)) {                                    \
            atvs_set_error(__VA_ARGS__);                  \
            return (code);                                \
        }                                                 \
    } while (0)

#define ATVS_CUDA(call)                                                               \
    do {                                                                              \
        cudaError_t e__ = (call);                                                     \
        if (e__ != cudaSuccess) {                                                     \
            atvs_set_error("%s:%d %s -> %s", __FILE__, __LINE__, #call,               \
                           cudaGetErrorString(e__));                                  \
            return (int)e__;                                                          \
        }                                                                             \
    } while (0)

void atvs_count_launch();
// device counter (one per device, allocated on first use - never during stream capture: every path is warmed up
// eagerly first) of fp16 raw-output rows that had to be clamped to +-65504; read with atvs_saturation_count()
unsigned long long* atvs_sat_ptr();
int atvs_concurrency();          // api.cu: passes the caller runs side by side on the current device
#define ATVS_LAUNCH_CHECK()              \
    do {                                 \
        atvs_count_launch();             \
        ATVS_CUDA(cudaPeekAtLastError()); \
    } while (0)

// State the library keeps per device (include/atvs.h) is indexed by the device ordinal.
#define ATVS_MAX_DEVICES 64
// *dev = the calling thread's current device, which every launch and query of the library applies to; 0, or the
// failing call's code with the message set (also for an ordinal beyond ATVS_MAX_DEVICES)
int atvs_current_device(int* dev);
int atvs_num_sms();              // api.cu: SMs of the current device (148 when it cannot be read)

// Opts KERNEL in to 227 KB of dynamic shared memory.  A function attribute belongs to the device that was current
// when it was set, so it is set once per (kernel, device); threads that race on a first launch set the same value.
template <auto KERNEL>
int atvs_max_dynamic_smem() {
    static std::atomic<bool> done[ATVS_MAX_DEVICES];
    int dev = 0;
    if (const int rc = atvs_current_device(&dev)) return rc;
    if (!done[dev].load(std::memory_order_acquire)) {
        ATVS_CUDA(cudaFuncSetAttribute(KERNEL, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
        done[dev].store(true, std::memory_order_release);
    }
    return 0;
}
