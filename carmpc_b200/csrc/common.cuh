// Shared host/device helpers of the carmpc B200 library (sm_100a only).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string>

#include "../../include/carmpc.h"

namespace carmpc {

constexpr int kNumSMsFallback = 148;     // B200: 2 dies x 74 SMs
constexpr int kWarp = 32;

enum HandleKind : uint32_t { kPolytope = 0x504f4c59u, kRollout = 0x524f4c4cu, kQP = 0x51504144u, kShard = 0x53485244u,
                         kQPCheck = 0x51434b52u };

struct HandleBase {
    uint32_t kind;
    int device;
    virtual ~HandleBase() {}
};

void set_error(const char* fmt, ...);

#define CARMPC_CUDA(call)                                                                   \
    do {                                                                                    \
        cudaError_t err__ = (call);                                                         \
        if (err__ != cudaSuccess) {                                                         \
            ::carmpc::set_error("%s failed at %s:%d: %s", #call, __FILE__, __LINE__,        \
                                cudaGetErrorString(err__));                                 \
            return CARMPC_ERR_CUDA;                                                         \
        }                                                                                   \
    } while (0)

#define CARMPC_REQUIRE(cond, msg)                                                           \
    do {                                                                                    \
        if (!(cond)) {                                                                      \
            ::carmpc::set_error("invalid argument: %s (%s)", msg, #cond);                   \
            return CARMPC_ERR_INVALID;                                                      \
        }                                                                                   \
    } while (0)

int sm_count();

// Dynamic shared-memory opt-in and occupancy of a kernel, cached per (function, device, size): both are host-side
// driver calls of several microseconds, which adds up for pipelines of many small launches (closed-loop steps).
// per_sm (nullable) receives the resident CTAs per SM.
int kernel_config(const void* fn, int threads, size_t smem, int* per_sm);

template <class T>
inline T* check_handle(void* h, HandleKind kind) {
    if (h == nullptr) return nullptr;
    HandleBase* b = static_cast<HandleBase*>(h);
    return b->kind == kind ? static_cast<T*>(b) : nullptr;
}

// streaming 128-bit global load that does not allocate in L1 (read-once data)
__device__ __forceinline__ double2 ld_stream_f64x2(const double* p) {
    double2 r;
    asm volatile("ld.global.nc.L1::no_allocate.v2.f64 {%0, %1}, [%2];" : "=d"(r.x), "=d"(r.y) : "l"(p));
    return r;
}
__device__ __forceinline__ double ld_stream_f64(const double* p) {
    double r;
    asm volatile("ld.global.nc.L1::no_allocate.f64 %0, [%1];" : "=d"(r) : "l"(p));
    return r;
}

// Packed float32 pairs (sm_100a FFMA2): one instruction issues two IEEE fmas, lane-wise identical to fmaf.  A pair built
// from the same scalar twice is folded by ptxas into a broadcast operand (R.F32), so "scalar x pair + pair" costs one slot.
typedef unsigned long long f32x2;
__device__ __forceinline__ f32x2 pack2(float lo, float hi) {
    f32x2 r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
    return r;
}
__device__ __forceinline__ void unpack2(f32x2 v, float& lo, float& hi) {
    asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v));
}
__device__ __forceinline__ f32x2 ffma2(f32x2 a, f32x2 b, f32x2 c) {
    f32x2 d;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c));
    return d;
}

}  // namespace carmpc
