// Shared helpers for the sm_100a learner kernels.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>
#include <stdlib.h>

#include "../../include/impala_b200.h"

#define IMPALA_FULL_MASK 0xffffffffu

static inline int64_t impala_round_up(int64_t x, int64_t a) { return (x + a - 1) / a * a; }

struct MlpLayout {
    int64_t oW1, ob1, oW2, ob2, total;
};

static inline MlpLayout impala_make_layout(int O, int H, int N2) {
    MlpLayout l;
    const int64_t al = IMPALA_PARAM_ALIGN;
    l.oW1 = 0;
    l.ob1 = impala_round_up(l.oW1 + (int64_t)H * O, al);
    l.oW2 = impala_round_up(l.ob1 + H, al);
    l.ob2 = impala_round_up(l.oW2 + (int64_t)N2 * H, al);
    l.total = impala_round_up(l.ob2 + N2, al);
    return l;
}

// Kernels this library has launched (or recorded into a capturing stream) since it was loaded;
// defined in abi.cu, read through impala_launch_count().
extern long long g_impala_launches;

// Called once after every kernel launch of the library.
static inline int impala_launch_status() {
    __atomic_fetch_add(&g_impala_launches, 1, __ATOMIC_RELAXED);
    cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? IMPALA_OK : (int)e;
}

// SM count of the current device (cached per device).
static inline cudaError_t impala_sm_count(int* out) {
    static int cached[64] = {0};
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    if (dev < 0 || dev >= 64 || !cached[dev]) {
        int n = 0;
        if ((e = cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev)) != cudaSuccess) return e;
        if (dev < 0 || dev >= 64) return *out = n, cudaSuccess;
        cached[dev] = n;
    }
    *out = cached[dev];
    return cudaSuccess;
}

static inline int impala_env_int(const char* name, int dflt) {
    const char* v = getenv(name);
    return (v && *v) ? atoi(v) : dflt;
}

// A persistent launch of `grid` CTAs shared by two tile lists (policy / value network): how many
// CTAs take list A so that the slower side finishes earliest, for per-tile cost weights wa, wb.
static inline int impala_pair_split(int tiles_a, int tiles_b, int grid, int64_t wa, int64_t wb) {
    int best = 1;
    int64_t best_cost = INT64_MAX, best_sum = INT64_MAX;
    for (int na = 1; na < grid; ++na) {
        const int nb = grid - na;
        if (na > tiles_a || nb > tiles_b) continue;
        const int64_t ca = (int64_t)((tiles_a + na - 1) / na) * wa, cb = (int64_t)((tiles_b + nb - 1) / nb) * wb;
        const int64_t cost = ca > cb ? ca : cb, sum = ca + cb;
        if (cost < best_cost || (cost == best_cost && sum < best_sum)) best = na, best_cost = cost, best_sum = sum;
    }
    return best;
}

__device__ __forceinline__ double warp_sum_f64(double x) {
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) x += __shfl_xor_sync(IMPALA_FULL_MASK, x, off);
    return x;
}

// For kernels that contain a grid-wide barrier: a cooperative launch FAILS (instead of the barrier
// hanging) when the CTAs cannot all be resident, e.g. under an MPS SM limit or in a green context.
template <typename... KArgs, typename... Args>
static inline cudaError_t impala_launch_cooperative(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem,
                                                    cudaStream_t st, Args&&... args) {
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = grid, cfg.blockDim = block, cfg.dynamicSmemBytes = smem, cfg.stream = st;
    cudaLaunchAttribute attr;
    attr.id = cudaLaunchAttributeCooperative;
    attr.val.cooperative = 1;
    cfg.attrs = &attr, cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}

// ---- push-model all-reduce over peer memory, LL ("low latency") format (protocol: see optim.cu)
// One float64 travels as 16 bytes  [lo32 | step32 | hi32 | step32] : each 8-byte half carries the
// step number it belongs to, 8-byte stores are single NVLink transactions, so a reader that sees
// both halves tagged with the step it is waiting for has the value - no fence, no separate flag,
// no acknowledgement on the data path.
struct PushArgs {
    ulonglong2* const* gather;  // device array [world]: every rank's gather buffer (peer-mapped)
    const long long* seq;       // this rank's step counter (device, 1 word); the step in flight is *seq + 1
    int64_t slot_stride;        // LL elements between two ranks' slots
    int64_t buf_stride;         // LL elements between the two parity buffers
    int rank, world;
};
__device__ __forceinline__ void ll_store(ulonglong2* dst, double v, unsigned step) {
    const unsigned long long bits = (unsigned long long)__double_as_longlong(v);
    const unsigned long long tag = (unsigned long long)step << 32;
    const unsigned long long lo = (bits & 0xffffffffull) | tag, hi = (bits >> 32) | tag;
    // plain (weak) 16-byte store: LL needs no ordering between elements, only that each 8-byte half
    // lands whole - which any aligned 8-byte store does
    asm volatile("st.global.v2.u64 [%0], {%1, %2};" ::"l"(dst), "l"(lo), "l"(hi) : "memory");
}
__device__ __forceinline__ ulonglong2 ll_load(const ulonglong2* src) {
    ulonglong2 w;
    asm volatile("ld.volatile.global.v2.u64 {%0, %1}, [%2];" : "=l"(w.x), "=l"(w.y) : "l"(src) : "memory");
    return w;
}
__device__ __forceinline__ bool ll_ready(const ulonglong2& w, unsigned step) {
    return (unsigned)(w.x >> 32) == step && (unsigned)(w.y >> 32) == step;
}
__device__ __forceinline__ double ll_value(const ulonglong2& w) {
    return __longlong_as_double((long long)((w.x & 0xffffffffull) | (w.y << 32)));
}
