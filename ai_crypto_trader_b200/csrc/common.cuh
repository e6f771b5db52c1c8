// Shared helpers for the b200bt kernels (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <atomic>
#include "b200bt.h"

namespace b200bt {

void set_error(const char* fmt, ...);
int check_device();
extern std::atomic<int64_t> g_launches;

inline int cuda_status(cudaError_t e, const char* what) {
    if (e == cudaSuccess) return B200BT_OK;
    set_error("%s: %s", what, cudaGetErrorString(e));
    return (int)e;
}

#define B200BT_REQUIRE(cond, code, ...)        \
    do {                                       \
        if (!(cond)) {                         \
            ::b200bt::set_error(__VA_ARGS__);  \
            return (code);                     \
        }                                      \
    } while (0)

// B200BT_TRACE_LAUNCHES=1 (debugging a stall): every launch is named on stderr and waited for, so the last name without a
// "done" is the kernel that does not finish.
inline bool trace_launches() {
    static const bool v = getenv("B200BT_TRACE_LAUNCHES") != nullptr;
    return v;
}

#define B200BT_LAUNCH_CHECK(what)                                       \
    do {                                                                \
        ::b200bt::g_launches.fetch_add(1, std::memory_order_relaxed);   \
        cudaError_t e__ = cudaGetLastError();                           \
        if (e__ != cudaSuccess) return ::b200bt::cuda_status(e__, what); \
        if (::b200bt::trace_launches()) {                               \
            fprintf(stderr, "[b200bt] %s ...", what); fflush(stderr);   \
            e__ = cudaDeviceSynchronize();                              \
            fprintf(stderr, " done (%d)\n", (int)e__); fflush(stderr);  \
        }                                                               \
    } while (0)

constexpr unsigned FULL = 0xffffffffu;

// Zone map of a sweep's price / RSI rows (b200bt_zone_map, csrc/sweep_chunked.cu): (min, max) per 32-bar block ("coarse")
// and per 4-bar group ("fine") of every row.  Layout: coarse [S][P + 1][zone_row_stride(N)] float2, then fine
// [S][P + 1][zone_fine_stride(N)] float2, row 0 = price; rows are 16-byte aligned and padded with (NaN, NaN).
constexpr int ZONE_BLOCK = 32;          // bars per coarse range
constexpr int ZONE_TILE = 128;          // bars per tile of the thread-per-lane scan (fine rows hold whole tiles)
__host__ __device__ constexpr int64_t zone_row_stride(int64_t N) { return (((N + ZONE_BLOCK - 1) / ZONE_BLOCK) + 1) & ~(int64_t)1; }
__host__ __device__ constexpr int64_t zone_fine_stride(int64_t N) { return ((N + ZONE_TILE - 1) / ZONE_TILE) * (ZONE_TILE / 4); }

// RSI from the two Wilder averages, ta.momentum.RSIIndicator: 100 if D == 0 else 100 - 100 / (1 + U / D), rounded to fp32.
// Evaluated as 100 U / (U + D) with ONE reciprocal: the two float64 divisions of the literal form were half of the RSI
// bank kernel's instructions.  The forms agree to ~2e-14 absolute (1.5 ulp each), so they round to the same fp32 value
// except on a ~1e-8 fraction of double-rounding ties -- below the 2e-6 the bank is tested at against float64 pandas.
// A D below the smallest normal double counts as 0: thousands of equal closes decay the averages into the subnormals, where
// the serial recurrence either rounds them to exactly 0 (period 2) or leaves them stuck at the smallest subnormal, and
// the scan's reassociated products round them differently; no price move is that small.  A sum still that small takes
// the literal form.
__device__ __forceinline__ float rsi_value(double U, double D) {
    if (D < 2.2250738585072014e-308) return 100.0f;
    const double S = U + D;
    if (S < 1e-290) return (float)(100.0 - 100.0 / (1.0 + U / D));
    return (float)((100.0 * U) * __drcp_rn(S));
}

// Seam states of RSI's Wilder averages over time tiles of `tile` bars (csrc/indicators.cu): seam[(sym P + p)(T - 1) + k]
// = (U, D) after the last bar of tile k of row (sym, p), k < T - 1, T = ceil(N / tile); a kernel that starts tile k + 1
// from it continues the serial recurrence exactly.
int rsi_seam_states(const float* close, int S, int64_t N, int64_t ld, const int* periods_host, int P, int tile, double2* seam,
                    cudaStream_t st);

__device__ __forceinline__ double shfl_up_d(double v, int d) {
    return __shfl_up_sync(FULL, v, d);
}
__device__ __forceinline__ double shfl_d(double v, int src) {
    return __shfl_sync(FULL, v, src);
}
__device__ __forceinline__ double shfl_xor_d(double v, int m) {
    return __shfl_xor_sync(FULL, v, m);
}

__device__ __forceinline__ double warp_sum_d(double v) {
#pragma unroll
    for (int m = 16; m > 0; m >>= 1) v += shfl_xor_d(v, m);
    return v;
}
__device__ __forceinline__ double warp_max_d(double v) {
#pragma unroll
    for (int m = 16; m > 0; m >>= 1) v = fmax(v, shfl_xor_d(v, m));
    return v;
}
__device__ __forceinline__ double warp_min_d(double v) {
#pragma unroll
    for (int m = 16; m > 0; m >>= 1) v = fmin(v, shfl_xor_d(v, m));
    return v;
}

// Trade-hash contribution of one event (event index, event word): two 32-bit multiply-xorshift
// mixes; the lane hash is the xor over all events (oracle/sim_oracle.c computes the same).
__host__ __device__ __forceinline__ uint64_t event_hash(uint32_t index, uint32_t word) {
    uint32_t a = (index * 0x9E3779B1u) ^ word;
    a *= 0x85EBCA77u;
    a ^= a >> 15;
    uint32_t b = (word * 0xC2B2AE3Du) ^ ((index << 13) | (index >> 19));
    b *= 0x27D4EB2Fu;
    b ^= b >> 16;
    return ((uint64_t)b << 32) | a;
}

}  // namespace b200bt
