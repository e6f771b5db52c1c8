// Family 1: rolling indicators over fp32 OHLCV (sm_100a).
//
// Data layout: every series is a row of a row-major [S][N] fp32 matrix; a bank
// is [S][P][N].  One CTA owns one (symbol, time-tile): it stages the close tile
// in shared memory once and its warps loop over the
// periods of the bank, so HBM sees 4 B/bar of input and 4 B/bar per output row.
//
// Linear recurrences (Wilder / EMA) are evaluated time-parallel: each lane
// folds K consecutive bars into an affine map, the warp composes the 32 maps
// with a shuffle scan, and the lanes replay their bars from the scanned state.
// Tiles are joined by an exact carry, not by a warm-up halo: RSI is the ratio
// U / (U + D) of two Wilder averages, and a ratio keeps its value when both
// terms decay, so a tile started from a zero state inside a run of equal closes
// reads 100 where the serial recurrence keeps the RSI the run started with.
// rsi_tile_end_kernel folds every tile but the last from a zero state into its
// end state, rsi_seam_kernel composes those per row into the true state at
// every seam (a warp scan over the tiles), and rsi_bank_kernel starts each tile
// from that state.
#include <math.h>
#include "common.cuh"

namespace b200bt {

constexpr int RSI_TILE = 4096;   // bars written per CTA
constexpr int RSI_K = 4;         // bars per lane per step
constexpr int RSI_STEP = 32 * RSI_K;
constexpr int RSI_MAX_P = 128;

struct RsiBankParams {
    int periods[RSI_MAX_P];
};

// (U, D) after the last bar of tile k of row (sym, p), from a zero state at the tile's first bar; every tile but the last
// of the series (those are whole).  One CTA per (tile, symbol), warps over the periods.  Lane l folds the 4-bar groups
// l, l + 32, ... of the tile: acc = acc * om^128 + (group folded from 0); the tile's state is the sum of the lanes'
// accumulators weighted by om^(4 (31 - l)).
__global__ void __launch_bounds__(256)
rsi_tile_end_kernel(const float* __restrict__ close, int64_t ld, const __grid_constant__ RsiBankParams prm, int P, int tile,
                    double2* __restrict__ ends) {
    extern __shared__ float s_c[];  // [tile + 1], s_c[i] = close[tile_start - 1 + i]
    const int sym = blockIdx.y;
    const int64_t tile_start = (int64_t)blockIdx.x * tile;
    const float* row = close + (int64_t)sym * ld;
    for (int i = threadIdx.x; i <= tile; i += blockDim.x) {
        const int64_t t = tile_start - 1 + i;
        s_c[i] = __ldg(row + (t < 0 ? 0 : t));          // diff = 0 at bar 0
    }
    __syncthreads();
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nwarp = blockDim.x >> 5;
    for (int pi = warp; pi < P; pi += nwarp) {
        const double alpha = 1.0 / (double)prm.periods[pi];
        const double om = 1.0 - alpha;
        const double a128 = pow(om, (double)RSI_STEP), wl = pow(om, (double)(RSI_K * (31 - lane)));
        double accU = 0.0, accD = 0.0;
        for (int base = 0; base < tile; base += RSI_STEP) {
            const int i = base + lane * RSI_K;
            double yU = 0.0, yD = 0.0;
#pragma unroll
            for (int j = 0; j < RSI_K; ++j) {
                const double df = (double)s_c[i + j + 1] - (double)s_c[i + j];
                yU = yU * om + alpha * (df > 0.0 ? df : 0.0);
                yD = yD * om + alpha * (df < 0.0 ? -df : 0.0);
            }
            accU = accU * a128 + yU;
            accD = accD * a128 + yD;
        }
        const double eU = warp_sum_d(accU * wl), eD = warp_sum_d(accD * wl);
        if (lane == 0) ends[((int64_t)sym * P + pi) * gridDim.x + blockIdx.x] = make_double2(eU, eD);
    }
}

// In place, one warp per row (sym, p) of `n_seam` entries: tile ends from a zero state -> the true (U, D) after the last
// bar of each tile, C_k = m C_{k-1} + E_k with m = om^tile, 32 tiles per step of an affine shuffle scan.
__global__ void __launch_bounds__(256)
rsi_seam_kernel(const __grid_constant__ RsiBankParams prm, int P, int rows, int n_seam, int tile, double2* __restrict__ seam) {
    const int lane = threadIdx.x & 31;
    const int r = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (r >= rows) return;
    const double om = 1.0 - 1.0 / (double)prm.periods[r % P];
    double mp[5];
#pragma unroll
    for (int i = 0; i < 5; ++i) mp[i] = pow(om, (double)tile * (double)(1 << i));
    const double ml = pow(om, (double)tile * (double)(lane + 1));
    double2* s = seam + (int64_t)r * n_seam;
    double cU = 0.0, cD = 0.0;
    for (int k0 = 0; k0 < n_seam; k0 += 32) {
        const int k = k0 + lane;
        const double2 e = k < n_seam ? s[k] : make_double2(0.0, 0.0);
        double yU = e.x, yD = e.y;
#pragma unroll
        for (int i = 0; i < 5; ++i) {
            const double upU = shfl_up_d(yU, 1 << i), upD = shfl_up_d(yD, 1 << i);
            if (lane >= (1 << i)) {
                yU += mp[i] * upU;
                yD += mp[i] * upD;
            }
        }
        yU += ml * cU;
        yD += ml * cD;
        if (k < n_seam) s[k] = make_double2(yU, yD);
        cU = shfl_d(yU, 31);
        cD = shfl_d(yD, 31);
    }
}

// ta.momentum.RSIIndicator semantics (binance_ml_strategy.py:112):
//   diff = close.diff(1); up = max(diff,0); dn = max(-diff,0)  (bar 0: 0)
//   U,D = ewm(alpha=1/w, adjust=False).mean() of up, dn  (y0 = x0)
//   rsi = 100 if D == 0 else 100 - 100/(1 + U/D), defined for t >= w-1
// Optional zone rows (zc / zf: coarse and fine parts of a sweep zone map, already offset to this launch's first symbol,
// rows of P_all + 1 entries per symbol with row 0 = price): the bank's (min, max) ranges are produced from the values in
// registers while they are written -- a lane's four bars ARE one 4-bar group, eight lanes one 32-bar block -- and the price
// row's from the staged closes, so the first sweep of a fresh bank already skips quiet blocks.
#ifndef B200BT_RSI_MIN_BLOCKS
#define B200BT_RSI_MIN_BLOCKS 3
#endif
__global__ void __launch_bounds__(256, B200BT_RSI_MIN_BLOCKS)
rsi_bank_kernel(const float* __restrict__ close, int64_t N, int64_t ld,
                const __grid_constant__ RsiBankParams prm, int P, int fill, const double2* __restrict__ seam,
                float* __restrict__ out, int vec_ok, float2* __restrict__ zc, float2* __restrict__ zf, int P_all, int p0) {
    extern __shared__ float s_close[];  // [RSI_TILE + 1], s_close[i] = close[tile_start - 1 + i]
    const int sym = blockIdx.y;
    const int64_t tile_start = (int64_t)blockIdx.x * RSI_TILE;
    const int64_t tile_end = min(tile_start + (int64_t)RSI_TILE, N);
    const int64_t s0 = tile_start;  // first bar staged
    const float* row = close + (int64_t)sym * ld;
    const int n_stage = RSI_TILE + 1;
    for (int i = threadIdx.x; i < n_stage; i += blockDim.x) {
        int64_t t = s0 - 1 + i;
        t = t < 0 ? 0 : (t >= N ? N - 1 : t);  // clamp: diff = 0 outside the series
        s_close[i] = __ldg(row + t);
    }
    __syncthreads();

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nwarp = blockDim.x >> 5;
    const float qnan = __int_as_float(0x7fc00000);
    const int64_t zstride = zone_row_stride(N), fstride = zone_fine_stride(N);
    const bool last_tile = tile_end == N;
    if (zc && p0 == 0) {
        // price row (row 0): ranges of the staged closes; s_close[t - s0 + 1] = close[t]
        float2* pc = zc + (int64_t)sym * (P_all + 1) * zstride;
        float2* pf = zf + (int64_t)sym * (P_all + 1) * fstride;
        for (int64_t t = tile_start + (int64_t)threadIdx.x * 4; t < tile_start + RSI_TILE; t += (int64_t)blockDim.x * 4) {
            float lo = qnan, hi = qnan;
#pragma unroll
            for (int j = 0; j < 4; ++j)
                if (t + j < N) { const float v = s_close[(int)(t + j - s0) + 1]; lo = fminf(lo, v); hi = fmaxf(hi, v); }
            if ((t >> 2) < fstride) pf[t >> 2] = make_float2(lo, hi);
#pragma unroll
            for (int m = 1; m < 8; m <<= 1) { lo = fminf(lo, __shfl_xor_sync(FULL, lo, m)); hi = fmaxf(hi, __shfl_xor_sync(FULL, hi, m)); }
            if ((lane & 7) == 0 && (t >> 5) < zstride) pc[t >> 5] = make_float2(lo, hi);
        }
        if (last_tile) {    // padding of the rows (whole tiles / even stride): ranges no compare is true for
            for (int64_t g = ((tile_start + RSI_TILE) >> 2) + threadIdx.x; g < fstride; g += blockDim.x) pf[g] = make_float2(qnan, qnan);
            for (int64_t b = ((tile_start + RSI_TILE) >> 5) + threadIdx.x; b < zstride; b += blockDim.x) pc[b] = make_float2(qnan, qnan);
        }
    }
    for (int pi = warp; pi < P; pi += nwarp) {
        const int w = prm.periods[pi];
        float* orow = out + ((int64_t)sym * P + pi) * N;
        float2* zcr = zc ? zc + ((int64_t)sym * (P_all + 1) + 1 + p0 + pi) * zstride : nullptr;
        float2* zfr = zc ? zf + ((int64_t)sym * (P_all + 1) + 1 + p0 + pi) * fstride : nullptr;
        const double alpha = 1.0 / (double)w;
        const double om = 1.0 - alpha;
        const double om2 = om * om, a4 = om2 * om2;  // per-lane chunk multiplier (K = 4)
        double apow[5];
        apow[0] = a4;
#pragma unroll
        for (int i = 1; i < 5; ++i) apow[i] = apow[i - 1] * apow[i - 1];
        double alane = 1.0;  // a4^(lane+1)
        {
            int e = lane + 1;
            double b = a4;
#pragma unroll
            for (int i = 0; i < 6; ++i) {
                if (e & 1) alane *= b;
                b *= b;
                e >>= 1;
            }
        }
        double carryU = 0.0, carryD = 0.0;     // the true state before the tile's first bar (rsi_seam_kernel)
        if (blockIdx.x > 0) {
            const double2 c = seam[((int64_t)sym * P + pi) * (gridDim.x - 1) + blockIdx.x - 1];
            carryU = c.x;
            carryD = c.y;
        }
        for (int64_t base = tile_start; base < tile_end; base += RSI_STEP) {
            const int64_t t = base + lane * RSI_K;
            const int si = (int)(t - s0);  // s_close[si] = close[t-1]
            double x[RSI_K + 1];
#pragma unroll
            for (int j = 0; j <= RSI_K; ++j) x[j] = (double)s_close[min(si + j, n_stage - 1)];
            double u[RSI_K], d[RSI_K];
#pragma unroll
            for (int j = 0; j < RSI_K; ++j) {
                double df = x[j + 1] - x[j];
                u[j] = df > 0.0 ? df : 0.0;
                d[j] = df < 0.0 ? -df : 0.0;
            }
            double yU = 0.0, yD = 0.0;
#pragma unroll
            for (int j = 0; j < RSI_K; ++j) {
                yU = yU * om + alpha * u[j];
                yD = yD * om + alpha * d[j];
            }
#pragma unroll
            for (int i = 0; i < 5; ++i) {
                double upU = shfl_up_d(yU, 1 << i), upD = shfl_up_d(yD, 1 << i);
                if (lane >= (1 << i)) {
                    yU += apow[i] * upU;
                    yD += apow[i] * upD;
                }
            }
            const double endU = yU + alane * carryU, endD = yD + alane * carryD;
            double U = shfl_up_d(endU, 1), D = shfl_up_d(endD, 1);
            if (lane == 0) { U = carryU; D = carryD; }
            carryU = shfl_d(endU, 31);
            carryD = shfl_d(endD, 31);
            float r[RSI_K];
#pragma unroll
            for (int j = 0; j < RSI_K; ++j) {
                U = U * om + alpha * u[j];
                D = D * om + alpha * d[j];
                r[j] = rsi_value(U, D);
            }
            const bool mine = t < tile_end;
            if (mine) {
                if (vec_ok && t + RSI_K <= tile_end) {
                    *reinterpret_cast<float4*>(orow + t) = make_float4(r[0], r[1], r[2], r[3]);
                } else {
#pragma unroll
                    for (int j = 0; j < RSI_K; ++j)
                        if (t + j < tile_end) orow[t + j] = r[j];
                }
            }
            if (zcr) {
                // this lane's four bars are one 4-bar group, eight lanes (the tile start is a multiple of 32) one 32-bar block
                float lo = qnan, hi = qnan;
#pragma unroll
                for (int j = 0; j < RSI_K; ++j)
                    if (mine && t + j < tile_end) { lo = fminf(lo, r[j]); hi = fmaxf(hi, r[j]); }
                if (mine) zfr[t >> 2] = make_float2(lo, hi);
#pragma unroll
                for (int m = 1; m < 8; m <<= 1) { lo = fminf(lo, __shfl_xor_sync(FULL, lo, m)); hi = fmaxf(hi, __shfl_xor_sync(FULL, hi, m)); }
                const int64_t tb = t & ~(int64_t)31;
                if ((lane & 7) == 0 && tb < tile_end) zcr[tb >> 5] = make_float2(lo, hi);
            }
        }
        if (zcr && last_tile) {
            for (int64_t g = ((tile_end + 3) >> 2) + lane; g < fstride; g += 32) zfr[g] = make_float2(qnan, qnan);
            for (int64_t b = ((tile_end + 31) >> 5) + lane; b < zstride; b += 32) zcr[b] = make_float2(qnan, qnan);
        }
        if (tile_start == 0 && w > 1) {
            // min_periods = w: bars [0, w-1) are undefined -> back-fill or NaN.
            __syncwarp();
            float v;
            if (fill) v = (w - 1 < N) ? orow[w - 1] : 0.0f;  // all-NaN column -> fillna(0)
            else v = __int_as_float(0x7fc00000);
            __syncwarp();
            const int64_t lim = min((int64_t)(w - 1), N);
            for (int64_t t = lane; t < lim; t += 32) orow[t] = v;
            if (zcr) {
                // the ranges of the groups / blocks that hold re-filled bars follow the final values
                __syncwarp();
                for (int64_t g = lane; g * 4 < lim + 4 && g * 4 < N; g += 32) {
                    float lo = qnan, hi = qnan;
                    for (int j = 0; j < 4; ++j)
                        if (g * 4 + j < N) { const float x = orow[g * 4 + j]; lo = fminf(lo, x); hi = fmaxf(hi, x); }
                    zfr[g] = make_float2(lo, hi);
                }
                for (int64_t b = lane; b * 32 < lim + 32 && b * 32 < N; b += 32) {
                    float lo = qnan, hi = qnan;
                    for (int j = 0; j < 32; ++j)
                        if (b * 32 + j < N) { const float x = orow[b * 32 + j]; lo = fminf(lo, x); hi = fmaxf(hi, x); }
                    zcr[b] = make_float2(lo, hi);
                }
            }
        }
    }
}

// Seam states of the Wilder averages of RSI over tiles of `tile` bars (a multiple of RSI_STEP): seam[(sym P + p)(T - 1) + k]
// = (U, D) after the last bar of tile k, k < T - 1, T = ceil(N / tile).  Nothing to do for a single tile.
int rsi_seam_states(const float* close, int S, int64_t N, int64_t ld, const int* periods_host, int P, int tile, double2* seam,
                    cudaStream_t st) {
    const int64_t T = (N + tile - 1) / tile;
    if (T < 2) return B200BT_OK;
    B200BT_REQUIRE(P <= RSI_MAX_P && tile % RSI_STEP == 0, B200BT_ELIMIT, "rsi seam states: bad tiling");
    RsiBankParams prm;
    for (int i = 0; i < P; ++i) prm.periods[i] = periods_host[i];
    const size_t smem = (size_t)(tile + 1) * sizeof(float);
    cudaError_t e = cudaFuncSetAttribute(rsi_tile_end_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return cuda_status(e, "rsi seam states: cudaFuncSetAttribute");
    rsi_tile_end_kernel<<<dim3((unsigned)(T - 1), (unsigned)S), 256, smem, st>>>(close, ld, prm, P, tile, seam);
    B200BT_LAUNCH_CHECK("rsi tile end launch");
    const int rows = S * P;
    rsi_seam_kernel<<<(unsigned)((rows + 7) / 8), 256, 0, st>>>(prm, P, rows, (int)(T - 1), tile, seam);
    B200BT_LAUNCH_CHECK("rsi seam launch");
    return B200BT_OK;
}

}  // namespace b200bt

using namespace b200bt;

static int rsi_bank_impl(const float* close, int S, int64_t N, int64_t ld, const int* periods_host, int P, int fill,
                         float* out, float* zones, int S_total, int sym0, b200bt_stream_t stream);

extern "C" int b200bt_rsi_bank(const float* close, int S, int64_t N, int64_t ld,
                               const int* periods_host, int P, int fill,
                               float* out, b200bt_stream_t stream) {
    return rsi_bank_impl(close, S, N, ld, periods_host, P, fill, out, nullptr, 0, 0, stream);
}

extern "C" int b200bt_rsi_bank_zones(const float* close, int S, int64_t N, int64_t ld, const int* periods_host, int P,
                                     float* out, float* zones, int S_total, int sym0, b200bt_stream_t stream) {
    B200BT_REQUIRE(zones && S_total >= S && sym0 >= 0 && sym0 + S <= S_total, B200BT_EINVAL, "rsi_bank_zones: bad zone-map arguments");
    B200BT_REQUIRE(((uintptr_t)zones & 15) == 0, B200BT_EINVAL, "rsi_bank_zones: zone map must be 16-byte aligned");
    return rsi_bank_impl(close, S, N, ld, periods_host, P, 1, out, zones, S_total, sym0, stream);
}

static int rsi_bank_launches(const float* close, int S, int64_t N, int64_t ld, const int* periods_host, int P, int fill,
                             float* out, float* zones, int S_total, int sym0, double2* seam, cudaStream_t st) {
    const bool vec_ok = (N % 4 == 0) && (((uintptr_t)out & 15) == 0);
    const size_t smem = (size_t)(RSI_TILE + 4) * sizeof(float);
    for (int p0 = 0; p0 < P; p0 += RSI_MAX_P) {
        const int pc = (P - p0) < RSI_MAX_P ? (P - p0) : RSI_MAX_P;
        RsiBankParams prm;
        for (int i = 0; i < pc; ++i) prm.periods[i] = periods_host[p0 + i];
        int rc = rsi_seam_states(close, S, N, ld, periods_host + p0, pc, RSI_TILE, seam, st);
        if (rc) return rc;
        dim3 grid((unsigned)((N + RSI_TILE - 1) / RSI_TILE), (unsigned)S);
        // the launch writes rows [p0, p0+pc) of every symbol: pass the full-P row pitch via (P, pi offset)
        float2* zc = zones ? (float2*)zones + (int64_t)sym0 * (P + 1) * zone_row_stride(N) : nullptr;
        float2* zf = zones ? (float2*)zones + (int64_t)S_total * (P + 1) * zone_row_stride(N) + (int64_t)sym0 * (P + 1) * zone_fine_stride(N) : nullptr;
        rsi_bank_kernel<<<grid, 256, smem, st>>>(close, N, ld, prm, pc, fill, seam,
                                                  out + (int64_t)p0 * N, vec_ok ? 1 : 0, zc, zf, P, p0);
        B200BT_LAUNCH_CHECK("rsi_bank launch");
    }
    return B200BT_OK;
}

static int rsi_bank_impl(const float* close, int S, int64_t N, int64_t ld, const int* periods_host, int P, int fill,
                         float* out, float* zones, int S_total, int sym0, b200bt_stream_t stream) {
    B200BT_REQUIRE(close && out && periods_host, B200BT_EINVAL, "rsi_bank: null pointer");
    B200BT_REQUIRE(S > 0 && N > 0 && P > 0 && ld >= N, B200BT_EINVAL, "rsi_bank: bad sizes S=%d N=%lld P=%d", S, (long long)N, P);
    B200BT_REQUIRE(P <= RSI_MAX_P, B200BT_ELIMIT, "rsi_bank: at most %d periods per call", RSI_MAX_P);
    for (int i = 0; i < P; ++i)
        B200BT_REQUIRE(periods_host[i] >= 1 && periods_host[i] <= RSI_TILE, B200BT_ELIMIT, "rsi_bank: window %d outside [1,%d]",
                       periods_host[i], RSI_TILE);
    int rc = check_device();
    if (rc) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    // seam states of one launch's rows, stream-ordered: concurrent calls on other streams get their own
    const int64_t T = (N + RSI_TILE - 1) / RSI_TILE;
    double2* seam = nullptr;
    if (T > 1) {
        cudaError_t e = cudaMallocAsync((void**)&seam, (size_t)S * (P < RSI_MAX_P ? P : RSI_MAX_P) * (T - 1) * sizeof(double2), st);
        if (e != cudaSuccess) return cuda_status(e, "rsi_bank: seam states");
    }
    rc = rsi_bank_launches(close, S, N, ld, periods_host, P, fill, out, zones, S_total, sym0, seam, st);
    if (seam) {
        cudaError_t e = cudaFreeAsync(seam, st);
        if (!rc && e != cudaSuccess) rc = cuda_status(e, "rsi_bank: seam states");
    }
    return rc;
}
