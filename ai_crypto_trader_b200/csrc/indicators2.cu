// Family 1 (continued): EMA / MACD / SMA / Bollinger / stochastic / Williams %R /
// Ichimoku / ATR / VWAP over fp32 OHLCV, plus the TechnicalAnalyzer NaN policy (sm_100a).
//
// Reference call sites: binance_ml_strategy.py:63-182 (TechnicalAnalyzer, via the third-party
// `ta` package, whose definitions are restated in oracle/indicators_ref.py) and
// services/market_monitor_service.py:219-301.
//
// Common scheme: one CTA per (symbol, time tile).  The input tile plus a halo is staged in
// shared memory once; arithmetic is fp64 so a float64 CPU evaluation rounds to the same
// fp32 outputs; undefined leading values are written as NaN and, when the caller asks for
// the reference's `_handle_nan_values` policy, resolved by the nanfill kernels
// (ffill -> bfill -> 0).
//   * exponential recurrences (EMA, MACD, ATR): time-parallel affine warp scan, tiles made
//     independent by a warm-up halo that attenuates the unknown state below 2^-60 (RSI, a
//     ratio of two such averages that a halo cannot make exact, is carried across the seams:
//     rsi_seam_states, csrc/indicators.cu);
//   * window sums (SMA, Bollinger, VWAP, %D): fp64 prefix sums of tile-offset values in
//     shared memory, window sum = difference of two prefixes;
//   * window extrema (stochastic, Williams, Ichimoku): direct scan of the window in shared
//     memory (exact: min/max do not round).
#include <math.h>
#include "common.cuh"

namespace b200bt {

constexpr int IND_TILE = 2048;
constexpr int IND_THREADS = 256;
constexpr int IND_MAX_WINDOW = 1024;
constexpr int IND_MAX_P = 64;
__device__ __forceinline__ float nanf32() { return __int_as_float(0x7fc00000); }

struct BankParams {
    int window[IND_MAX_P];
    int halo[IND_MAX_P];
};

// ---------------------------------------------------------------------------------
// Affine warp scan: y_t = om*y_{t-1} + b_t over 32 lanes x K consecutive bars per lane.
// In: b[K] per lane (already scaled), carry = state before the block's first bar.
// Out: y[K] = states after each of the lane's bars; carry updated to the state after the
// block's last bar.  apow[i] = (om^K)^(2^i), alane = (om^K)^(lane+1).
// ---------------------------------------------------------------------------------
template <int K>
struct AffineScan {
    double om, apow[5], alane;
    __device__ void init(double om_, int lane) {
        om = om_;
        double a = 1.0;
#pragma unroll
        for (int j = 0; j < K; ++j) a *= om;
        apow[0] = a;
#pragma unroll
        for (int i = 1; i < 5; ++i) apow[i] = apow[i - 1] * apow[i - 1];
        alane = 1.0;
        int e = lane + 1;
        double b = a;
#pragma unroll
        for (int i = 0; i < 6; ++i) {
            if (e & 1) alane *= b;
            b *= b;
            e >>= 1;
        }
    }
    __device__ void run(const double (&b)[K], double& carry, double (&y)[K], int lane) const {
        double acc = 0.0;
#pragma unroll
        for (int j = 0; j < K; ++j) acc = acc * om + b[j];
#pragma unroll
        for (int i = 0; i < 5; ++i) {
            const double up = shfl_up_d(acc, 1 << i);
            if (lane >= (1 << i)) acc += apow[i] * up;
        }
        const double end = acc + alane * carry;
        double st = shfl_up_d(end, 1);
        if (lane == 0) st = carry;
        carry = shfl_d(end, 31);
#pragma unroll
        for (int j = 0; j < K; ++j) {
            st = st * om + b[j];
            y[j] = st;
        }
    }
};

__device__ __forceinline__ void stage_row(const float* __restrict__ row, int64_t N, int64_t s0, int n_stage,
                                          float* __restrict__ dst) {
    for (int i = threadIdx.x; i < n_stage; i += blockDim.x) {
        int64_t t = s0 + i;
        t = t < 0 ? 0 : (t >= N ? N - 1 : t);
        dst[i] = __ldg(row + t);
    }
}

static int halo_for(double om) {
    // om^L <= 2^-60
    if (!(om > 0.0)) return 4;
    double L = ceil(60.0 * log(2.0) / -log(om));
    if (!(L < 1e9)) L = 1e9;
    return ((int)L + 3) & ~3;
}

// ---------------------------------------------------------------------------------
// EMA bank: ta.trend.EMAIndicator = close.ewm(span=w, min_periods=w, adjust=False).mean()
// (binance_ml_strategy.py:79-83): y_0 = x_0, alpha = 2/(w+1), defined for t >= w-1.
// ---------------------------------------------------------------------------------
__global__ void __launch_bounds__(IND_THREADS)
ema_bank_kernel(const float* __restrict__ x, int64_t N, int64_t ld, const __grid_constant__ BankParams prm, int P,
                int halo_max, float* __restrict__ out) {
    extern __shared__ float s_x[];  // s_x[i] = x[s0 + i]
    const int sym = blockIdx.y;
    const int64_t tile_start = (int64_t)blockIdx.x * IND_TILE;
    const int64_t tile_end = min(tile_start + (int64_t)IND_TILE, N);
    const int64_t s0 = max((int64_t)0, tile_start - halo_max);
    const int n_stage = (int)(tile_start + IND_TILE - s0);
    stage_row(x + (int64_t)sym * ld, N, s0, n_stage, s_x);
    __syncthreads();
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nwarp = blockDim.x >> 5;
    constexpr int K = 4;
    for (int pi = warp; pi < P; pi += nwarp) {
        const int w = prm.window[pi];
        float* orow = out + ((int64_t)sym * P + pi) * N;
        const double alpha = 2.0 / ((double)w + 1.0), om = 1.0 - alpha;
        AffineScan<K> sc;
        sc.init(om, lane);
        int64_t start = max(s0, tile_start - prm.halo[pi]) & ~(int64_t)3;
        double carry = (start == 0) ? (double)s_x[(int)(0 - s0)] : 0.0;  // y_{-1} := x_0 gives y_0 = x_0
        for (int64_t base = start; base < tile_end; base += 32 * K) {
            const int64_t t = base + lane * K;
            double b[K], y[K];
#pragma unroll
            for (int j = 0; j < K; ++j) b[j] = alpha * (double)s_x[min((int)(t + j - s0), n_stage - 1)];
            sc.run(b, carry, y, lane);
#pragma unroll
            for (int j = 0; j < K; ++j)
                if (t + j >= tile_start && t + j < tile_end) orow[t + j] = (t + j >= w - 1) ? (float)y[j] : nanf32();
        }
    }
}

// ---------------------------------------------------------------------------------
// MACD (ta.trend.MACD, binance_ml_strategy.py:91-94): line = EMA_fast - EMA_slow (defined where
// both are), signal = ewm(span=sign, min_periods=sign, adjust=False) of the line seeded with its
// first defined value, diff = line - signal.  One warp per CTA does the three scans in sequence.
// ---------------------------------------------------------------------------------
// (one warp; o_ef / o_es: optional outputs of the two EMAs themselves, ta.trend.EMAIndicator semantics, :79-83)
__device__ __forceinline__ void macd_tile(const float* __restrict__ x, int64_t N, int64_t ld, int fast, int slow, int sign,
                                          int halo_ema, int halo_sig, float* __restrict__ o_line, float* __restrict__ o_sig,
                                          float* __restrict__ o_diff, float* __restrict__ o_ef, float* __restrict__ o_es,
                                          double* __restrict__ s_line, int sym, int64_t tile_start) {
    const int lane = threadIdx.x & 31;
    const int64_t tile_end = min(tile_start + (int64_t)IND_TILE, N);
    const int64_t s1 = max((int64_t)0, tile_start - halo_sig) & ~(int64_t)3;   // first bar whose line is needed
    const int64_t s0 = max((int64_t)0, s1 - halo_ema) & ~(int64_t)3;           // first bar the EMAs start from
    const float* row = x + (int64_t)sym * ld;
    constexpr int K = 4;
    const double af = 2.0 / ((double)fast + 1.0), as = 2.0 / ((double)slow + 1.0), ag = 2.0 / ((double)sign + 1.0);
    AffineScan<K> sf, ss, sg;
    sf.init(1.0 - af, lane);
    ss.init(1.0 - as, lane);
    sg.init(1.0 - ag, lane);
    const int first_line = max(fast, slow) - 1;            // first defined line value
    const int first_sig = first_line + sign - 1;           // first defined signal value
    const double x0 = (double)__ldg(row);
    double cf = (s0 == 0) ? x0 : 0.0, cs = cf;
    for (int64_t base = s0; base < tile_end; base += 32 * K) {
        const int64_t t = base + lane * K;
        double bf[K], bs[K], yf[K], ys[K];
#pragma unroll
        for (int j = 0; j < K; ++j) {
            const int64_t tt = min(t + j, N - 1);
            const double v = (double)__ldg(row + tt);
            bf[j] = af * v;
            bs[j] = as * v;
        }
        sf.run(bf, cf, yf, lane);
        ss.run(bs, cs, ys, lane);
#pragma unroll
        for (int j = 0; j < K; ++j) {
            if (t + j >= s1 && t + j < tile_end) s_line[t + j - s1] = yf[j] - ys[j];
            if (o_ef && t + j >= tile_start && t + j < tile_end) {
                o_ef[(int64_t)sym * N + t + j] = (t + j >= fast - 1) ? (float)yf[j] : nanf32();
                o_es[(int64_t)sym * N + t + j] = (t + j >= slow - 1) ? (float)ys[j] : nanf32();
            }
        }
    }
    __syncwarp();
    // signal: starts at max(s1, first_line); seeded with the line itself at first_line
    int64_t g0 = max(s1, (int64_t)first_line) & ~(int64_t)3;
    if (g0 < s1) g0 = s1;
    double cg = 0.0;
    const bool seeded = (g0 <= first_line);  // this tile contains the seed bar
    for (int64_t base = g0; base < tile_end; base += 32 * K) {
        const int64_t t = base + lane * K;
        double b[K], y[K];
#pragma unroll
        for (int j = 0; j < K; ++j) {
            const int64_t tt = t + j;
            double v = (tt >= s1 && tt < tile_end) ? s_line[tt - s1] : 0.0;
            if (seeded && tt < first_line) v = 0.0;
            // seed bar: y = line  <=>  b = line with zero incoming state (scale 1 instead of alpha)
            b[j] = (seeded && tt == first_line) ? v : ag * v;
            if (tt >= tile_end) b[j] = 0.0;
        }
        sg.run(b, cg, y, lane);
#pragma unroll
        for (int j = 0; j < K; ++j) {
            const int64_t tt = t + j;
            if (tt >= tile_start && tt < tile_end) {
                const double line = s_line[tt - s1];
                const int64_t o = (int64_t)sym * N + tt;
                o_line[o] = tt >= first_line ? (float)line : nanf32();
                o_sig[o] = tt >= first_sig ? (float)y[j] : nanf32();
                o_diff[o] = tt >= first_sig ? (float)(line - y[j]) : nanf32();
            }
        }
    }
    // bars of this tile before the first signal bar that the loop above did not visit
    for (int64_t tt = tile_start + lane; tt < min(tile_end, g0); tt += 32) {
        const int64_t o = (int64_t)sym * N + tt;
        o_line[o] = tt >= first_line ? (float)s_line[tt - s1] : nanf32();
        o_sig[o] = nanf32();
        o_diff[o] = nanf32();
    }
}

__global__ void __launch_bounds__(32)
macd_kernel(const float* __restrict__ x, int64_t N, int64_t ld, int fast, int slow, int sign, int halo_ema, int halo_sig,
            float* __restrict__ o_line, float* __restrict__ o_sig, float* __restrict__ o_diff) {
    extern __shared__ double s_line[];  // line over [s1, tile_end)
    macd_tile(x, N, ld, fast, slow, sign, halo_ema, halo_sig, o_line, o_sig, o_diff, nullptr, nullptr, s_line, blockIdx.y,
              (int64_t)blockIdx.x * IND_TILE);
}

// ---------------------------------------------------------------------------------
// Block-wide inclusive prefix sum of n doubles in shared memory (n <= IND_THREADS * 16).
// ---------------------------------------------------------------------------------
__device__ void block_prefix_sum(double* __restrict__ s, int n, double* __restrict__ s_warp) {
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int per = (n + blockDim.x - 1) / blockDim.x;
    const int lo = min(tid * per, n), hi = min(lo + per, n);
    double run = 0.0;
    for (int i = lo; i < hi; ++i) { run += s[i]; s[i] = run; }
    double inc = run;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const double up = shfl_up_d(inc, d);
        if (lane >= d) inc += up;
    }
    if (lane == 31) s_warp[warp] = inc;
    __syncthreads();
    if (warp == 0) {
        double v = lane < (int)(blockDim.x >> 5) ? s_warp[lane] : 0.0;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const double up = shfl_up_d(v, d);
            if (lane >= d) v += up;
        }
        if (lane < (int)(blockDim.x >> 5)) s_warp[lane] = v;
    }
    __syncthreads();
    const double off = (inc - run) + (warp > 0 ? s_warp[warp - 1] : 0.0);
    for (int i = lo; i < hi; ++i) s[i] += off;
    __syncthreads();
}

// ---------------------------------------------------------------------------------
// SMA bank (ta.trend.SMAIndicator = rolling(w, min_periods=w).mean(); :67-76).
// ---------------------------------------------------------------------------------
__global__ void __launch_bounds__(IND_THREADS)
sma_bank_kernel(const float* __restrict__ x, int64_t N, int64_t ld, const __grid_constant__ BankParams prm, int P,
                int halo_max, float* __restrict__ out) {
    extern __shared__ double s_pre[];  // s_pre[i+1] = sum_{k<=i} (x[s0+k] - c), s_pre[0] = 0
    __shared__ double s_warp[32];
    const int sym = blockIdx.y;
    const int64_t tile_start = (int64_t)blockIdx.x * IND_TILE;
    const int64_t tile_end = min(tile_start + (int64_t)IND_TILE, N);
    const int64_t s0 = max((int64_t)0, tile_start - halo_max);
    const int n_stage = (int)(tile_end - s0);
    const float* row = x + (int64_t)sym * ld;
    const double c = (double)__ldg(row + tile_start);  // tile offset keeps the prefix small
    if (threadIdx.x == 0) s_pre[0] = 0.0;
    for (int i = threadIdx.x; i < n_stage; i += blockDim.x) s_pre[i + 1] = (double)__ldg(row + s0 + i) - c;
    __syncthreads();
    block_prefix_sum(s_pre + 1, n_stage, s_warp);
    for (int pi = 0; pi < P; ++pi) {
        const int w = prm.window[pi];
        float* orow = out + ((int64_t)sym * P + pi) * N;
        for (int64_t t = tile_start + threadIdx.x; t < tile_end; t += blockDim.x) {
            float v = nanf32();
            if (t >= w - 1) {
                const int i = (int)(t - s0);
                v = (float)((s_pre[i + 1] - s_pre[i + 1 - w]) / (double)w + c);
            }
            orow[t] = v;
        }
    }
}

// ---------------------------------------------------------------------------------
// Bollinger bands (ta.volatility.BollingerBands(close, 20, 2); :148-156):
// mid = rolling mean, std = rolling std(ddof=0), high/low = mid +- k*std,
// width = (high-low)/mid, position = (close-low)/(high-low) with NaN where the range is 0.
// ---------------------------------------------------------------------------------
__global__ void __launch_bounds__(IND_THREADS)
bollinger_kernel(const float* __restrict__ x, int64_t N, int64_t ld, int w, double kdev, float* __restrict__ o_high,
                 float* __restrict__ o_mid, float* __restrict__ o_low, float* __restrict__ o_width,
                 float* __restrict__ o_pos) {
    extern __shared__ double s_buf[];  // [0, n+1): prefix of d, [n+1, 2n+2): prefix of d^2
    __shared__ double s_warp[32];
    const int sym = blockIdx.y;
    const int64_t tile_start = (int64_t)blockIdx.x * IND_TILE;
    const int64_t tile_end = min(tile_start + (int64_t)IND_TILE, N);
    const int64_t s0 = max((int64_t)0, tile_start - (w - 1));
    const int n = (int)(tile_end - s0);
    double* p1 = s_buf;
    double* p2 = s_buf + (IND_TILE + IND_MAX_WINDOW + 1);
    const float* row = x + (int64_t)sym * ld;
    const double c = (double)__ldg(row + tile_start);
    if (threadIdx.x == 0) { p1[0] = 0.0; p2[0] = 0.0; }
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
        const double d = (double)__ldg(row + s0 + i) - c;
        p1[i + 1] = d;
        p2[i + 1] = d * d;
    }
    __syncthreads();
    block_prefix_sum(p1 + 1, n, s_warp);
    block_prefix_sum(p2 + 1, n, s_warp);
    for (int64_t t = tile_start + threadIdx.x; t < tile_end; t += blockDim.x) {
        const int64_t o = (int64_t)sym * N + t;
        if (t < w - 1) {
            o_high[o] = o_mid[o] = o_low[o] = o_width[o] = o_pos[o] = nanf32();
            continue;
        }
        const int i = (int)(t - s0);
        const double m1 = (p1[i + 1] - p1[i + 1 - w]) / (double)w;   // mean of d
        const double m2 = (p2[i + 1] - p2[i + 1 - w]) / (double)w;   // mean of d^2
        double var = m2 - m1 * m1;
        if (var < 0.0) var = 0.0;
        const double sd = sqrt(var), mid = m1 + c;
        const double hi = mid + kdev * sd, lo = mid - kdev * sd;
        const double rng = hi - lo;
        const double close = (double)__ldg(row + t);
        o_high[o] = (float)hi;
        o_mid[o] = (float)mid;
        o_low[o] = (float)lo;
        o_width[o] = (float)(rng / mid);
        o_pos[o] = rng == 0.0 ? nanf32() : (float)((close - lo) / rng);
    }
}

// ---------------------------------------------------------------------------------
// Rolling extrema helpers + stochastic / Williams %R / Ichimoku.
// ---------------------------------------------------------------------------------
__device__ __forceinline__ float window_max(const float* __restrict__ s, int i, int w) {
    float m = s[i];
    for (int k = 1; k < w; ++k) m = fmaxf(m, s[i - k]);
    return m;
}
__device__ __forceinline__ float window_min(const float* __restrict__ s, int i, int w) {
    float m = s[i];
    for (int k = 1; k < w; ++k) m = fminf(m, s[i - k]);
    return m;
}

// mode 0: stochastic (%K into o_a, %D = rolling mean(smooth) of %K into o_b)   :121-127
// mode 1: Williams %R into o_a                                                 :135-140
// mode 2: Ichimoku a, b (w1 conversion, w2 base, w3 span b)                    :102-104
// (whole CTA; s_hl: 3 (IND_TILE + 2 IND_MAX_WINDOW) floats of shared memory -- highs, lows, %K scratch; ends with every
// thread past its last shared-memory access only after the caller's next barrier)
__device__ __forceinline__ void extrema_tile(const float* __restrict__ high, const float* __restrict__ low, const float* __restrict__ close,
                                             int64_t N, int64_t ld, int mode, int w1, int w2, int w3, float* __restrict__ o_a,
                                             float* __restrict__ o_b, float* __restrict__ s_hl, int sym, int64_t tile_start) {
    const int64_t tile_end = min(tile_start + (int64_t)IND_TILE, N);
    const int wmax = max(w1, max(w2, w3));
    const int extra = (mode == 0) ? (w2 - 1) : 0;  // %D needs %K of the previous smooth-1 bars
    const int64_t s0 = max((int64_t)0, tile_start - (wmax - 1) - extra);
    const int n = (int)(tile_end - s0);
    float* sh = s_hl;
    float* sl = s_hl + (IND_TILE + 2 * IND_MAX_WINDOW);
    float* sk = sl + (IND_TILE + 2 * IND_MAX_WINDOW);
    stage_row(high + (int64_t)sym * ld, N, s0, n, sh);
    stage_row(low + (int64_t)sym * ld, N, s0, n, sl);
    __syncthreads();
    const float* crow = close ? close + (int64_t)sym * ld : nullptr;
    if (mode == 0) {
        for (int i = threadIdx.x; i < n; i += blockDim.x) {
            const int64_t t = s0 + i;
            float k = nanf32();
            if (i >= w1 - 1) {  // (s0 == 0: same as t >= w1-1; s0 > 0: the window must lie inside the staged halo)
                const double lo = (double)window_min(sl, i, w1), hi = (double)window_max(sh, i, w1);
                k = (float)(100.0 * ((double)__ldg(crow + t) - lo) / (hi - lo));   // 0/0 -> NaN as in pandas
            }
            sk[i] = k;
        }
        __syncthreads();
        for (int64_t t = tile_start + threadIdx.x; t < tile_end; t += blockDim.x) {
            const int i = (int)(t - s0);
            const int64_t o = (int64_t)sym * N + t;
            o_a[o] = sk[i];
            float d = nanf32();
            if (t >= w1 - 1 + w2 - 1) {
                // %D over the float64 %K values (recomputed: the reference averages float64 %K)
                double acc = 0.0;
                for (int k = 0; k < w2; ++k) {
                    const int ii = i - k;
                    const double lo = (double)window_min(sl, ii, w1), hi = (double)window_max(sh, ii, w1);
                    acc += 100.0 * ((double)__ldg(crow + s0 + ii) - lo) / (hi - lo);
                }
                d = (float)(acc / (double)w2);
            }
            o_b[o] = d;
        }
    } else if (mode == 1) {
        for (int64_t t = tile_start + threadIdx.x; t < tile_end; t += blockDim.x) {
            const int i = (int)(t - s0);
            float v = nanf32();
            if (t >= w1 - 1) {
                const double hi = (double)window_max(sh, i, w1), lo = (double)window_min(sl, i, w1);
                v = (float)(-100.0 * (hi - (double)__ldg(crow + t)) / (hi - lo));
            }
            o_a[(int64_t)sym * N + t] = v;
        }
    } else {
        for (int64_t t = tile_start + threadIdx.x; t < tile_end; t += blockDim.x) {
            const int i = (int)(t - s0);
            const int64_t o = (int64_t)sym * N + t;
            float a = nanf32(), b = nanf32();
            if (t >= max(w1, w2) - 1) {
                const double conv = 0.5 * ((double)window_max(sh, i, w1) + (double)window_min(sl, i, w1));
                const double base = 0.5 * ((double)window_max(sh, i, w2) + (double)window_min(sl, i, w2));
                a = (float)(0.5 * (conv + base));
            }
            if (t >= w3 - 1) b = (float)(0.5 * ((double)window_max(sh, i, w3) + (double)window_min(sl, i, w3)));
            o_a[o] = a;
            o_b[o] = b;
        }
    }
}

__global__ void __launch_bounds__(IND_THREADS)
extrema_kernel(const float* __restrict__ high, const float* __restrict__ low, const float* __restrict__ close,
               int64_t N, int64_t ld, int mode, int w1, int w2, int w3, float* __restrict__ o_a, float* __restrict__ o_b) {
    extern __shared__ float s_hl[];  // [halo + tile] highs, then lows, then %K scratch
    extrema_tile(high, low, close, N, ld, mode, w1, w2, w3, o_a, o_b, s_hl, blockIdx.y, (int64_t)blockIdx.x * IND_TILE);
}

// ---------------------------------------------------------------------------------
// ATR bank (ta.volatility.AverageTrueRange; :164): TR_t = max(h-l, |h-c_{t-1}|, |l-c_{t-1}|),
// TR_0 = h_0-l_0; atr[t<w-1] = 0, atr[w-1] = mean(TR[0:w]), atr[i] = (atr[i-1](w-1)+TR[i])/w.
// ---------------------------------------------------------------------------------
// (whole CTA; `tr`: (halo_max + IND_TILE + IND_MAX_WINDOW + 8) doubles of shared memory; window i of `prm` goes to warp i % nwarp
// and is written to out + ((sym * P + i) * N))
__device__ __forceinline__ void atr_tile(const float* __restrict__ high, const float* __restrict__ low, const float* __restrict__ close,
                                         int64_t N, int64_t ld, const BankParams& prm, int P, int halo_max,
                                         float* __restrict__ out, double* __restrict__ tr, int sym, int64_t tile_start) {
    const int64_t tile_end = min(tile_start + (int64_t)IND_TILE, N);
    int64_t s0 = max((int64_t)0, tile_start - halo_max) & ~(int64_t)3;
    if (s0 < IND_MAX_WINDOW) s0 = 0;  // a pass that crosses a seed bar t = w-1 needs TR from bar 0
    const int n_stage = (int)(tile_start + IND_TILE - s0);
    const float* hr = high + (int64_t)sym * ld;
    const float* lr = low + (int64_t)sym * ld;
    const float* cr = close + (int64_t)sym * ld;
    for (int i = threadIdx.x; i < n_stage; i += blockDim.x) {
        const int64_t t = s0 + i;
        double v = 0.0;
        if (t < N) {
            const double h = (double)__ldg(hr + t), l = (double)__ldg(lr + t);
            v = h - l;
            if (t > 0) {
                const double pc = (double)__ldg(cr + t - 1);
                v = fmax(v, fmax(fabs(h - pc), fabs(l - pc)));
            }
        }
        tr[i] = v;
    }
    __syncthreads();
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nwarp = blockDim.x >> 5;
    constexpr int K = 4;
    for (int pi = warp; pi < P; pi += nwarp) {
        const int w = prm.window[pi];
        float* orow = out + ((int64_t)sym * P + pi) * N;
        const double alpha = 1.0 / (double)w, om = ((double)w - 1.0) / (double)w;
        AffineScan<K> sc;
        sc.init(om, lane);
        int64_t start = max(s0, tile_start - prm.halo[pi]) & ~(int64_t)3;
        const bool has_seed = (start <= w - 1);     // this pass crosses the seed bar t = w-1
        double seed = 0.0;
        if (has_seed && w - 1 < N) {
            for (int k = 0; k < w; ++k) seed += tr[(int)(k - s0)];   // s0 == 0 whenever has_seed
            seed /= (double)w;
        }
        if (has_seed) start = 0;
        double carry = 0.0;
        for (int64_t base = start; base < tile_end; base += 32 * K) {
            const int64_t t = base + lane * K;
            double b[K], y[K];
#pragma unroll
            for (int j = 0; j < K; ++j) {
                const int64_t tt = t + j;
                double v = alpha * tr[min((int)(tt - s0), n_stage - 1)];
                if (has_seed) v = tt < w - 1 ? 0.0 : (tt == w - 1 ? seed : v);   // zeros, then the seed, then the recurrence
                b[j] = v;
            }
            sc.run(b, carry, y, lane);
#pragma unroll
            for (int j = 0; j < K; ++j)
                if (t + j >= tile_start && t + j < tile_end) orow[t + j] = (t + j >= w - 1) ? (float)y[j] : 0.0f;
        }
    }
}

__global__ void __launch_bounds__(IND_THREADS)
atr_bank_kernel(const float* __restrict__ high, const float* __restrict__ low, const float* __restrict__ close,
                int64_t N, int64_t ld, const __grid_constant__ BankParams prm, int P, int halo_max,
                float* __restrict__ out) {
    extern __shared__ float s_tr[];  // true range over [s0, tile_end), float64
    atr_tile(high, low, close, N, ld, prm, P, halo_max, out, reinterpret_cast<double*>(s_tr), blockIdx.y, (int64_t)blockIdx.x * IND_TILE);
}

// ---------------------------------------------------------------------------------
// VWAP (ta.volume.VolumeWeightedAveragePrice, window 14; :173-179):
// sum_w(tp*v)/sum_w(v), tp = (h+l+c)/3.
// ---------------------------------------------------------------------------------
// (whole CTA; s_buf: 2 (IND_TILE + IND_MAX_WINDOW + 1) doubles, s_warp: 32 doubles of shared memory)
__device__ __forceinline__ void vwap_tile(const float* __restrict__ high, const float* __restrict__ low, const float* __restrict__ close,
                                          const float* __restrict__ volume, int64_t N, int64_t ld, int w, float* __restrict__ out,
                                          double* __restrict__ s_buf, double* __restrict__ s_warp, int sym, int64_t tile_start) {
    const int64_t tile_end = min(tile_start + (int64_t)IND_TILE, N);
    const int64_t s0 = max((int64_t)0, tile_start - (w - 1));
    const int n = (int)(tile_end - s0);
    double* p1 = s_buf;
    double* p2 = s_buf + (IND_TILE + IND_MAX_WINDOW + 1);
    const int64_t ro = (int64_t)sym * ld;
    if (threadIdx.x == 0) { p1[0] = 0.0; p2[0] = 0.0; }
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
        const int64_t t = s0 + i;
        const double tp = ((double)__ldg(high + ro + t) + (double)__ldg(low + ro + t) + (double)__ldg(close + ro + t)) / 3.0;
        const double v = (double)__ldg(volume + ro + t);
        p1[i + 1] = tp * v;
        p2[i + 1] = v;
    }
    __syncthreads();
    block_prefix_sum(p1 + 1, n, s_warp);
    block_prefix_sum(p2 + 1, n, s_warp);
    for (int64_t t = tile_start + threadIdx.x; t < tile_end; t += blockDim.x) {
        float v = nanf32();
        if (t >= w - 1) {
            const int i = (int)(t - s0);
            v = (float)((p1[i + 1] - p1[i + 1 - w]) / (p2[i + 1] - p2[i + 1 - w]));
        }
        out[(int64_t)sym * N + t] = v;
    }
}

__global__ void __launch_bounds__(IND_THREADS)
vwap_kernel(const float* __restrict__ high, const float* __restrict__ low, const float* __restrict__ close,
            const float* __restrict__ volume, int64_t N, int64_t ld, int w, float* __restrict__ out) {
    extern __shared__ double s_buf[];
    __shared__ double s_warp[32];
    vwap_tile(high, low, close, volume, N, ld, w, out, s_buf, s_warp, blockIdx.y, (int64_t)blockIdx.x * IND_TILE);
}

// ---------------------------------------------------------------------------------
// NaN policy of TechnicalAnalyzer._handle_nan_values (:28-38): ffill, then bfill, then 0.
// Pass 1: per (row, tile) last / first non-NaN value.  Pass 2: fill inside each tile with the
// carry from the nearest earlier tile (or, before the first valid value, the first valid value).
// ---------------------------------------------------------------------------------
constexpr int NF_TILE = 4096;

__global__ void __launch_bounds__(256)
nanfill_scan_kernel(const float* __restrict__ x, int64_t N, int tiles, float* __restrict__ t_last, float* __restrict__ t_first,
                    float* __restrict__ t_nans) {
    const int row = blockIdx.y, tile = blockIdx.x;
    const int64_t lo = (int64_t)tile * NF_TILE, hi = min(lo + (int64_t)NF_TILE, N);
    const float* r = x + (int64_t)row * N;
    int last = -1, first = 0x7fffffff, nans = 0;
    for (int64_t t = lo + threadIdx.x; t < hi; t += blockDim.x) {
        if (!isnan(r[t])) { last = max(last, (int)(t - lo)); first = min(first, (int)(t - lo)); }
        else ++nans;
    }
    __shared__ int s_last[8], s_first[8], s_nans[8];
    last = __reduce_max_sync(FULL, last);
    first = __reduce_min_sync(FULL, first);
    nans = __reduce_add_sync(FULL, nans);
    if ((threadIdx.x & 31) == 0) { s_last[threadIdx.x >> 5] = last; s_first[threadIdx.x >> 5] = first; s_nans[threadIdx.x >> 5] = nans; }
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int i = 1; i < 8; ++i) { last = max(last, s_last[i]); first = min(first, s_first[i]); nans += s_nans[i]; }
        last = max(last, s_last[0]);
        first = min(first, s_first[0]);
        t_last[(int64_t)row * tiles + tile] = last >= 0 ? r[lo + last] : nanf32();
        t_first[(int64_t)row * tiles + tile] = first != 0x7fffffff ? r[lo + first] : nanf32();
        t_nans[(int64_t)row * tiles + tile] = (float)nans;      // almost every tile has none: the apply pass skips it
    }
}

__global__ void __launch_bounds__(256)
nanfill_apply_kernel(float* __restrict__ x, int64_t N, int tiles, const float* __restrict__ t_last,
                     const float* __restrict__ t_first, const float* __restrict__ t_nans) {
    const int row = blockIdx.y;
    __shared__ float s_carry, s_firstvalid;
    __shared__ int s_idx[NF_TILE];
    // a CTA walks tiles blockIdx.x, blockIdx.x + gridDim.x, ...; almost all of them hold no NaN and are skipped
    for (int tile = blockIdx.x; tile < tiles; tile += gridDim.x) {
    if (t_nans[(int64_t)row * tiles + tile] == 0.0f) continue;
    __syncthreads();
    const int64_t lo = (int64_t)tile * NF_TILE, hi = min(lo + (int64_t)NF_TILE, N);
    float* r = x + (int64_t)row * N;
    if (threadIdx.x == 0) {
        float c = nanf32();
        for (int k = tile - 1; k >= 0 && isnan(c); --k) c = t_last[(int64_t)row * tiles + k];
        float f = nanf32();
        for (int k = 0; k < tiles && isnan(f); ++k) f = t_first[(int64_t)row * tiles + k];
        s_carry = c;
        s_firstvalid = f;
    }
    // index of the last valid element at or before each position (block-level max-scan, done per warp chunk)
    const int n = (int)(hi - lo);
    for (int i = threadIdx.x; i < n; i += blockDim.x) s_idx[i] = isnan(r[lo + i]) ? -1 : i;
    __syncthreads();
    if (threadIdx.x < 32) {
        // 32 lanes x 128 contiguous positions: serial running max per lane, then a warp scan of lane totals
        const int per = NF_TILE / 32, a = threadIdx.x * per, b = min(a + per, n);
        int run = -1;
        for (int i = a; i < b; ++i) { run = max(run, s_idx[i]); s_idx[i] = run; }
        int inc = run;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const int up = __shfl_up_sync(FULL, inc, d);
            if ((int)threadIdx.x >= d) inc = max(inc, up);
        }
        const int before = __shfl_up_sync(FULL, inc, 1);
        if (threadIdx.x > 0 && before >= 0)
            for (int i = a; i < b; ++i) s_idx[i] = max(s_idx[i], before);
    }
    __syncthreads();
    const float carry = s_carry, fv = s_firstvalid;
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
        float v = r[lo + i];
        if (isnan(v)) {
            const int j = s_idx[i];
            if (j >= 0) v = r[lo + j];            // ffill inside the tile (source is a valid element, never rewritten)
            else if (!isnan(carry)) v = carry;    // ffill across tiles
            else if (!isnan(fv)) v = fv;          // bfill before the first valid value
            else v = 0.0f;                        // all-NaN column
            r[lo + i] = v;
        }
    }
    }
}

// ---------------------------------------------------------------------------------
// TechnicalAnalyzer._calculate_all_indicators (binance_ml_strategy.py:40-182) in three launches.  Each launch stages its
// inputs once per (symbol, tile) and writes every column that depends on them, with the reference's own windows:
//   A  close                     -> ema_12, ema_26, macd, macd_signal, macd_diff (one warp), rsi_14 (second warp)
//   B  close                     -> sma_20, sma_50, sma_200, bb_high, bb_mid, bb_low, bb_width, bb_position
//   C  high, low, close, volume  -> stoch_k, stoch_d, williams_r, ichimoku_a, ichimoku_b, atr_14, vwap_14
// Columns are [S][N] blocks of one [21][S][N] allocation in the order of b200bt_analyzer_column (include/b200bt.h).  The
// leading undefined bars (t < window - 1) of the columns that cannot be undefined anywhere else are filled by the CTA of
// tile 0 itself (bfill with the first defined value, 0 for a series shorter than the window: `_handle_nan_values` :28-38);
// the five columns that can be undefined in mid-series (zero high-low range, zero Bollinger range, zero volume) sit at the
// end of the allocation and go through the general ffill / bfill kernels in ONE batched call.
// ---------------------------------------------------------------------------------
struct LeadFill { float* col[8]; int first[8]; int n; };

// CTA of tile 0, after a barrier: col[t] = col[first] for t < first (0 when the series ends before `first`)
__device__ __forceinline__ void lead_fill(const LeadFill& lf, int sym, int64_t N) {
    for (int c = 0; c < lf.n; ++c) {
        float* o = lf.col[c] + (int64_t)sym * N;
        const int f = lf.first[c];
        const float v = f < N ? o[f] : 0.0f;
        for (int64_t t = threadIdx.x; t < min((int64_t)f, N); t += blockDim.x) o[t] = v;
    }
}

__global__ void __launch_bounds__(64)
analyzer_a_kernel(const float* __restrict__ x, int64_t N, int64_t ld, int fast, int slow, int sign, int halo_ema, int halo_sig,
                  int w_rsi, const double2* __restrict__ rsi_seam, float* __restrict__ o_ef, float* __restrict__ o_es,
                  float* __restrict__ o_line, float* __restrict__ o_sig, float* __restrict__ o_diff, float* __restrict__ o_rsi, const LeadFill lf) {
    extern __shared__ double s_line[];
    const int sym = blockIdx.y, lane = threadIdx.x & 31;
    const int64_t tile_start = (int64_t)blockIdx.x * IND_TILE, tile_end = min(tile_start + (int64_t)IND_TILE, N);
    if (threadIdx.x < 32) {
        macd_tile(x, N, ld, fast, slow, sign, halo_ema, halo_sig, o_line, o_sig, o_diff, o_ef, o_es, s_line, sym, tile_start);
    } else {
        // RSI (ta.momentum.RSIIndicator, :112): Wilder averages of the up / down moves, y0 = x0 (both 0 at bar 0), started
        // from their true state at the tile's first bar
        const float* row = x + (int64_t)sym * ld;
        constexpr int K = 4;
        const double alpha = 1.0 / (double)w_rsi;
        AffineScan<K> sc;
        sc.init(1.0 - alpha, lane);
        double cu = 0.0, cd = 0.0;
        if (blockIdx.x > 0) {
            const double2 c = rsi_seam[(int64_t)sym * (gridDim.x - 1) + blockIdx.x - 1];
            cu = c.x;
            cd = c.y;
        }
        for (int64_t base = tile_start; base < tile_end; base += 32 * K) {
            const int64_t t = base + lane * K;
            double xs[K + 1], bu[K], bd[K], yu[K], yd[K];
#pragma unroll
            for (int j = 0; j <= K; ++j) {
                int64_t tt = t - 1 + j;
                tt = tt < 0 ? 0 : (tt >= N ? N - 1 : tt);
                xs[j] = (double)__ldg(row + tt);
            }
#pragma unroll
            for (int j = 0; j < K; ++j) {
                const double df = xs[j + 1] - xs[j];
                bu[j] = alpha * (df > 0.0 ? df : 0.0);
                bd[j] = alpha * (df < 0.0 ? -df : 0.0);
            }
            sc.run(bu, cu, yu, lane);
            sc.run(bd, cd, yd, lane);
#pragma unroll
            for (int j = 0; j < K; ++j)
                if (t + j < tile_end) {
                    o_rsi[(int64_t)sym * N + t + j] = (t + j >= w_rsi - 1) ? rsi_value(yu[j], yd[j]) : nanf32();
                }
        }
    }
    if (tile_start == 0) {
        __syncthreads();
        lead_fill(lf, sym, N);
    }
}

__global__ void __launch_bounds__(IND_THREADS)
analyzer_b_kernel(const float* __restrict__ x, int64_t N, int64_t ld, int w0, int w1, int w2, int w_bb, double kdev,
                  float* __restrict__ o_s0, float* __restrict__ o_s1, float* __restrict__ o_s2, float* __restrict__ o_high,
                  float* __restrict__ o_mid, float* __restrict__ o_low, float* __restrict__ o_width, float* __restrict__ o_pos,
                  int halo, const LeadFill lf) {
    extern __shared__ double s_buf[];   // prefix of d = x - c, then prefix of d^2 (IND_TILE + IND_MAX_WINDOW + 1 each)
    __shared__ double s_warp[32];
    const int sym = blockIdx.y;
    const int64_t tile_start = (int64_t)blockIdx.x * IND_TILE, tile_end = min(tile_start + (int64_t)IND_TILE, N);
    const int64_t s0 = max((int64_t)0, tile_start - halo);
    const int n = (int)(tile_end - s0);
    double* p1 = s_buf;
    double* p2 = s_buf + (IND_TILE + IND_MAX_WINDOW + 1);
    const float* row = x + (int64_t)sym * ld;
    const double c = (double)__ldg(row + tile_start);   // tile offset keeps the prefixes small (sum of squares without cancellation)
    if (threadIdx.x == 0) { p1[0] = 0.0; p2[0] = 0.0; }
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
        const double d = (double)__ldg(row + s0 + i) - c;
        p1[i + 1] = d;
        p2[i + 1] = d * d;
    }
    __syncthreads();
    block_prefix_sum(p1 + 1, n, s_warp);
    block_prefix_sum(p2 + 1, n, s_warp);
    const int ws[3] = {w0, w1, w2};
    float* const os[3] = {o_s0, o_s1, o_s2};
    for (int64_t t = tile_start + threadIdx.x; t < tile_end; t += blockDim.x) {
        const int i = (int)(t - s0);
        const int64_t o = (int64_t)sym * N + t;
#pragma unroll
        for (int k = 0; k < 3; ++k)      // ta.trend.SMAIndicator (:67-76)
            os[k][o] = (t >= ws[k] - 1) ? (float)((p1[i + 1] - p1[i + 1 - ws[k]]) / (double)ws[k] + c) : nanf32();
        if (t < w_bb - 1) {              // ta.volatility.BollingerBands (:148-156)
            o_high[o] = o_mid[o] = o_low[o] = o_width[o] = o_pos[o] = nanf32();
            continue;
        }
        const double m1 = (p1[i + 1] - p1[i + 1 - w_bb]) / (double)w_bb;
        const double m2 = (p2[i + 1] - p2[i + 1 - w_bb]) / (double)w_bb;
        double var = m2 - m1 * m1;
        if (var < 0.0) var = 0.0;
        const double sd = sqrt(var), mid = m1 + c;
        const double hi = mid + kdev * sd, lo = mid - kdev * sd;
        const double rng = hi - lo;
        const double close = (double)__ldg(row + t);
        o_high[o] = (float)hi;
        o_mid[o] = (float)mid;
        o_low[o] = (float)lo;
        o_width[o] = (float)(rng / mid);
        o_pos[o] = rng == 0.0 ? nanf32() : (float)((close - lo) / rng);
    }
    if (tile_start == 0) {
        __syncthreads();
        lead_fill(lf, sym, N);
    }
}

// C: one backward walk of the staged highs / lows per bar serves every window (the reference's are nested: 9 <= 14 <= 26 <= 52),
// %D averages the float64 %K values kept in shared memory, the ATR recurrence runs on all eight warps (a 256-bar sub-tile
// each, its own warm-up halo) instead of one, VWAP on block-wide prefix sums.  Phases reuse the shared memory.
__global__ void __launch_bounds__(IND_THREADS)
analyzer_c_kernel(const float* __restrict__ high, const float* __restrict__ low, const float* __restrict__ close,
                  const float* __restrict__ volume, int64_t N, int64_t ld, int w_st, int smooth, int i1, int i2, int i3,
                  int w_atr, int atr_halo, int w_vwap, float* __restrict__ o_k, float* __restrict__ o_d,
                  float* __restrict__ o_wr, float* __restrict__ o_ia, float* __restrict__ o_ib, float* __restrict__ o_atr,
                  float* __restrict__ o_vwap, const LeadFill lf) {
    extern __shared__ __align__(16) unsigned char s_raw[];
    __shared__ double s_warp[32];
    const int sym = blockIdx.y;
    const int64_t tile_start = (int64_t)blockIdx.x * IND_TILE, tile_end = min(tile_start + (int64_t)IND_TILE, N);
    const int64_t ro = (int64_t)sym * ld;
    // ---- phase 1: window extrema -> stochastic %K / %D, Williams %R, Ichimoku a / b ----
    {
        const int halo = max(i3 - 1, w_st - 1 + smooth - 1);
        const int64_t s0 = max((int64_t)0, tile_start - halo);
        const int n = (int)(tile_end - s0);
        constexpr int CAP = IND_TILE + 256;                         // (the host checks halo <= 256)
        float* sh = reinterpret_cast<float*>(s_raw);
        float* sl = sh + CAP;
        float* sc = sl + CAP;
        double* skd = reinterpret_cast<double*>(sc + CAP);          // float64 %K of the staged bars
        stage_row(high + ro, N, s0, n, sh);
        stage_row(low + ro, N, s0, n, sl);
        stage_row(close + ro, N, s0, n, sc);
        __syncthreads();
        for (int i = threadIdx.x; i < n; i += blockDim.x) {
            const int64_t t = s0 + i;
            // running (max high, min low) over the last k bars, captured at the windows in ascending order
            float mh = -INFINITY, ml = INFINITY;
            int k = 0;
            const int have = i + 1;                                  // staged bars at or before this one
            auto upto = [&](int w) { const int lim = min(w, have); for (; k < lim; ++k) { mh = fmaxf(mh, sh[i - k]); ml = fminf(ml, sl[i - k]); } };
            upto(i1);
            const double h1 = (double)mh, l1 = (double)ml;
            upto(w_st);
            const double hs = (double)mh, ls = (double)ml;
            upto(i2);
            const double h2 = (double)mh, l2 = (double)ml;
            upto(i3);
            const double h3 = (double)mh, l3 = (double)ml;
            const double c = (double)sc[i];
            // (s0 == 0: "i >= w - 1" is "t >= w - 1"; s0 > 0: every window lies inside the staged halo)
            const double kk = (i >= w_st - 1) ? 100.0 * (c - ls) / (hs - ls) : (double)nanf32();       // 0/0 -> NaN as in pandas
            skd[i] = kk;
            if (t >= tile_start) {
                const int64_t o = (int64_t)sym * N + t;
                o_k[o] = (float)kk;
                o_wr[o] = (t >= w_st - 1) ? (float)(-100.0 * (hs - c) / (hs - ls)) : nanf32();
                float a = nanf32(), b = nanf32();
                if (t >= max(i1, i2) - 1) a = (float)(0.5 * (0.5 * (h1 + l1) + 0.5 * (h2 + l2)));
                if (t >= i3 - 1) b = (float)(0.5 * (h3 + l3));
                o_ia[o] = a;
                o_ib[o] = b;
            }
        }
        __syncthreads();
        for (int64_t t = tile_start + threadIdx.x; t < tile_end; t += blockDim.x) {
            const int i = (int)(t - s0);
            float d = nanf32();
            if (t >= w_st - 1 + smooth - 1) {
                double acc = 0.0;
                for (int q = 0; q < smooth; ++q) acc += skd[i - q];
                d = (float)(acc / (double)smooth);
            }
            o_d[(int64_t)sym * N + t] = d;
        }
        __syncthreads();
    }
    // ---- phase 2: ATR (ta.volatility.AverageTrueRange; :164), a 256-bar sub-tile per warp ----
    {
        double* tr = reinterpret_cast<double*>(s_raw);
        int64_t s0 = max((int64_t)0, tile_start - atr_halo) & ~(int64_t)3;
        if (s0 < IND_MAX_WINDOW) s0 = 0;                             // a pass that crosses the seed bar t = w-1 needs TR from bar 0
        const int n_stage = (int)(tile_start + IND_TILE - s0);
        for (int i = threadIdx.x; i < n_stage; i += blockDim.x) {
            const int64_t t = s0 + i;
            double v = 0.0;
            if (t < N) {
                const double h = (double)__ldg(high + ro + t), l = (double)__ldg(low + ro + t);
                v = h - l;
                if (t > 0) {
                    const double pc = (double)__ldg(close + ro + t - 1);
                    v = fmax(v, fmax(fabs(h - pc), fabs(l - pc)));
                }
            }
            tr[i] = v;
        }
        __syncthreads();
        const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nwarp = blockDim.x >> 5;
        constexpr int K = 4;
        const int w = w_atr;
        const double alpha = 1.0 / (double)w, om = ((double)w - 1.0) / (double)w;
        AffineScan<K> scn;
        scn.init(om, lane);
        const int sub = IND_TILE / (int)nwarp;
        const int64_t sub_start = tile_start + (int64_t)warp * sub, sub_end = min(sub_start + sub, tile_end);
        if (sub_start < sub_end) {
            int64_t start = max(s0, sub_start - atr_halo) & ~(int64_t)3;
            const bool has_seed = (start <= w - 1);                  // this pass crosses the seed bar t = w-1
            double seed = 0.0;
            if (has_seed && w - 1 < N) {
                for (int q = 0; q < w; ++q) seed += tr[(int)(q - s0)];   // s0 == 0 whenever has_seed
                seed /= (double)w;
            }
            if (has_seed) start = 0;
            double carry = 0.0;
            for (int64_t base = start; base < sub_end; base += 32 * K) {
                const int64_t t = base + lane * K;
                double b[K], y[K];
#pragma unroll
                for (int j = 0; j < K; ++j) {
                    const int64_t tt = t + j;
                    double v = alpha * tr[min((int)(tt - s0), n_stage - 1)];
                    if (has_seed) v = tt < w - 1 ? 0.0 : (tt == w - 1 ? seed : v);   // zeros, then the seed, then the recurrence
                    b[j] = v;
                }
                scn.run(b, carry, y, lane);
#pragma unroll
                for (int j = 0; j < K; ++j)
                    if (t + j >= sub_start && t + j < sub_end) o_atr[(int64_t)sym * N + t + j] = (t + j >= w - 1) ? (float)y[j] : 0.0f;
            }
        }
        __syncthreads();
    }
    // ---- phase 3: VWAP ----
    vwap_tile(high, low, close, volume, N, ld, w_vwap, o_vwap, reinterpret_cast<double*>(s_raw), s_warp, sym, tile_start);
    if (tile_start == 0) {
        __syncthreads();
        lead_fill(lf, sym, N);
    }
}

}  // namespace b200bt

using namespace b200bt;

#define IND_COMMON_CHECKS(name)                                                                         \
    B200BT_REQUIRE(S > 0 && N > 0 && ld >= N, B200BT_EINVAL, name ": bad sizes S=%d N=%lld", S, (long long)N); \
    {                                                                                                   \
        int rc__ = check_device();                                                                      \
        if (rc__) return rc__;                                                                          \
    }

// the EMA bank gives each window to a warp: few windows -> small CTAs, so that the SM fills with busy warps
// (measured: 102 -> 85 us for two spans; the ATR bank, dominated by staging three rows, is faster with 256 threads)
static unsigned bank_threads(int P) { return 32u * (unsigned)(P < 2 ? 2 : (P > 8 ? 8 : P)); }
static dim3 ind_grid(int64_t N, int S) { return dim3((unsigned)((N + IND_TILE - 1) / IND_TILE), (unsigned)S); }

extern "C" int b200bt_nanfill(float* x, int64_t rows, int64_t N, float* workspace, b200bt_stream_t stream) {
    B200BT_REQUIRE(x && workspace && rows > 0 && N > 0, B200BT_EINVAL, "nanfill: bad argument");
    int rc = check_device();
    if (rc) return rc;
    const int tiles = (int)((N + NF_TILE - 1) / NF_TILE);
    float* t_last = workspace;
    float* t_first = workspace + rows * tiles;
    float* t_nans = t_first + rows * tiles;
    dim3 grid((unsigned)tiles, (unsigned)rows);
    nanfill_scan_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(x, N, tiles, t_last, t_first, t_nans);
    B200BT_LAUNCH_CHECK("nanfill scan");
    nanfill_apply_kernel<<<dim3((unsigned)(tiles < 16 ? tiles : 16), (unsigned)rows), 256, 0, (cudaStream_t)stream>>>(
        x, N, tiles, t_last, t_first, t_nans);
    B200BT_LAUNCH_CHECK("nanfill apply");
    return B200BT_OK;
}

extern "C" int64_t b200bt_nanfill_workspace_floats(int64_t rows, int64_t N) {
    return 3 * rows * ((N + NF_TILE - 1) / NF_TILE);
}

static int fill_bank_params(const int* w_host, int P, bool wilder, BankParams& prm, int& halo_max, const char* name) {
    B200BT_REQUIRE(w_host && P > 0 && P <= IND_MAX_P, B200BT_ELIMIT, "%s: 1..%d windows per call", name, IND_MAX_P);
    halo_max = 0;
    for (int i = 0; i < P; ++i) {
        const int w = w_host[i];
        B200BT_REQUIRE(w >= 1 && w <= IND_MAX_WINDOW, B200BT_ELIMIT, "%s: window %d outside [1,%d]", name, w, IND_MAX_WINDOW);
        prm.window[i] = w;
        const double om = wilder ? ((double)w - 1.0) / (double)w : 1.0 - 2.0 / ((double)w + 1.0);
        prm.halo[i] = halo_for(om);
        if (prm.halo[i] > halo_max) halo_max = prm.halo[i];
    }
    return B200BT_OK;
}

extern "C" int b200bt_ema_bank(const float* x, int S, int64_t N, int64_t ld, const int* spans_host, int P, float* out,
                               b200bt_stream_t stream) {
    B200BT_REQUIRE(x && out, B200BT_EINVAL, "ema_bank: null pointer");
    IND_COMMON_CHECKS("ema_bank");
    BankParams prm;
    int halo_max;
    int rc = fill_bank_params(spans_host, P, false, prm, halo_max, "ema_bank");
    if (rc) return rc;
    const size_t smem = (size_t)(halo_max + IND_TILE + 8) * sizeof(float);
    B200BT_REQUIRE(smem <= 200 * 1024, B200BT_ELIMIT, "ema_bank: span too long for the shared-memory tile");
    cudaError_t e = cudaFuncSetAttribute(ema_bank_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return cuda_status(e, "ema_bank: cudaFuncSetAttribute");
    ema_bank_kernel<<<ind_grid(N, S), bank_threads(P), smem, (cudaStream_t)stream>>>(x, N, ld, prm, P, halo_max, out);
    B200BT_LAUNCH_CHECK("ema_bank launch");
    return B200BT_OK;
}

extern "C" int b200bt_macd(const float* x, int S, int64_t N, int64_t ld, int fast, int slow, int sign, float* line,
                           float* signal, float* diff, b200bt_stream_t stream) {
    B200BT_REQUIRE(x && line && signal && diff, B200BT_EINVAL, "macd: null pointer");
    IND_COMMON_CHECKS("macd");
    B200BT_REQUIRE(fast >= 1 && slow >= 1 && sign >= 1 && fast <= 512 && slow <= 512 && sign <= 512, B200BT_ELIMIT,
                   "macd: spans must be in [1,512]");
    const int halo_ema = halo_for(1.0 - 2.0 / ((double)(fast > slow ? fast : slow) + 1.0));
    const int halo_sig = halo_for(1.0 - 2.0 / ((double)sign + 1.0));
    const size_t smem = (size_t)(halo_sig + IND_TILE + 8) * sizeof(double);
    B200BT_REQUIRE(smem <= 200 * 1024, B200BT_ELIMIT, "macd: signal span too long for the shared-memory tile");
    cudaError_t e = cudaFuncSetAttribute(macd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return cuda_status(e, "macd: cudaFuncSetAttribute");
    macd_kernel<<<ind_grid(N, S), 32, smem, (cudaStream_t)stream>>>(x, N, ld, fast, slow, sign, halo_ema, halo_sig, line,
                                                                     signal, diff);
    B200BT_LAUNCH_CHECK("macd launch");
    return B200BT_OK;
}

extern "C" int b200bt_sma_bank(const float* x, int S, int64_t N, int64_t ld, const int* windows_host, int P, float* out,
                               b200bt_stream_t stream) {
    B200BT_REQUIRE(x && out, B200BT_EINVAL, "sma_bank: null pointer");
    IND_COMMON_CHECKS("sma_bank");
    BankParams prm;
    int halo_max = 0;
    B200BT_REQUIRE(windows_host && P > 0 && P <= IND_MAX_P, B200BT_ELIMIT, "sma_bank: 1..%d windows per call", IND_MAX_P);
    for (int i = 0; i < P; ++i) {
        B200BT_REQUIRE(windows_host[i] >= 1 && windows_host[i] <= IND_MAX_WINDOW, B200BT_ELIMIT, "sma_bank: window %d outside [1,%d]",
                       windows_host[i], IND_MAX_WINDOW);
        prm.window[i] = windows_host[i];
        prm.halo[i] = windows_host[i] - 1;
        if (prm.halo[i] > halo_max) halo_max = prm.halo[i];
    }
    const size_t smem = (size_t)(halo_max + IND_TILE + 2) * sizeof(double);
    cudaError_t e = cudaFuncSetAttribute(sma_bank_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return cuda_status(e, "sma_bank: cudaFuncSetAttribute");
    sma_bank_kernel<<<ind_grid(N, S), IND_THREADS, smem, (cudaStream_t)stream>>>(x, N, ld, prm, P, halo_max, out);
    B200BT_LAUNCH_CHECK("sma_bank launch");
    return B200BT_OK;
}

extern "C" int b200bt_bollinger(const float* x, int S, int64_t N, int64_t ld, int window, double k, float* high,
                                float* mid, float* low, float* width, float* pos, b200bt_stream_t stream) {
    B200BT_REQUIRE(x && high && mid && low && width && pos, B200BT_EINVAL, "bollinger: null pointer");
    IND_COMMON_CHECKS("bollinger");
    B200BT_REQUIRE(window >= 1 && window <= IND_MAX_WINDOW, B200BT_ELIMIT, "bollinger: window outside [1,%d]", IND_MAX_WINDOW);
    const size_t smem = (size_t)2 * (IND_TILE + IND_MAX_WINDOW + 1) * sizeof(double);
    cudaError_t e = cudaFuncSetAttribute(bollinger_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return cuda_status(e, "bollinger: cudaFuncSetAttribute");
    bollinger_kernel<<<ind_grid(N, S), IND_THREADS, smem, (cudaStream_t)stream>>>(x, N, ld, window, k, high, mid, low, width, pos);
    B200BT_LAUNCH_CHECK("bollinger launch");
    return B200BT_OK;
}

static int launch_extrema(const float* high, const float* low, const float* close, int S, int64_t N, int64_t ld, int mode,
                          int w1, int w2, int w3, float* a, float* b, b200bt_stream_t stream, const char* name) {
    B200BT_REQUIRE(high && low && a, B200BT_EINVAL, "%s: null pointer", name);
    B200BT_REQUIRE(S > 0 && N > 0 && ld >= N, B200BT_EINVAL, "%s: bad sizes", name);
    B200BT_REQUIRE(w1 >= 1 && w2 >= 1 && w3 >= 1 && w1 <= IND_MAX_WINDOW && w2 <= IND_MAX_WINDOW && w3 <= IND_MAX_WINDOW,
                   B200BT_ELIMIT, "%s: window outside [1,%d]", name, IND_MAX_WINDOW);
    int rc = check_device();
    if (rc) return rc;
    const size_t smem = (size_t)3 * (IND_TILE + 2 * IND_MAX_WINDOW) * sizeof(float);
    cudaError_t e = cudaFuncSetAttribute(extrema_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return cuda_status(e, "extrema: cudaFuncSetAttribute");
    extrema_kernel<<<ind_grid(N, S), IND_THREADS, smem, (cudaStream_t)stream>>>(high, low, close, N, ld, mode, w1, w2, w3, a, b);
    B200BT_LAUNCH_CHECK("extrema launch");
    return B200BT_OK;
}

extern "C" int b200bt_stochastic(const float* high, const float* low, const float* close, int S, int64_t N, int64_t ld,
                                 int window, int smooth, float* k, float* d, b200bt_stream_t stream) {
    B200BT_REQUIRE(close && d, B200BT_EINVAL, "stochastic: null pointer");
    return launch_extrema(high, low, close, S, N, ld, 0, window, smooth, 1, k, d, stream, "stochastic");
}

extern "C" int b200bt_williams_r(const float* high, const float* low, const float* close, int S, int64_t N, int64_t ld,
                                 int lbp, float* out, b200bt_stream_t stream) {
    B200BT_REQUIRE(close, B200BT_EINVAL, "williams_r: null pointer");
    return launch_extrema(high, low, close, S, N, ld, 1, lbp, 1, 1, out, nullptr, stream, "williams_r");
}

extern "C" int b200bt_ichimoku(const float* high, const float* low, int S, int64_t N, int64_t ld, int w1, int w2, int w3,
                               float* a, float* b, b200bt_stream_t stream) {
    B200BT_REQUIRE(b, B200BT_EINVAL, "ichimoku: null pointer");
    return launch_extrema(high, low, nullptr, S, N, ld, 2, w1, w2, w3, a, b, stream, "ichimoku");
}

extern "C" int b200bt_atr_bank(const float* high, const float* low, const float* close, int S, int64_t N, int64_t ld,
                               const int* windows_host, int P, float* out, b200bt_stream_t stream) {
    B200BT_REQUIRE(high && low && close && out, B200BT_EINVAL, "atr_bank: null pointer");
    IND_COMMON_CHECKS("atr_bank");
    BankParams prm;
    int halo_max;
    int rc = fill_bank_params(windows_host, P, true, prm, halo_max, "atr_bank");
    if (rc) return rc;
    for (int i = 0; i < P; ++i) B200BT_REQUIRE(prm.window[i] <= IND_TILE / 2, B200BT_ELIMIT, "atr_bank: window too long");
    const size_t smem = (size_t)(halo_max + IND_TILE + IND_MAX_WINDOW + 8) * sizeof(double);
    B200BT_REQUIRE(smem <= 200 * 1024, B200BT_ELIMIT, "atr_bank: window too long for the shared-memory tile");
    cudaError_t e = cudaFuncSetAttribute(atr_bank_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return cuda_status(e, "atr_bank: cudaFuncSetAttribute");
    atr_bank_kernel<<<ind_grid(N, S), IND_THREADS, smem, (cudaStream_t)stream>>>(high, low, close, N, ld, prm, P, halo_max, out);
    B200BT_LAUNCH_CHECK("atr_bank launch");
    return B200BT_OK;
}

extern "C" int b200bt_vwap(const float* high, const float* low, const float* close, const float* volume, int S, int64_t N,
                           int64_t ld, int window, float* out, b200bt_stream_t stream) {
    B200BT_REQUIRE(high && low && close && volume && out, B200BT_EINVAL, "vwap: null pointer");
    IND_COMMON_CHECKS("vwap");
    B200BT_REQUIRE(window >= 1 && window <= IND_MAX_WINDOW, B200BT_ELIMIT, "vwap: window outside [1,%d]", IND_MAX_WINDOW);
    const size_t smem = (size_t)2 * (IND_TILE + IND_MAX_WINDOW + 1) * sizeof(double);
    cudaError_t e = cudaFuncSetAttribute(vwap_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return cuda_status(e, "vwap: cudaFuncSetAttribute");
    vwap_kernel<<<ind_grid(N, S), IND_THREADS, smem, (cudaStream_t)stream>>>(high, low, close, volume, N, ld, window, out);
    B200BT_LAUNCH_CHECK("vwap launch");
    return B200BT_OK;
}

// TechnicalAnalyzer._calculate_all_indicators for S symbols: three fused launches + one batched NaN-policy call.
// The workspace holds the RSI column's seam states (S x (tiles - 1) double2) during launch A, then the NaN policy's tile
// summaries.
extern "C" int64_t b200bt_analyzer_workspace_floats(int S, int64_t N) {
    const int64_t seam = (int64_t)4 * S * ((N + IND_TILE - 1) / IND_TILE - 1);
    const int64_t nf = b200bt_nanfill_workspace_floats((int64_t)5 * S, N);
    return seam > nf ? seam : nf;
}

extern "C" int b200bt_analyzer(const float* high, const float* low, const float* close, const float* volume, int S, int64_t N,
                               int64_t ld, float* cols, float* workspace, b200bt_stream_t stream) {
    B200BT_REQUIRE(high && low && close && volume && cols && workspace, B200BT_EINVAL, "analyzer: null pointer");
    IND_COMMON_CHECKS("analyzer");
    B200BT_REQUIRE(((uintptr_t)workspace & 15) == 0, B200BT_EINVAL, "analyzer: workspace must be 16-byte aligned");
    cudaStream_t st = (cudaStream_t)stream;
    const int64_t plane = (int64_t)S * N;
    auto col = [&](int c) { return cols + (int64_t)c * plane; };
    // the reference's windows (binance_ml_strategy.py:67-179)
    const int fast = 12, slow = 26, sign = 9, w_rsi = 14, w_bb = 20, w_st = 14, smooth = 3, w_wr = 14, w_atr = 14, w_vwap = 14;
    const int sma_w[3] = {20, 50, 200}, ich[3] = {9, 26, 52};
    // A: close -> ema_12, ema_26, macd, macd_signal, macd_diff, rsi
    {
        const int halo_ema = halo_for(1.0 - 2.0 / ((double)slow + 1.0)), halo_sig = halo_for(1.0 - 2.0 / ((double)sign + 1.0));
        double2* rsi_seam = reinterpret_cast<double2*>(workspace);
        int rc = rsi_seam_states(close, S, N, ld, &w_rsi, 1, IND_TILE, rsi_seam, st);
        if (rc) return rc;
        const size_t smem = (size_t)(halo_sig + IND_TILE + 8) * sizeof(double);
        cudaError_t e = cudaFuncSetAttribute(analyzer_a_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return cuda_status(e, "analyzer: cudaFuncSetAttribute");
        LeadFill lf{};
        const int cs[6] = {B200BT_COL_EMA_12, B200BT_COL_EMA_26, B200BT_COL_MACD, B200BT_COL_MACD_SIGNAL, B200BT_COL_MACD_DIFF, B200BT_COL_RSI};
        const int fs[6] = {fast - 1, slow - 1, slow - 1, slow - 1 + sign - 1, slow - 1 + sign - 1, w_rsi - 1};
        lf.n = 6;
        for (int i = 0; i < 6; ++i) { lf.col[i] = col(cs[i]); lf.first[i] = fs[i]; }
        analyzer_a_kernel<<<ind_grid(N, S), 64, smem, st>>>(close, N, ld, fast, slow, sign, halo_ema, halo_sig, w_rsi, rsi_seam,
                                                           col(B200BT_COL_EMA_12), col(B200BT_COL_EMA_26), col(B200BT_COL_MACD),
                                                           col(B200BT_COL_MACD_SIGNAL), col(B200BT_COL_MACD_DIFF), col(B200BT_COL_RSI), lf);
        B200BT_LAUNCH_CHECK("analyzer A launch");
    }
    // B: close -> sma_20, sma_50, sma_200, Bollinger
    {
        const int halo = sma_w[2] - 1;
        const size_t smem = (size_t)2 * (IND_TILE + IND_MAX_WINDOW + 1) * sizeof(double);
        cudaError_t e = cudaFuncSetAttribute(analyzer_b_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return cuda_status(e, "analyzer: cudaFuncSetAttribute");
        LeadFill lf{};
        const int cs[7] = {B200BT_COL_SMA_20, B200BT_COL_SMA_50, B200BT_COL_SMA_200, B200BT_COL_BB_HIGH, B200BT_COL_BB_MID, B200BT_COL_BB_LOW,
                           B200BT_COL_BB_WIDTH};
        const int fs[7] = {sma_w[0] - 1, sma_w[1] - 1, sma_w[2] - 1, w_bb - 1, w_bb - 1, w_bb - 1, w_bb - 1};
        lf.n = 7;
        for (int i = 0; i < 7; ++i) { lf.col[i] = col(cs[i]); lf.first[i] = fs[i]; }
        analyzer_b_kernel<<<ind_grid(N, S), IND_THREADS, smem, st>>>(close, N, ld, sma_w[0], sma_w[1], sma_w[2], w_bb, 2.0,
                                                                    col(B200BT_COL_SMA_20), col(B200BT_COL_SMA_50), col(B200BT_COL_SMA_200),
                                                                    col(B200BT_COL_BB_HIGH), col(B200BT_COL_BB_MID), col(B200BT_COL_BB_LOW),
                                                                    col(B200BT_COL_BB_WIDTH), col(B200BT_COL_BB_POSITION), halo, lf);
        B200BT_LAUNCH_CHECK("analyzer B launch");
    }
    // C: high, low, close, volume -> stochastic, Williams %R, Ichimoku, ATR, VWAP
    {
        B200BT_REQUIRE(w_wr == w_st && ich[0] <= w_st && w_st <= ich[1] && ich[1] <= ich[2], B200BT_EINVAL, "analyzer: windows must nest");
        BankParams prm;
        int atr_halo;
        int rc = fill_bank_params(&w_atr, 1, true, prm, atr_halo, "analyzer");
        if (rc) return rc;
        B200BT_REQUIRE(ich[2] - 1 <= 256 && w_st + smooth - 2 <= 256, B200BT_ELIMIT, "analyzer: window too long");
        size_t smem = (size_t)3 * (IND_TILE + 256) * sizeof(float) + (size_t)(IND_TILE + 256) * sizeof(double);
        const size_t smem_atr = (size_t)(atr_halo + IND_TILE + IND_MAX_WINDOW + 8) * sizeof(double);
        const size_t smem_vwap = (size_t)2 * (IND_TILE + IND_MAX_WINDOW + 1) * sizeof(double);
        if (smem_atr > smem) smem = smem_atr;
        if (smem_vwap > smem) smem = smem_vwap;
        cudaError_t e = cudaFuncSetAttribute(analyzer_c_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return cuda_status(e, "analyzer: cudaFuncSetAttribute");
        LeadFill lf{};
        lf.n = 2;
        lf.col[0] = col(B200BT_COL_ICHIMOKU_A); lf.first[0] = ich[1] - 1;
        lf.col[1] = col(B200BT_COL_ICHIMOKU_B); lf.first[1] = ich[2] - 1;
        analyzer_c_kernel<<<ind_grid(N, S), IND_THREADS, smem, st>>>(high, low, close, volume, N, ld, w_st, smooth, ich[0], ich[1], ich[2],
                                                                    w_atr, atr_halo, w_vwap, col(B200BT_COL_STOCH_K), col(B200BT_COL_STOCH_D),
                                                                    col(B200BT_COL_WILLIAMS_R), col(B200BT_COL_ICHIMOKU_A),
                                                                    col(B200BT_COL_ICHIMOKU_B), col(B200BT_COL_ATR), col(B200BT_COL_VWAP), lf);
        B200BT_LAUNCH_CHECK("analyzer C launch");
    }
    // NaN policy of the five columns that can be undefined in mid-series (they are the last five of the allocation)
    return b200bt_nanfill(col(B200BT_COL_VWAP), (int64_t)5 * S, N, workspace, stream);
}
