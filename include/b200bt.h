/*
 * b200bt.h -- C-ABI of the B200-native backtest / evolution / Monte-Carlo engine.
 *
 * This is the drop-in boundary below the reference's Python call surface
 * (zd87pl/ai-crypto-trader; SURVEY.md section 8b).  The reference has no FFI
 * of its own -- every function on the path is plain Python -- so each entry
 * point below cites the reference function (file:line, relative to the
 * reference tree) whose arithmetic it replaces.  All pointers are DEVICE
 * pointers unless a name ends in `_host`.  No torch types cross this
 * boundary: sizes are plain integers, `stream` is a `cudaStream_t` passed as
 * `void*`.  Every function returns 0 on success and a non-zero status on
 * failure (a `cudaError_t` value, or one of the B200BT_E* codes); nothing
 * throws across the boundary.  `b200bt_last_error()` returns a thread-local,
 * human-readable description of the last failure.
 *
 * There is NO CPU fallback behind this ABI.  If no sm_100 device is present
 * the compute entry points return B200BT_ENODEVICE.
 */
#ifndef B200BT_H_
#define B200BT_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B200BT_ABI_VERSION 1

#define B200BT_OK 0
#define B200BT_EINVAL 10001   /* bad argument (null pointer, size <= 0, ...)   */
#define B200BT_ENODEVICE 10002 /* no CUDA device / wrong architecture          */
#define B200BT_ELIMIT 10003   /* argument exceeds a documented limit           */

typedef void* b200bt_stream_t; /* cudaStream_t */

int b200bt_abi_version(void);
const char* b200bt_last_error(void);
/* Number of kernels launched by this library in this process (all threads);
 * bench.py reports the delta over the timed region as `gpu_launches`. */
int64_t b200bt_launch_count(void);

/* ------------------------------------------------------------------------
 * Family 1: rolling indicators over fp32 OHLCV.
 * Series layout: row-major [S][N] fp32, one row per symbol ("SoA per field").
 * Bank layout:   row-major [S][P][N] fp32, one row per (symbol, period).
 * Arithmetic is fp64 internally (so that a float64 CPU evaluation of the same
 * recurrence rounds to the same fp32 value), outputs are fp32.
 * NaN policy follows TechnicalAnalyzer._handle_nan_values
 * (binance_ml_strategy.py:28-38): leading undefined values are back-filled
 * with the first defined value (`fill=1`) or written as NaN (`fill=0`).
 * ------------------------------------------------------------------------ */

/* RSI bank.  Replaces ta.momentum.RSIIndicator(close, window=w).rsi() as called
 * at binance_ml_strategy.py:112 (and services/market_monitor_service.py:228),
 * for every window in periods_host[0..P).  Wilder smoothing
 * ewm(alpha=1/w, adjust=False) of up/down moves; rsi = 100 where the smoothed
 * down move is 0. */
int b200bt_rsi_bank(const float* close, int S, int64_t N, int64_t ld,
                    const int* periods_host, int P, int fill,
                    float* out, b200bt_stream_t stream);

/* TechnicalAnalyzer._calculate_all_indicators + _handle_nan_values (binance_ml_strategy.py:28-182) for S symbols in three
 * fused launches (close -> EMA / MACD / RSI; close -> SMA / Bollinger; high, low, close, volume -> stochastic / Williams %R /
 * Ichimoku / ATR / VWAP) plus one batched NaN-policy call, with the reference's windows (20/50/200, 12/26/9, 9/26/52, 14, 14/3,
 * 14, 20 x 2.0, 14, 14).  cols: [B200BT_ANALYZER_COLUMNS][S][N] fp32 (device, out), column c at cols + c * S * N in the order
 * below; workspace: b200bt_analyzer_workspace_floats(S, N) floats (device, 16-byte aligned). */
enum b200bt_analyzer_column {
    B200BT_COL_SMA_20 = 0, B200BT_COL_SMA_50, B200BT_COL_SMA_200, B200BT_COL_EMA_12, B200BT_COL_EMA_26, B200BT_COL_MACD,
    B200BT_COL_MACD_SIGNAL, B200BT_COL_MACD_DIFF, B200BT_COL_ICHIMOKU_A, B200BT_COL_ICHIMOKU_B, B200BT_COL_RSI, B200BT_COL_BB_HIGH,
    B200BT_COL_BB_MID, B200BT_COL_BB_LOW, B200BT_COL_BB_WIDTH, B200BT_COL_ATR,
    /* columns that can be undefined in mid-series (zero volume / zero range): general ffill-bfill pass */
    B200BT_COL_VWAP, B200BT_COL_STOCH_K, B200BT_COL_STOCH_D, B200BT_COL_WILLIAMS_R, B200BT_COL_BB_POSITION,
    B200BT_ANALYZER_COLUMNS
};
int64_t b200bt_analyzer_workspace_floats(int S, int64_t N);
int b200bt_analyzer(const float* high, const float* low, const float* close, const float* volume, int S, int64_t N, int64_t ld,
                    float* cols, float* workspace, b200bt_stream_t stream);

/* b200bt_rsi_bank (NaN policy applied) that also writes the bank's rows of a sweep zone map (see b200bt_zone_map: row 0 =
 * the close prices, rows 1..P = the RSI rows) while the values are in registers, so that the first sweep of a fresh bank can
 * already skip quiet blocks.  `zones` is the WHOLE zone map of S_total symbols (b200bt_zone_map_floats(P, S_total, N) floats);
 * this call fills the rows of symbols [sym0, sym0 + S), whose closes / bank rows `close` / `out` point at. */
int b200bt_rsi_bank_zones(const float* close, int S, int64_t N, int64_t ld, const int* periods_host, int P,
                          float* out, float* zones, int S_total, int sym0, b200bt_stream_t stream);

/* EMA bank: ta.trend.EMAIndicator(close, window=w) = ewm(span=w, min_periods=w, adjust=False)
 * (binance_ml_strategy.py:79-83).  out [S][P][N]; undefined leading values are NaN. */
int b200bt_ema_bank(const float* x, int S, int64_t N, int64_t ld, const int* spans_host, int P,
                    float* out, b200bt_stream_t stream);

/* SMA bank: ta.trend.SMAIndicator = rolling(w, min_periods=w).mean() (:67-76). out [S][P][N]. */
int b200bt_sma_bank(const float* x, int S, int64_t N, int64_t ld, const int* windows_host, int P,
                    float* out, b200bt_stream_t stream);

/* MACD: ta.trend.MACD(close, slow, fast, sign) (:91-94).  line/signal/diff each [S][N]. */
int b200bt_macd(const float* x, int S, int64_t N, int64_t ld, int fast, int slow, int sign,
                float* line, float* signal, float* diff, b200bt_stream_t stream);

/* Bollinger bands: ta.volatility.BollingerBands(close, window, k) plus the analyzer's
 * bb_width and bb_position (zero range -> NaN) (:148-156).  Five outputs, each [S][N]. */
int b200bt_bollinger(const float* x, int S, int64_t N, int64_t ld, int window, double k,
                     float* high, float* mid, float* low, float* width, float* position,
                     b200bt_stream_t stream);

/* Stochastic oscillator %K / %D: ta.momentum.StochasticOscillator(high, low, close, window,
 * smooth_window) (:121-127). */
int b200bt_stochastic(const float* high, const float* low, const float* close, int S, int64_t N,
                      int64_t ld, int window, int smooth, float* k, float* d, b200bt_stream_t stream);

/* Williams %R: ta.momentum.WilliamsRIndicator(high, low, close, lbp) (:135-140). */
int b200bt_williams_r(const float* high, const float* low, const float* close, int S, int64_t N,
                      int64_t ld, int lbp, float* out, b200bt_stream_t stream);

/* Ichimoku a / b: ta.trend.IchimokuIndicator(high, low, w1, w2, w3, visual=False) (:102-104). */
int b200bt_ichimoku(const float* high, const float* low, int S, int64_t N, int64_t ld, int w1, int w2,
                    int w3, float* a, float* b, b200bt_stream_t stream);

/* ATR bank: ta.volatility.AverageTrueRange(high, low, close, window=w) (:164); zeros before
 * bar w-1 (ta writes 0, not NaN).  out [S][P][N]. */
int b200bt_atr_bank(const float* high, const float* low, const float* close, int S, int64_t N,
                    int64_t ld, const int* windows_host, int P, float* out, b200bt_stream_t stream);

/* VWAP: ta.volume.VolumeWeightedAveragePrice(high, low, close, volume, window) (:173-179). */
int b200bt_vwap(const float* high, const float* low, const float* close, const float* volume, int S,
                int64_t N, int64_t ld, int window, float* out, b200bt_stream_t stream);

/* Multi-timeframe (BASELINE configs[3]; recipe: services/market_monitor_service.py:219-301, where
 * each timeframe is its own kline series, :168-171).  b200bt_resample derives clock-aligned k-minute
 * OHLCV [5][S][M] from 1-minute (or bar_minutes) OHLCV [5][S][N]; M = b200bt_resample_bars(...).
 * b200bt_align maps a higher-timeframe series [S][M] back onto the base clock [S][N] using the last
 * COMPLETED higher-timeframe bar (NaN before the first one). */
int64_t b200bt_resample_bars(int64_t N, int64_t minute0, int bar_minutes, int k);
int b200bt_resample(const float* ohlcv, int S, int64_t N, int64_t minute0, int bar_minutes, int k,
                    float* out, int64_t M, b200bt_stream_t stream);
int b200bt_align(const float* src, int S, int64_t M, int64_t N, int64_t minute0, int bar_minutes, int k,
                 float* out, b200bt_stream_t stream);

/* TechnicalAnalyzer._handle_nan_values (:28-38) on `rows` contiguous rows of length N, in place:
 * forward-fill, then back-fill, then 0.  workspace: b200bt_nanfill_workspace_floats(rows, N) floats. */
int64_t b200bt_nanfill_workspace_floats(int64_t rows, int64_t N);
int b200bt_nanfill(float* x, int64_t rows, int64_t N, float* workspace, b200bt_stream_t stream);

/* ------------------------------------------------------------------------
 * Family 2: the per-bar entry/exit/stop/PnL state machine over
 * (GA-individual x symbol) lanes.
 * Replaces, for a whole population at once:
 *   StrategyEvaluationSystem._simulate_trades   services/strategy_evaluation.py:746-878
 *   StrategyPerformanceMetrics.calculate_metrics services/strategy_evaluation.py:32-228
 *   StrategyEvaluationSystem._calculate_strategy_score              :579-633
 * which GeneticAlgorithm.evaluate_population (services/genetic_algorithm.py:119-133)
 * calls once per individual.
 * ------------------------------------------------------------------------ */

/* One GA individual, already decoded by the host:
 *  rsi_row       row of the RSI bank holding this individual's rsi_period
 *  rsi_lo        `rsi < rsi_oversold`  is evaluated as  r < rsi_lo  (fp32)
 *  rsi_hi        `rsi > rsi_overbought` is evaluated as r > rsi_hi  (fp32)
 *                (host rounds the float64 thresholds up/down to fp32 so the
 *                 fp32 compare decides exactly like the float64 one)
 *  take_profit   take_profit/100  (float64, strategy_evaluation.py:773)
 *  stop_loss     stop_loss/100    (float64, :774)
 *  position_size dollars, 10000*min(max_position_size,20)/100 (:762-764)
 */
typedef struct b200bt_individual {
    int32_t rsi_row;
    float rsi_lo;
    float rsi_hi;
    int32_t reserved;
    double take_profit;
    double stop_loss;
    double position_size;
} b200bt_individual; /* 40 bytes */

/* Per-lane result, 20 x 8 bytes.  Field meaning follows calculate_metrics
 * (strategy_evaluation.py:187-225) on the lane's trade RECORDS (an entry and
 * an exit record per round trip, as the reference emits them). */
typedef struct b200bt_lane_stats {
    double n_records;      /* total_trades                                   */
    double n_wins;         /* #records with pnl > 0                          */
    double n_losses;       /* #records with pnl < 0                          */
    double total_profit;   /* sum of positive pnl                            */
    double total_loss;     /* sum of negative pnl (<= 0)                     */
    double net_profit;     /* total_profit + total_loss                      */
    double max_drawdown;   /* fraction of peak equity                        */
    double sharpe_ratio;   /* daily-bucket Sharpe, sqrt(252) annualised      */
    double n_days;         /* distinct calendar days holding a record        */
    double largest_profit;
    double largest_loss;
    double sum_duration_bars; /* sum over round trips of exit_bar-entry_bar  */
    double score;          /* _calculate_strategy_score                      */
    double win_rate;
    double profit_factor;  /* +inf when total_loss == 0 (reference :113)     */
    /* ingredients of calculate_advanced_metrics (strategy_evaluation.py:231-319) that need the daily buckets */
    double sortino_ratio;  /* mean(daily) / std(negative dailies, ddof 0) * sqrt(252); +inf without a negative
                              spread, 0 without daily buckets (:250-263)      */
    double n_negative_days;
    double downside_deviation; /* np.std of the negative daily sums           */
    double mean_daily_pnl; /* profit_per_day (:307-312)                       */
    uint64_t trade_hash;   /* xor of event_hash(event_index, event word) over all events */
} b200bt_lane_stats; /* 160 bytes */

/* Scoring rule (config.json evolution.optimization_goals; SURVEY 8-a15). */
#define B200BT_PRIMARY_SHARPE 0
#define B200BT_PRIMARY_RETURN_PCT 1
#define B200BT_PRIMARY_PROFIT_FACTOR 2
#define B200BT_PRIMARY_WIN_RATE 3
#define B200BT_PRIMARY_NET_PROFIT 4
/* any other scalar key of the metrics dict may be the primary metric (`metrics.get(primary, 0)`, :589-590) */
#define B200BT_PRIMARY_TOTAL_TRADES 5
#define B200BT_PRIMARY_MAX_DRAWDOWN 6
#define B200BT_PRIMARY_TOTAL_PROFIT 7
#define B200BT_PRIMARY_TOTAL_LOSS 8
#define B200BT_PRIMARY_LARGEST_PROFIT 9
#define B200BT_PRIMARY_LARGEST_LOSS 10
#define B200BT_PRIMARY_AVERAGE_PROFIT 11
#define B200BT_PRIMARY_AVERAGE_LOSS 12
/* keys only calculate_advanced_metrics adds (:231-319): present when the score is taken on the advanced dict
 * (evaluate_strategy :545-557); on the plain dict (cross_validate_strategy :683-691) the host passes ZERO for them */
#define B200BT_PRIMARY_SORTINO 13
#define B200BT_PRIMARY_EXPECTANCY 14
#define B200BT_PRIMARY_CALMAR 15
#define B200BT_PRIMARY_PROFIT_PER_DAY 16
#define B200BT_PRIMARY_RECOVERY_FACTOR 17
#define B200BT_PRIMARY_ZERO 99           /* a key the metrics dict does not hold: metrics.get(key, 0) */
#define B200BT_SEC_MAX_DRAWDOWN 1
#define B200BT_SEC_WIN_RATE 2
#define B200BT_SEC_PROFIT_FACTOR 4
#define B200BT_SEC_EXPECTANCY 8          /* score *= 1 + min(expectancy / 100, 1) (:615-620); set by the host only when
                                            the score is taken on the advanced dict (else the key is absent: factor 1) */

typedef struct b200bt_sweep_config {
    double initial_capital;  /* 10000.0 (strategy_evaluation.py:33,761)       */
    int64_t minute0;         /* minutes since 1970-01-01T00:00Z of bar 0      */
    int32_t bar_minutes;     /* bar spacing; day = (minute0+t*bar_minutes)/1440 */
    int32_t primary;         /* B200BT_PRIMARY_*                              */
    int32_t secondary_mask;  /* B200BT_SEC_* bits                             */
    int32_t variant;         /* kernel variant selector, 0 = default          */
    int32_t gap_bar;         /* > 0: the series is two pieces glued at this bar (training folds of            */
    int32_t gap_minutes;     /*      cross_validate_strategy :674-682): bars >= gap_bar lie gap_minutes later  */
} b200bt_sweep_config;   /* 40 bytes */

/* Event word written to the optional trade buffer: bits 0..29 bar index,
 * bit 30 = 1 for an exit record, bit 31 = 1 for side "sell"
 * (short entry / long exit).  */
#define B200BT_EVENT_EXIT 0x40000000u
#define B200BT_EVENT_SELL 0x80000000u

/* Run the population sweep.
 *  price   [S][N] fp32 (row stride ld_price)       close prices
 *  rsi     [S][P][N] fp32 (row stride ld_rsi)      RSI bank
 *  indiv   [pop] individuals (device)
 *  order   [pop] int32 (device) evaluation order of individuals (a permutation;
 *          the host sorts by rsi_row so neighbouring warps share a stream);
 *          may be NULL for identity
 *  stats   [pop][S] lane stats (device, out)
 *  events  optional [pop][S][event_cap] uint32 (device, out), first event_cap
 *          event words per lane; NULL to skip
 * Limits: N < 2^30.
 */
int b200bt_sweep(const float* price, int64_t ld_price,
                 const float* rsi, int64_t ld_rsi, int P,
                 int S, int64_t N,
                 const b200bt_individual* indiv, const int32_t* order, int pop,
                 const b200bt_sweep_config* cfg_host,
                 b200bt_lane_stats* stats,
                 uint32_t* events, int64_t event_cap,
                 b200bt_stream_t stream);

/* Time-chunked form of b200bt_sweep (same results; csrc/sweep_chunked.cu).  Expensive lanes are split
 * into n_chunks time chunks scanned concurrently, each started `warm` bars early from the flat state;
 * the chunk-boundary states are verified lane by lane and a chunk whose assumed state was wrong is re-scanned from the
 * true state until its trajectory meets the recorded one again (the rest of the recorded events is then kept).
 * max_repair_rounds: 0 = no repair, 1 = one chunk-parallel pass (every wrong chunk re-scanned once, trusting its
 * predecessor's recorded end state), >= 2 = that pass plus a lane-sequential one beside the metrics kernels that finishes
 * the lanes whose re-scans run through chunk after chunk; nothing is read back.
 * A lane that still has a mismatch (or lost events to a full pool) is flagged in lane_invalid[pop][S]
 * (stats of flagged lanes are NOT written: re-evaluate those individuals with b200bt_sweep, passing them
 * as `order`).  One work item per (individual, chunk); `segment` = seg_base[individual] + chunk.
 *  items      [n_items] device      seg_base, n_chunks  [pop] device int32      n_seg = sum of n_chunks
 *  pool_blocks  event pool size in blocks of 256 events; a chunk that cannot get a block flags its lane
 *  workspace  b200bt_sweep_chunked_workspace_bytes(pool_blocks, S, n_seg) device bytes
 *  overflow_host_or_null  optional PINNED host int[4], written asynchronously on `stream` (read after synchronising it):
 *                         [0] = 1 if the event pool ran out (grow it next time), [1] = number of (individual, symbol)
 *                         lanes that were flagged and re-evaluated by the exact fallback, [2] = pool blocks handed out
 *                         (what the next sweep of a similar population needs), [3] = tiles of the thread-per-lane scan
 *                         whose bulk copy did not complete in time (b200bt_sweep_tiled; their work was redone, see there).
 * Flagged lanes are re-evaluated by the fused kernel (b200bt_sweep's) inside this call, from a device-side list: the call
 * reads nothing back and never synchronises; lane_invalid reports which lanes took that path. */
typedef struct b200bt_chunk_item {
    int32_t individual;
    int32_t chunk;
    int32_t n_chunks;
    int32_t segment;
} b200bt_chunk_item;

int64_t b200bt_sweep_chunked_workspace_bytes(int pool_blocks, int S, int n_seg);
int b200bt_sweep_chunked(const float* price, int64_t ld_price, const float* rsi, int64_t ld_rsi, int P,
                         int S, int64_t N, const b200bt_individual* indiv, const int32_t* order, int pop,
                         const b200bt_chunk_item* items, int n_items, const int32_t* seg_base,
                         const int32_t* n_chunks, int n_seg, int warm, int max_repair_rounds, int pool_blocks,
                         void* workspace, int64_t workspace_bytes, const b200bt_sweep_config* cfg_host,
                         b200bt_lane_stats* stats, uint32_t* events, int64_t event_cap,
                         unsigned char* lane_invalid, int* overflow_host_or_null, b200bt_stream_t stream);

/* Same contract as b200bt_sweep_chunked, thread-per-lane form: EVERY individual is cut into the same K time
 * chunks (chunk c of K covers [floor(N c / K) & ~511, ...)) and each THREAD steps the state machine of one (individual,
 * symbol, chunk) through shared-memory tiles.  Every warp stages its own tiles -- the price row and the RSI rows its 32
 * machines read -- through a private ring of bulk async copies (cp.async.bulk + mbarrier), so warps never wait for each other.
 * Verification, in-place repair, metrics and the lane_invalid / overflow outputs are those of b200bt_sweep_chunked.
 * slots: device int32[n_slots] (n_slots a multiple of 32): individual run by each thread slot, -1 = empty; 32 consecutive
 *        slots form a warp, which may read at most TWO distinct RSI rows (rsi_row) -- the host packs individuals by row and
 *        similar cost; a warp that breaks the rule is not scanned: its lanes are flagged in lane_invalid and the caller
 *        re-evaluates them with b200bt_sweep (exact).  NULL = identity (thread k runs individual k).
 * order: device int32[pop], the individuals in dispatch order (by predicted cost), NULL = identity: the order in which the
 *        per-chunk metrics kernels list their work (one thread per chunk: neighbours should hold similar record counts).
 * zones: optional zone map of the same price / RSI arrays (b200bt_zone_map), NULL = none: (min, max) per 32-bar
 *        block of every row, which lets a warp skip blocks in which none of its machines' thresholds can be crossed.
 * Shared memory does not depend on P (any number of RSI rows). */
int64_t b200bt_zone_map_floats(int P, int S, int64_t N);     /* floats in the zone map: coarse (32-bar) ranges [S][P+1][ceil(N/32) rounded up to even][2], then fine (4-bar) ranges [S][P+1][ceil(N/128)*32][2]; 16-byte aligned */
int b200bt_zone_map(const float* price, int64_t ld_price, const float* rsi, int64_t ld_rsi, int P, int S, int64_t N,
                    float* zones, b200bt_stream_t stream);
int64_t b200bt_sweep_tiled_workspace_bytes(int pool_blocks, int S, int pop, int K);
int b200bt_sweep_tiled(const float* price, int64_t ld_price, const float* rsi, int64_t ld_rsi, int P, int S,
                       int64_t N, const float* zones, const b200bt_individual* indiv, const int32_t* slots, int n_slots,
                       const int32_t* order, int pop, int K, int warm, int max_repair_rounds, int pool_blocks, void* workspace, int64_t workspace_bytes,
                       const b200bt_sweep_config* cfg, b200bt_lane_stats* stats, uint32_t* events,
                       int64_t event_cap, unsigned char* lane_invalid, int* overflow_host_or_null,
                       b200bt_stream_t stream);

/* Measurement hook (bench.py's roofline): a pair of caller-owned cudaEvent_t that the following b200bt_sweep_tiled calls of
 * this process record on their stream immediately before and after the scan kernel (lane_scan_kernel); NULL, NULL switches
 * it off.  The caller reads cudaEventElapsedTime after synchronising.  Not thread-safe (one measuring thread). */
int b200bt_sweep_scan_timing(void* start_event, void* stop_event);
/* Bound of one tile wait of the scan kernel in SM clocks (0 = the default, ~20 ms).  A tile whose bulk copy does not complete
 * within the bound is not waited for any longer: the work item is marked as lost (its chunks are re-scanned by the repair pass
 * or its lanes re-run by the exact fallback), the warp stops using its tile ring, and overflow_host[3] counts the event.  Results
 * do not depend on it.  A negative value -k is the test hook: every warp gives up at the k-th tile of an item as if it had
 * not arrived. */
int b200bt_sweep_scan_wait_cycles(int64_t cycles);

/* fitness[i] = mean over symbols of stats[i][s].score  (float64, device). */
int b200bt_fitness_reduce(const b200bt_lane_stats* stats, int pop, int S,
                          double* fitness, b200bt_stream_t stream);

/* ------------------------------------------------------------------------
 * The reference's own single-symbol bar loop (BASELINE configs[0]):
 *   StrategyTester.backtest_strategy   backtesting/strategy_tester.py:156-312
 *   open_position / close_position     :314-369
 *   PositionSizer.calculate_position_size  binance_ml_strategy.py:251-291
 * One warp per symbol; the entry gate (technical signal x AI decision, constant per
 * symbol in the reference, SURVEY 8-a6) is decided on the host and passed as can_enter.
 * ------------------------------------------------------------------------ */
typedef struct b200bt_bt_params {
    double initial_balance;
    double position_pct;       /* 0.25 / 0.20 / 0.15 by volatility class (:256-264)      */
    double stop_loss_pct;      /* 0.02 / 0.015 / 0.01 -- a FRACTION compared with a PERCENT
                                  pnl (strategy_tester.py:206-215), quirk kept            */
    double take_profit_pct;    /* 2 x stop_loss_pct (:287)                                */
    double volume_factor;      /* min(avg_volume/50000, 1) (:267)                         */
    double max_risk_per_trade; /* 0.15                                                    */
    int32_t can_enter;         /* technical BUY x strength>=70 x AI gate (:371-401)       */
    int32_t skip;              /* 10 (:192)                                               */
} b200bt_bt_params; /* 56 bytes */

/* stats  [S][16] float64: final_balance, total_trades, winning, losing, total_profit,
 *                         total_loss(positive), max_drawdown, max_drawdown_pct, n_equity_points, open_at_end
 * trades [S][trade_cap][8] float64: entry_bar, exit_bar, reason(1 SL,2 TP,3 end), entry_price,
 *                         quantity, position_size, pnl, pnl_pct
 * equity [S][equity_cap][2] float64: bar, cash balance at that (flat or entry) bar */
int b200bt_backtest_ref(const float* price, int64_t ld, int S, int64_t N,
                        const b200bt_bt_params* params, double* stats, double* trades,
                        int64_t trade_cap, double* equity, int64_t equity_cap,
                        b200bt_stream_t stream);

/* ------------------------------------------------------------------------
 * Family 3: Monte-Carlo risk projection.
 * Replaces the path generation and per-path loops of
 *   MonteCarloService.run_monte_carlo_simulation  services/monte_carlo_service.py:197-394
 * Randomness: Philox4x32-10, counter = (path index lo, hi, step/4, mode),
 * key = seed; normals by Box-Muller on 24-bit uniforms.  A path's values depend
 * only on (seed, path_offset + local index, step), never on sharding.
 * Outputs: finals[n] = S_T, maxdd[n] = max_t (runmax_t - S_t)/runmax_t (:327-336),
 * optional paths[(steps+1)][n] fp32 (the reference's `paths` array, shape (days, n)).
 * ------------------------------------------------------------------------ */

/* Geometric Brownian motion (:266-273): `steps` = days-1 multiplicative steps of
 * exp((mu - sigma^2/2) dt + sigma sqrt(dt) Z). */
int b200bt_mc_gbm(double s0, double mu, double sigma, double dt, int64_t n_paths, int steps,
                  uint64_t seed, uint64_t path_offset, float* finals, float* maxdd,
                  float* paths_or_null, b200bt_stream_t stream);

/* 'historical' simulation (:277-298): bootstrap of the return sample with
 * replacement.  block_len = 1 reproduces the reference (iid); block_len > 1 is a
 * circular block bootstrap.  log_returns != 0: P_t = P_{t-1} exp(r); else
 * P_t = P_{t-1} (1 + r).  `returns` is a device array of R <= 12288 fp32 values. */
int b200bt_mc_bootstrap(const float* returns, int R, int block_len, int log_returns, double s0,
                        int64_t n_paths, int steps, uint64_t seed, uint64_t path_offset,
                        float* finals, float* maxdd, float* paths_or_null, b200bt_stream_t stream);

/* Exact order statistics: out[r] = ranks[r]-th smallest (0-based) of x[0..n).
 * ranks_dev: device int64[n_ranks], ASCENDING, n_ranks <= 64.  Two-level radix
 * select; workspace of b200bt_select_workspace_bytes(n_ranks) device bytes.
 * Feeds np.percentile's linear interpolation (:308-317) on the host side. */
int64_t b200bt_select_workspace_bytes(int n_ranks);
int b200bt_select(const float* x, int64_t n, const int64_t* ranks_dev, int n_ranks, float* out,
                  void* workspace, int64_t workspace_bytes, b200bt_stream_t stream);

/* Moments of the final prices (:305-336).  out7 (device, float64):
 *  [0] sum S_T  [1] sum pct  [2] #(S_T > s0)  [3] sum maxdd  [4] max maxdd
 *  [5] sum pct[pct <= var_threshold]  [6] #(pct <= var_threshold)
 * with pct = (S_T/s0 - 1)*100 in float64; maxdd may be NULL. */
int b200bt_mc_moments(const float* finals, const float* maxdd, int64_t n, double s0,
                      double var_threshold, double* out7, b200bt_stream_t stream);

/* ---- portfolio risk (SURVEY 8-f4) -------------------------------------------------------------------
 * Replaces the numeric core of services/portfolio_risk_service.py. */

/* Simple returns, df['close'].pct_change() (portfolio_risk_service.py:208): out[s][0] = NaN,
 * out[s][t] = close[s][t]/close[s][t-1] - 1 in float64, stored fp32.  close, out: device [S][ld]. */
int b200bt_pct_change(const float* close, int64_t ld, int S, int64_t N, float* out, int64_t ld_out,
                      b200bt_stream_t stream);

/* Tail sums for historical CVaR (calculate_conditional_var :248-284), NaN entries skipped (dropna):
 * out4 (device, float64) = [ sum x[x <= threshold], #(x <= threshold), #(non-NaN), sum non-NaN ].
 * Deterministic (fixed-order fold of per-CTA partials). */
int64_t b200bt_tail_stats_workspace_bytes(int64_t n);
int b200bt_tail_stats(const float* x, int64_t n, double threshold, double* out4, void* workspace,
                      int64_t workspace_bytes, b200bt_stream_t stream);

/* Pearson correlation matrix of S return rows (calculate_asset_correlation :286-326, pandas
 * DataFrame.corr(): pairwise-complete observations, NaN = missing; NaN out for <1 joint observation or zero
 * variance).  x: device [S][ld] fp32, out: device float64 [S][S], S <= 512. */
int64_t b200bt_correlation_workspace_bytes(int S, int64_t N);
int b200bt_correlation(const float* x, int64_t ld, int S, int64_t N, double* out, void* workspace,
                       int64_t workspace_bytes, b200bt_stream_t stream);

/* ---- GA operators on the device (SURVEY 8-f2) -------------------------------------------------------
 * The operators of services/genetic_algorithm.py:83-252 over a device matrix params [pop][genes] float64 (integer
 * genes hold integral values).  Ranges: host arrays lo / hi / is_int of length genes (<= 64).  Randomness is
 * Philox4x32-10 keyed by (seed; generation, slot): parity with the reference's Mersenne-twister stream is
 * DISTRIBUTIONAL (same operators and probabilities), results are a pure function of (seed, generation, inputs). */

/* initialize_population (:83-117): rows >= n_seeded are drawn uniformly from the ranges (randint / uniform),
 * rows < n_seeded (already written by the caller) are clamped to the ranges. */
int b200bt_ga_init(double* params, int pop, int genes, int n_seeded, const double* lo, const double* hi,
                   const int* is_int, uint64_t seed, b200bt_stream_t stream);

/* selection + crossover + mutation (:135-252) -> params_out (must not alias params).
 * ranked: device int32[pop], indices by descending fitness (stable); selected_workspace: device int32[pop].
 * elites = max(1, int(elitism_pct * pop)) best, copied unchanged to the first rows; every other selected slot is the
 * winner of a tournament of `tournament` (<= 8) distinct contenders; offspring pairs come from two uniform draws
 * of the selected list, uniform crossover with probability crossover_rate, per-gene mutation with mutation_rate. */
int b200bt_ga_next_generation(const double* params, const double* fitness, const int32_t* ranked, int pop, int genes,
                              const double* lo, const double* hi, const int* is_int, double elitism_pct,
                              int tournament, double crossover_rate, double mutation_rate, uint64_t seed,
                              uint32_t generation, int32_t* selected_workspace, double* params_out,
                              b200bt_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* B200BT_H_ */
