// Device code shared by the fused population sweep (sweep.cu) and the time-chunked sweep
// (sweep_chunked.cu): per-warp shared-memory working set, the bar scan, the event-batch
// arithmetic (calculate_metrics) and the score epilogue.
#pragma once
#include <math.h>
#include "common.cuh"

namespace b200bt {

// the fused sweep over a device-side list of individuals (sweep.cu): the exact fallback of the time-chunked sweeps
int launch_sweep(const float* price, int64_t ld_price, const float* rsi, int64_t ld_rsi, int P, int S, int64_t N,
                 const b200bt_individual* indiv, const int32_t* order, int pop, const int* pop_dev,
                 const b200bt_sweep_config* cfg_host, b200bt_lane_stats* stats, uint32_t* events, int64_t event_cap,
                 cudaStream_t stream);

constexpr int SW_WARPS = 8;         // warps (lanes of the sweep) per CTA
#ifndef B200BT_SW_MIN_BLOCKS
#define B200BT_SW_MIN_BLOCKS 2
#endif
constexpr int SW_MIN_BLOCKS = B200BT_SW_MIN_BLOCKS;    // CTAs per SM the register budget is held to (<= 64 regs/thread)
#ifndef B200BT_SW_GROUP
#define B200BT_SW_GROUP 512
#endif
#ifndef B200BT_SW_STAGES
#define B200BT_SW_STAGES 2
#endif
// 512 bars x 2 stages measured best on the C2 workload (256x3: +5 %, 128x4: +18 %; tools/build_variant.py)
constexpr int SW_GROUP = B200BT_SW_GROUP;     // bars per cp.async group (per stream)
constexpr int SW_STAGES = B200BT_SW_STAGES;   // shared-memory ring depth per warp
constexpr int SW_EVQ = 128;         // event queue entries per warp (>= 32 + 64 new events per window pair)
constexpr float SW_MARGIN = 1e-6f;  // relative width of the fp32 screening band

// Warp-uniform per-lane constants of the bar scan (shared memory; read on events only).
struct ScanConst {
    float os_f, ob_f;
    // screening multipliers: candidate (c) and definite (d) bounds
    float hiL_c, hiL_d, loL_c, loL_d;  // long : TP above, SL below
    float hiS_c, hiS_d, loS_c, loS_d;  // short: SL above, TP below
};

// Everything only the event-batch code touches lives in shared memory (one slot
// per warp) so that the bar scan keeps a small register footprint.
struct WarpAcc {
    double tp, sl, size, fee1, fee2;
    double equity, peak, maxdd;
    double tot_profit, tot_loss, largest_p, largest_l;
    double day_sum, pivot, s1, s2;
    long long day_cur;
    long long sum_dur;
    unsigned long long hash;
    uint32_t* ev_out;
    unsigned n_win, n_loss, n_days, n_events;
    int day_valid, pivot_set;
    double npivot, ns1, ns2;     // negative days (DayAcc)
    unsigned n_neg;
    unsigned gap_bar, gap_minutes;   // calendar clock of a glued series (b200bt_sweep_config); gap_bar = ~0u: none
};

// Per-warp shared-memory working set.
struct __align__(16) WarpShared {
    float ring[SW_STAGES][2][SW_GROUP];  // cp.async ring: [stage][0 price | 1 rsi][bar]
    uint2 evq[SW_EVQ];                   // event queue: (event word, price bits), consumed 32 at a time
    WarpAcc acc;
    ScanConst sc;
};

struct DayAcc {
    double pivot, s1, s2;
    unsigned n_days;
    int pivot_set;
    // the negative days alone (Sortino's downside deviation), same shifted accumulation
    double npivot = 0.0, ns1 = 0.0, ns2 = 0.0;
    unsigned n_neg = 0;
};

__device__ __forceinline__ void day_complete(DayAcc& a, double x) {
    // shifted-data accumulation of the daily pnl sums (exactly 0 variance for equal days)
    if (!a.pivot_set) { a.pivot = x; a.pivot_set = 1; }
    const double y = x - a.pivot;
    a.s1 += y;
    a.s2 += y * y;
    a.n_days += 1;
    if (x < 0.0) {
        if (a.n_neg == 0) a.npivot = x;
        const double z = x - a.npivot;
        a.ns1 += z;
        a.ns2 += z * z;
        a.n_neg += 1;
    }
}

// PnL of one trade record (strategy_evaluation.py:798,:819,:836): an entry record costs the entry fee,
// an exit record realises quantity * move - both fees, with quantity = position_size / entry_price.
__device__ __forceinline__ double record_pnl(bool active, unsigned w, float pf, unsigned w_prev, float p_prev,
                                             double size, double fee1, double fee2, int& dur) {
    dur = 0;
    if (!active) return 0.0;
    if (w & B200BT_EVENT_EXIT) {
        const double e = (double)p_prev, px = (double)pf;
        const double qty = __ddiv_rn(size, e);
        const double diff = (w_prev & B200BT_EVENT_SELL) ? __dsub_rn(e, px) : __dsub_rn(px, e);
        dur = (int)((w & 0x3fffffffu) - (w_prev & 0x3fffffffu));
        return __dsub_rn(__dmul_rn(qty, diff), fee2);
    }
    return -fee1;
}

// Consume `cnt` events in time order (lane j holds event j: word w, price pf); an exit record is
// priced against the entry record that precedes it -- lane j-1, or for lane 0 the last event of
// the previous batch (w_carry, p_carry).  The trade-record metrics of calculate_metrics
// (strategy_evaluation.py:97-188) are advanced in `acc` (shared memory, one slot per warp).
static __device__ __noinline__ void batch_core(WarpAcc* __restrict__ acc, int cnt, unsigned w, float pf, unsigned w_carry,
                                        float p_carry, long long minute0, int bar_minutes, int64_t ev_cap) {
    const int lane = threadIdx.x & 31;
    const bool active = lane < cnt;
    float p_prev = __shfl_up_sync(FULL, pf, 1);
    unsigned w_prev = __shfl_up_sync(FULL, w, 1);
    if (lane == 0) { p_prev = p_carry; w_prev = w_carry; }
    const unsigned bar = w & 0x3fffffffu;

    int dur;
    const double pnl = record_pnl(active, w, pf, w_prev, p_prev, acc->size, acc->fee1, acc->fee2, dur);
    // wins / losses
    const bool win = active && pnl > 0.0, loss = active && pnl < 0.0;
    const unsigned n_win = acc->n_win + __popc(__ballot_sync(FULL, win));
    const unsigned n_loss = acc->n_loss + __popc(__ballot_sync(FULL, loss));
    double largest_p = acc->largest_p, largest_l = acc->largest_l;
    if (__any_sync(FULL, pnl > largest_p)) largest_p = fmax(largest_p, warp_max_d(win ? pnl : 0.0));   // rare after warm-up
    if (__any_sync(FULL, pnl < largest_l)) largest_l = fmin(largest_l, warp_min_d(loss ? pnl : 0.0));
    const long long sum_dur = acc->sum_dur + __reduce_add_sync(FULL, dur);

    // equity curve: inclusive scan of pnl, running peak, drawdown
    double cs = pnl;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        double up = shfl_up_d(cs, d);
        if (lane >= d) cs += up;
    }
    // gains by one butterfly; losses = batch total - gains (the total comes free from the scan)
    const double gains = warp_sum_d(win ? pnl : 0.0);
    const double tot_profit = acc->tot_profit + gains;
    const double tot_loss = __any_sync(FULL, loss) ? acc->tot_loss + (__shfl_sync(FULL, cs, 31) - gains) : acc->tot_loss;
    const double eq = acc->equity + cs;
    const double peak_in = acc->peak;
    double pk = peak_in;
    if (__any_sync(FULL, active && eq > peak_in)) {   // a new equity peak inside the batch (uncommon for most lanes)
        pk = active ? eq : -INFINITY;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            double up = shfl_up_d(pk, d);
            if (lane >= d) pk = fmax(pk, up);
        }
        pk = fmax(pk, peak_in);
    }
    double maxdd = acc->maxdd;
    {
        // dd_j = (pk-eq)/pk; a new maximum needs (pk-eq) > maxdd*pk (screen with a safety factor, then divide)
        const double gap = __dsub_rn(pk, eq);
        const bool cand = active && gap > 0.0 && gap >= maxdd * pk * (1.0 - 1e-12);
        if (__any_sync(FULL, cand)) maxdd = fmax(maxdd, warp_max_d(cand ? __ddiv_rn(gap, pk) : 0.0));
    }
    const double batch_sum = shfl_d(cs, 31);
    const double equity_out = acc->equity + batch_sum;
    const double peak_out = shfl_d(pk, cnt - 1);

    // daily buckets: segmented sum by calendar day over the batch, merged with the carry day
    // calendar day of a record, relative to bar 0's day (32-bit: the host checks N*bar_minutes < 2^31 - 1440)
    const int day = active ? (int)(((unsigned)minute0 + bar * (unsigned)bar_minutes + (bar >= acc->gap_bar ? acc->gap_minutes : 0u)) / 1440u) : 0;
    DayAcc da{acc->pivot, acc->s1, acc->s2, acc->n_days, acc->pivot_set, acc->npivot, acc->ns1, acc->ns2, acc->n_neg};
    const int day_valid = acc->day_valid;
    const int day_cur = (int)acc->day_cur;
    double day_sum = acc->day_sum;
    const int first_day = __shfl_sync(FULL, day, 0);
    const int last_day = __shfl_sync(FULL, day, cnt - 1);
    if (first_day == last_day && (!day_valid || first_day == day_cur)) {
        // common case: the whole batch falls into the open day
        day_sum = (day_valid ? day_sum : 0.0) + batch_sum;
    } else {
        const int day_prev = __shfl_up_sync(FULL, day, 1);
        const int day_next = __shfl_down_sync(FULL, day, 1);
        const bool head = active && (lane == 0 || day != day_prev);
        const bool tail = active && (lane == cnt - 1 || day != day_next);
        double seg = pnl;
        bool flag = head;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            double up = shfl_up_d(seg, d);
            int fup = __shfl_up_sync(FULL, (int)flag, d);
            if (lane >= d && !flag) { seg += up; flag = fup; }
        }
        const bool merge_carry = day_valid && (first_day == day_cur);
        // a tail in the first segment (its day == first_day) absorbs the carry
        if (tail && merge_carry && day == first_day) seg += day_sum;
        const bool last_seg_tail = tail && (lane == cnt - 1);
        // completed days: every tail except the batch's last one (which stays open) ...
        const double x = (tail && !last_seg_tail) ? seg : 0.0;
        unsigned done = __ballot_sync(FULL, tail && !last_seg_tail);
        // ... plus the carried day when the batch starts on a later day;
        // fold in time order (carry first, then lanes ascending)
        if (day_valid && !merge_carry) day_complete(da, day_sum);
        while (done) {
            const int j = __ffs(done) - 1;
            done &= done - 1;
            day_complete(da, shfl_d(x, j));
        }
        day_sum = shfl_d(seg, cnt - 1);
    }

    // trade hash + optional event buffer
    const unsigned n_events = acc->n_events;
    const unsigned long long h = active ? event_hash(n_events + lane, w) : 0ull;
    const unsigned hlo = __reduce_xor_sync(FULL, (unsigned)h);
    const unsigned hhi = __reduce_xor_sync(FULL, (unsigned)(h >> 32));
    uint32_t* ev_out = acc->ev_out;
    if (ev_out && active) {
        const long long idx = (long long)n_events + lane;
        if (idx < ev_cap) ev_out[idx] = w;
    }
    __syncwarp();
    if (lane == 0) {
        acc->n_win = n_win; acc->n_loss = n_loss;
        acc->tot_profit = tot_profit; acc->tot_loss = tot_loss;
        acc->largest_p = largest_p; acc->largest_l = largest_l;
        acc->sum_dur = sum_dur;
        acc->equity = equity_out; acc->peak = peak_out; acc->maxdd = maxdd;
        acc->pivot = da.pivot; acc->s1 = da.s1; acc->s2 = da.s2; acc->n_days = da.n_days; acc->pivot_set = da.pivot_set;
        acc->npivot = da.npivot; acc->ns1 = da.ns1; acc->ns2 = da.ns2; acc->n_neg = da.n_neg;
        acc->day_sum = day_sum; acc->day_cur = last_day; acc->day_valid = 1;
        acc->hash ^= ((unsigned long long)hhi << 32) | hlo;
        acc->n_events = n_events + cnt;
    }
    __syncwarp();
}

// Fused kernel: consume 32 (or the last few) queued events; batches there start on an entry record.
__device__ __forceinline__ void process_batch(WarpShared* __restrict__ ws, unsigned qtail, int cnt,
                                              long long minute0, int bar_minutes, int64_t ev_cap) {
    const uint2 evt = ws->evq[(qtail + (threadIdx.x & 31)) & (SW_EVQ - 1)];
    batch_core(&ws->acc, cnt, evt.x, __uint_as_float(evt.y), 0u, 0.f, minute0, bar_minutes, ev_cap);
}

// Metrics -> calculate_metrics' scalars and _calculate_strategy_score (strategy_evaluation.py:97-228,:579-633).
__device__ __forceinline__ void finalize_lane(const WarpAcc& a, const b200bt_sweep_config& cfg, b200bt_lane_stats& o) {
    DayAcc da{a.pivot, a.s1, a.s2, a.n_days, a.pivot_set, a.npivot, a.ns1, a.ns2, a.n_neg};
    if (a.day_valid) day_complete(da, a.day_sum);
    const double n_rec = (double)a.n_events;
    o.n_records = n_rec;
    o.n_wins = (double)a.n_win;
    o.n_losses = (double)a.n_loss;
    o.total_profit = a.tot_profit;
    o.total_loss = a.tot_loss;
    o.net_profit = a.tot_profit + a.tot_loss;
    o.max_drawdown = a.maxdd;
    o.n_days = (double)da.n_days;
    o.largest_profit = a.largest_p;
    o.largest_loss = a.largest_l;
    o.sum_duration_bars = (double)a.sum_dur;
    o.trade_hash = a.hash;
    double sharpe = 0.0, win_rate = 0.0, pf = 0.0;
    if (a.n_events >= 2) {
        win_rate = (double)a.n_win / n_rec;
        pf = (a.tot_loss != 0.0) ? fabs(a.tot_profit / a.tot_loss) : INFINITY;
        if (da.n_days > 1) {
            const double nd = (double)da.n_days;
            const double mean_y = da.s1 / nd;
            double var = da.s2 / nd - mean_y * mean_y;
            if (var < 0.0) var = 0.0;
            const double sd = sqrt(var);
            const double mean = da.pivot + mean_y;
            sharpe = sd > 0.0 ? (mean / sd) * sqrt(252.0) : 0.0;
        }
    }
    o.sharpe_ratio = sharpe;
    o.win_rate = win_rate;
    o.profit_factor = pf;
    // calculate_advanced_metrics (:250-263, :307-312): only a lane with >= 2 records has daily buckets
    double mean_daily = 0.0, downside = 0.0, sortino = 0.0;
    if (a.n_events >= 2 && da.n_days > 0) {
        mean_daily = da.pivot + da.s1 / (double)da.n_days;
        if (da.n_neg > 0) {
            const double nn = (double)da.n_neg, my = da.ns1 / nn;
            double var = da.ns2 / nn - my * my;
            downside = sqrt(var < 0.0 ? 0.0 : var);
        }
        sortino = downside > 0.0 ? (mean_daily / downside) * sqrt(252.0) : INFINITY;
    }
    o.sortino_ratio = sortino;
    o.n_negative_days = (a.n_events >= 2) ? (double)da.n_neg : 0.0;
    o.downside_deviation = downside;
    o.mean_daily_pnl = mean_daily;
    // every scalar key of the metrics dict can be the primary metric (:589-590)
    const double ret_pct = (o.net_profit / cfg.initial_capital) * 100.0;
    const double avg_p = a.n_win ? a.tot_profit / (double)a.n_win : 0.0, avg_l = a.n_loss ? a.tot_loss / (double)a.n_loss : 0.0;
    // calculate_advanced_metrics :302-310 (total_trades > 0)
    const double expectancy = a.n_events ? win_rate * avg_p - (1.0 - win_rate) * fabs(avg_l) : 0.0;
    double primary;
    switch (cfg.primary) {
        case B200BT_PRIMARY_RETURN_PCT: primary = ret_pct; break;
        case B200BT_PRIMARY_PROFIT_FACTOR: primary = pf; break;
        case B200BT_PRIMARY_WIN_RATE: primary = win_rate; break;
        case B200BT_PRIMARY_NET_PROFIT: primary = o.net_profit; break;
        case B200BT_PRIMARY_TOTAL_TRADES: primary = n_rec; break;
        case B200BT_PRIMARY_MAX_DRAWDOWN: primary = a.maxdd; break;
        case B200BT_PRIMARY_TOTAL_PROFIT: primary = a.tot_profit; break;
        case B200BT_PRIMARY_TOTAL_LOSS: primary = a.tot_loss; break;
        case B200BT_PRIMARY_LARGEST_PROFIT: primary = a.largest_p; break;
        case B200BT_PRIMARY_LARGEST_LOSS: primary = a.largest_l; break;
        case B200BT_PRIMARY_AVERAGE_PROFIT: primary = avg_p; break;
        case B200BT_PRIMARY_AVERAGE_LOSS: primary = avg_l; break;
        case B200BT_PRIMARY_SORTINO: primary = sortino; break;
        case B200BT_PRIMARY_EXPECTANCY: primary = expectancy; break;
        case B200BT_PRIMARY_CALMAR: primary = a.maxdd > 0.0 ? (ret_pct / 100.0) / a.maxdd : INFINITY; break;          // :243-249
        case B200BT_PRIMARY_PROFIT_PER_DAY: primary = mean_daily; break;
        case B200BT_PRIMARY_RECOVERY_FACTOR: primary = a.maxdd > 0.0 ? o.net_profit / (a.maxdd * 10000.0) : INFINITY; break;   // :296-300
        case B200BT_PRIMARY_ZERO: primary = 0.0; break;
        default: primary = sharpe; break;
    }
    double score = primary;
    if (cfg.secondary_mask & B200BT_SEC_MAX_DRAWDOWN) score *= (1.0 - a.maxdd);
    if (cfg.secondary_mask & B200BT_SEC_WIN_RATE) score *= (1.0 + win_rate);
    if (cfg.secondary_mask & B200BT_SEC_PROFIT_FACTOR) score *= (pf / 2.0);
    if (cfg.secondary_mask & B200BT_SEC_EXPECTANCY) score *= (1.0 + fmin(expectancy / 100.0, 1.0));
    o.score = score;
}

// Initial metrics state of a lane.
__device__ __forceinline__ void init_acc(WarpAcc& a, const b200bt_individual& iv, const b200bt_sweep_config& cfg, uint32_t* ev_out) {
    const double initial_capital = cfg.initial_capital;
    a.gap_bar = cfg.gap_bar > 0 ? (unsigned)cfg.gap_bar : 0xffffffffu;
    a.gap_minutes = (unsigned)cfg.gap_minutes;
    a.tp = iv.take_profit; a.sl = iv.stop_loss; a.size = iv.position_size;
    a.fee1 = __dmul_rn(a.size, 0.001); a.fee2 = __dmul_rn(a.size, 0.002);
    a.equity = initial_capital; a.peak = initial_capital; a.maxdd = 0.0;
    a.tot_profit = a.tot_loss = a.largest_p = a.largest_l = 0.0;
    a.day_sum = a.pivot = a.s1 = a.s2 = 0.0;
    a.day_cur = 0; a.sum_dur = 0; a.hash = 0ull;
    a.ev_out = ev_out;
    a.n_win = a.n_loss = a.n_days = a.n_events = 0;
    a.day_valid = a.pivot_set = 0;
    a.npivot = a.ns1 = a.ns2 = 0.0;
    a.n_neg = 0;
}

__device__ __forceinline__ void init_scan_const(ScanConst& c, const b200bt_individual& iv) {
    c.os_f = iv.rsi_lo;
    c.ob_f = iv.rsi_hi;
    const double mg = (double)SW_MARGIN, tp = iv.take_profit, sl = iv.stop_loss;
    c.hiL_c = (float)((1.0 + tp) * (1.0 - mg));
    c.hiL_d = (float)((1.0 + tp) * (1.0 + mg));
    c.loL_c = (float)((1.0 - sl) * (1.0 + mg));
    c.loL_d = (float)((1.0 - sl) * (1.0 - mg));
    c.loS_c = (float)((1.0 - tp) * (1.0 + mg));
    c.loS_d = (float)((1.0 - tp) * (1.0 - mg));
    c.hiS_c = (float)((1.0 + sl) * (1.0 - mg));
    c.hiS_d = (float)((1.0 + sl) * (1.0 + mg));
}

__device__ __forceinline__ void cp_async16(float* smem_dst, const float* gmem_src) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"((unsigned)__cvta_generic_to_shared(smem_dst)), "l"(gmem_src) : "memory");
}
__device__ __forceinline__ void cp_async4(float* smem_dst, const float* gmem_src) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"((unsigned)__cvta_generic_to_shared(smem_dst)), "l"(gmem_src) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N_>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N_) : "memory"); }

// ---- mbarrier + bulk async copies (sm_90+ PTX; the tile ring of the thread-per-lane scan) ------------------------
__device__ __forceinline__ unsigned smem_u32(const void* p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(unsigned long long* bar, unsigned count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_fence_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_arrive_expect_tx(unsigned long long* bar, unsigned bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(unsigned long long* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(unsigned long long* bar, unsigned parity) {
    unsigned ok;
    asm volatile("{\n.reg .pred p;\nmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\nselp.u32 %0, 1, 0, p;\n}"
                 : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity) : "memory");
    return ok != 0;
}
// bounded wait (there is no unbounded one): false when the phase has not completed `cycles` SM clocks after the first failed poll (the caller gives the
// work up and has it redone by the exact fallback instead of spinning for ever on a copy that does not arrive)
__device__ __forceinline__ bool mbar_wait_bounded(unsigned long long* bar, unsigned parity, long long cycles) {
    if (mbar_try_wait(bar, parity)) return true;
    const long long t0 = clock64();
    while (!mbar_try_wait(bar, parity))
        if (clock64() - t0 > cycles) return false;
    return true;
}
// global -> shared bulk copy (TMA engine, 16-byte aligned, size a multiple of 16), completion counted on `bar`
__device__ __forceinline__ void bulk_g2s(void* smem_dst, const void* gmem_src, unsigned bytes, unsigned long long* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(smem_u32(smem_dst)), "l"(gmem_src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// Machine state of one lane (warp-uniform registers).
struct Machine {
    int pos;                                   // 0 flat, +1 long, -1 short
    float e;                                   // entry price
    float rlo, rhi, plo, phi;                  // event thresholds of the current state (screening bounds)
    int entry_bar;                             // bar of the open position's entry (chunk-boundary check)
    unsigned qhead;                            // events pushed so far (queue head)
};

__device__ __forceinline__ bool fires(const Machine& m, float p, float r) {
    return (r < m.rlo) | (r > m.rhi) | (p <= m.plo) | (p >= m.phi);
}

// Advance the machine through every event of one 32-bar window (lane l holds bar t0+l).
// `emit` = false runs the machine without recording events (warm-up bars of a time chunk).
// `win` points at the window's 32 prices in the shared-memory ring (RSI values SW_GROUP floats further):
// the event bar's price / RSI are re-read from there with a warp-uniform address.
__device__ __forceinline__ void scan_window(const float p, const float r, const float* __restrict__ win, const int t0,
                                            WarpShared* __restrict__ ws, const ScanConst& c, Machine& m,
                                            const bool emit = true) {
    unsigned live = FULL;  // bars of the window not yet consumed
    while (true) {
        const unsigned hit = __ballot_sync(FULL, fires(m, p, r)) & live;
        if (hit == 0) break;
        const int kk = __ffs(hit) - 1;
        const float pk = win[kk];
        const float rk = win[SW_GROUP + kk];
        live = 0xfffffffeu << kk;
        const unsigned bar = (unsigned)(t0 + kk);
        unsigned word;
        bool ev = true;
        if (m.pos == 0) {
            // entry (strategy_evaluation.py:784-813): long has priority over short
            const bool lng = rk < c.os_f;
            m.e = pk;
            m.entry_bar = (int)bar;
            m.pos = lng ? 1 : -1;
            m.rlo = lng ? -INFINITY : c.os_f;
            m.rhi = lng ? c.ob_f : INFINITY;
            m.phi = pk * (lng ? c.hiL_c : c.hiS_c);
            m.plo = pk * (lng ? c.loL_c : c.loS_c);
            word = lng ? bar : (bar | B200BT_EVENT_SELL);
        } else {
            // exit candidate (:815-847); an RSI reversal is always definite, a price trigger inside the
            // fp32 screening band is decided with the reference's float64 expression
            if (!((rk < m.rlo) || (rk > m.rhi))) {
                const bool lng = m.pos > 0;
                const float hd = m.e * (lng ? c.hiL_d : c.hiS_d), ld = m.e * (lng ? c.loL_d : c.loS_d);
                if (!((pk >= hd) || (pk <= ld))) {
                    const double ed = (double)m.e, pd = (double)pk;
                    const double q = lng ? __ddiv_rn(__dsub_rn(pd, ed), ed) : __ddiv_rn(__dsub_rn(ed, pd), ed);
                    ev = (q >= ws->acc.tp) || (q <= -ws->acc.sl);
                }
            }
            if (ev) {
                word = bar | B200BT_EVENT_EXIT | (m.pos > 0 ? B200BT_EVENT_SELL : 0u);
                m.pos = 0;
                m.rlo = c.os_f; m.rhi = c.ob_f;
                m.plo = -INFINITY; m.phi = INFINITY;
            }
        }
        if (ev) {
            // every lane stores the same word to the same slot (one wavefront); while not recording, the
            // head does not advance and the slot is simply overwritten by the next event
            ws->evq[m.qhead & (SW_EVQ - 1)] = make_uint2(word, __float_as_uint(pk));
            m.qhead += emit ? 1u : 0u;
        }
    }
}

}  // namespace b200bt
