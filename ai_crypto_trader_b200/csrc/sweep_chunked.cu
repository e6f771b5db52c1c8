// Family 2, time-parallel form: the population sweep with every expensive lane split into
// TIME CHUNKS that are scanned concurrently (sm_100a).
//
// The trade state machine (strategy_evaluation.py:746-878) is serial in time, and the lanes of a
// GA population differ by two to three orders of magnitude in trade count, so at moderate
// population sizes the fused kernel (sweep.cu) is bounded by the serial event chain of its few
// heaviest lanes.  The machine, however, forgets: whenever it is flat, its future does not depend
// on its past.  A chunk [T_c, T_{c+1}) is therefore scanned by its own warp, which starts `warm`
// bars early in the flat state without recording, and records from T_c on.  Two trajectories that
// are ever flat at the same bar coincide from then on, so after the warm-up the chunk's assumed
// state (position side + entry bar) is almost always the true one.  It is VERIFIED, not trusted:
//   scan kernels    chunk_scan_kernel: one WARP per (individual, symbol, chunk) of the expensive lanes
//                   (b200bt_sweep_chunked), or lane_scan_kernel: every lane cut into the same K chunks and one
//                   THREAD per (individual, symbol, chunk) (b200bt_sweep_tiled, see "thread-per-lane scan").
//                   Events -> blocks of a global pool (bump allocator, singly linked per chunk), plus the
//                   chunk's assumed state at T_c and its end state.
//   verify / repair a chunk whose assumed state differs from its predecessor's end state is re-scanned from the true
//                   state until the trajectory meets the recorded one; the rest of the recorded chain is spliced on
//                   (chunk_scan_item<REPAIR>).  chunk_repair_kernel: one warp per chunk, on the critical path;
//                   lane_repair_kernel: one warp per lane, in time order, beside the metrics kernels (finish_chunks).
//   metrics kernels one warp per (individual, symbol, chunk) again (see "metrics, chunk-parallel" below), then
//                   one thread per (individual, symbol) checks end state of chunk c-1 == assumed state
//                   of chunk c for every boundary and merges the chunks' partial metrics.
// A lane with any mismatching boundary is flagged; the host re-evaluates flagged lanes with the
// fused (serial) kernel, so results never depend on the speculation being right.
#include <stddef.h>
#include "sweep_dev.cuh"

namespace b200bt {

constexpr int CK_BLOCK = 256;   // events per pool block
constexpr unsigned EVENT_BAR_MASK = ~(B200BT_EVENT_EXIT | B200BT_EVENT_SELL);   // event word = bar | flags

// Segment (one chunk of one lane) vocabulary.  A chunk's state at a bar is (position side, entry bar), the entry bar -1
// when flat.  A chunk that LOST its events (full pool, a tile that did not arrive, a warp not packed for the thread-per-lane
// scan) has no chain: its count is SEG_LOST, which sends it to the repair pass or its lane to the exact fallback.
constexpr unsigned SEG_LOST = 0xffffffffu;

__device__ __forceinline__ int2 seg_state(int pos, int entry_bar) { return make_int2(pos, pos != 0 ? entry_bar : -1); }

// The event pool and the per-segment tables, shared by every kernel of the time-chunked sweep.
struct SegTables {
    uint2* pool; int pool_blocks; int* next; unsigned* alloc; int* overflow;    // [pool_blocks][CK_BLOCK] events, chain links
    int* seg_first; unsigned* seg_count; int2* seg_in; int2* seg_out;          // [segs]: first block, events, assumed / end state
};

__device__ __forceinline__ void mark_lost(const SegTables& T, int seg) {
    T.seg_in[seg] = seg_state(0, 0);
    T.seg_out[seg] = seg_state(0, 0);
    T.seg_count[seg] = SEG_LOST;
}

// Appends a pool block to the chain of segment `seg`, whose last block is `cur_block` (-1: none yet).  -> the block, or
// -1 when the pool is exhausted (the overflow flag is raised; the caller drops the chunk's further events).
__device__ __forceinline__ int pool_append(const SegTables& T, int seg, int cur_block) {
    const int b = (int)atomicAdd(T.alloc, 1u);
    if (b >= T.pool_blocks) { atomicExch(T.overflow, 1); return -1; }
    T.next[b] = -1;
    if (cur_block < 0) T.seg_first[seg] = b; else T.next[cur_block] = b;
    return b;
}

struct ChunkScanArgs {
    const float* price; int64_t ld_price;
    const float* rsi; int64_t ld_rsi;
    int P, S; int64_t N;
    const b200bt_individual* indiv;
    const b200bt_chunk_item* items; int n_items; int n_seg;   // n_seg = segments per symbol
    int warm;
    SegTables T;
    const int32_t* n_chunks;
    unsigned char* redo;  // repair pass of the overlapped tail: individuals whose metrics must be recomputed
};

__device__ __forceinline__ int64_t chunk_begin(int64_t N, int c, int K) {
    if (c >= K) return N;
    return ((N * c) / K) & ~(int64_t)(SW_GROUP - 1);   // group aligned
}

// REPAIR = false: speculative pass over every (work item, symbol), warm-up from the flat state.
// REPAIR = true : re-scan of chunks whose assumed state was wrong, started AT T_c from the now known
//                 true state (end state of the preceding chunk); one work item per listed chunk.
template <bool VEC16, bool REPAIR>
__device__ __forceinline__ bool chunk_scan_item(const ChunkScanArgs& A, const b200bt_chunk_item item, const int sym, WarpShared* ws) {
    const int lane = threadIdx.x & 31;
    const b200bt_individual iv = A.indiv[item.individual];
    if (lane == 0) {
        ScanConst sc0;
        init_scan_const(sc0, iv);
        ws->sc = sc0;
        ws->acc.tp = iv.take_profit;   // only the screening-band decision reads these here
        ws->acc.sl = iv.stop_loss;
    }
    __syncwarp();
    const ScanConst c = ws->sc;
    const float* __restrict__ pr = A.price + (int64_t)sym * A.ld_price;
    const float* __restrict__ rr = A.rsi + ((int64_t)sym * A.P + iv.rsi_row) * A.ld_rsi;

    const int n = (int)A.N;
    const int T0 = (int)chunk_begin(A.N, item.chunk, item.n_chunks);       // first recorded bar
    const int T1 = (int)chunk_begin(A.N, item.chunk + 1, item.n_chunks);   // end (exclusive)
    int s0 = REPAIR ? T0 : T0 - A.warm;
    if (s0 < 0 || item.chunk == 0) s0 = 0;
    s0 &= ~(SW_GROUP - 1);
    const int seg = sym * A.n_seg + item.segment;

    Machine m;
    m.pos = 0; m.e = 0.f; m.entry_bar = 0;
    m.rlo = iv.rsi_lo; m.rhi = iv.rsi_hi; m.plo = -INFINITY; m.phi = INFINITY;
    m.qhead = 0;
    unsigned qtail = 0;
    if (REPAIR) {
        // true state at T0 = end state of the preceding chunk (position side, entry bar -> entry price)
        const int2 z = A.T.seg_out[seg - 1];
        if (z.x != 0) {
            const float e = __ldg(pr + z.y);
            m.pos = z.x; m.e = e; m.entry_bar = z.y;
            if (z.x > 0) {
                m.rlo = -INFINITY; m.rhi = c.ob_f;
                m.phi = e * c.hiL_c; m.plo = e * c.loL_c;
            } else {
                m.rlo = c.os_f; m.rhi = INFINITY;
                m.phi = e * c.hiS_c; m.plo = e * c.loS_c;
            }
        }
    }

    // REPAIR: the chain the speculative scan recorded for this chunk and the state it assumed at T0.  Two trajectories that
    // are in the same state at the same bar coincide from there on, so the re-scan stops at the first group boundary at
    // which its state equals the recorded trajectory's and splices the rest of the recorded events (below).
    int old_block = -1, old_idx = 0, old_pos = 0, old_ebar = -1;
    unsigned old_left = 0;
    bool old_ok = false, spliced = false;
    if (REPAIR) {
        const unsigned oc = A.T.seg_count[seg];
        const int2 oin = A.T.seg_in[seg];
        old_ok = oc != SEG_LOST;     // (a chunk whose events were dropped has no chain to splice)
        old_left = old_ok ? oc : 0u;
        old_block = A.T.seg_first[seg];
        old_pos = oin.x; old_ebar = oin.x != 0 ? oin.y : -1;
    }

    // event sink: 32 queued events -> one coalesced 256-byte store into the chunk's current pool block
    int cur_block = -1, fill = CK_BLOCK, dead = 0;
    auto flush = [&](int cnt) {
        if (fill == CK_BLOCK && !dead) {
            int b = 0;
            if (lane == 0) b = pool_append(A.T, seg, cur_block);
            b = __shfl_sync(FULL, b, 0);
            if (b < 0) dead = 1; else { cur_block = b; fill = 0; }
        }
        if (!dead) {
            if (lane < cnt) A.T.pool[(int64_t)cur_block * CK_BLOCK + fill + lane] = ws->evq[(qtail + lane) & (SW_EVQ - 1)];
            fill += 32;   // only the last flush of a chunk is partial
        }
        qtail += cnt;
    };

    constexpr int G = SW_GROUP;
    float* const sp = &ws->ring[0][0][0];
    const int n_full = n / G;
    const int g_begin = s0 / G, g_end = (T1 + G - 1) / G;
    int issued = g_begin;
    float* idst = sp + (g_begin % SW_STAGES) * (2 * G) + (VEC16 ? lane * 4 : lane);
    const float* ip = pr + (int64_t)g_begin * G + (VEC16 ? lane * 4 : lane);
    const float* ir = rr + (int64_t)g_begin * G + (VEC16 ? lane * 4 : lane);
    auto issue = [&]() {
        if (issued < n_full && issued < g_end) {
            if (VEC16) {
#pragma unroll
                for (int i = 0; i < G / 128; ++i) {
                    cp_async16(idst + i * 128, ip + i * 128);
                    cp_async16(idst + G + i * 128, ir + i * 128);
                }
            } else {
#pragma unroll
                for (int i = 0; i < G / 32; ++i) {
                    cp_async4(idst + i * 32, ip + i * 32);
                    cp_async4(idst + G + i * 32, ir + i * 32);
                }
            }
        } else if (issued < g_end) {
            const float qnan = __int_as_float(0x7fc00000);   // ragged last group of the series
            float* dst = sp + (issued % SW_STAGES) * (2 * G);
            for (int i = lane; i < G; i += 32) {
                const int t = issued * G + i;
                dst[i] = t < n ? __ldg(pr + t) : qnan;
                dst[G + i] = t < n ? __ldg(rr + t) : qnan;
            }
        }
        cp_async_commit();
        ++issued;
        ip += G; ir += G;
        idst = (issued % SW_STAGES == 0) ? idst - (SW_STAGES - 1) * (2 * G) : idst + 2 * G;
    };
#pragma unroll
    for (int g = 0; g < SW_STAGES - 1; ++g) issue();
    int cstage = g_begin % SW_STAGES;
    const float* cur = sp + cstage * (2 * G) + lane;
    for (int g = g_begin; g < g_end; ++g) {
        issue();
        cp_async_wait<SW_STAGES - 1>();
        __syncwarp();
        const bool emit = g * G >= T0;
        if (g * G == T0 && lane == 0) A.T.seg_in[seg] = seg_state(m.pos, m.entry_bar);
        if (REPAIR && old_ok && g > g_begin) {
            // state of the recorded trajectory before bar tb = g * G: consume its events with bar < tb
            const unsigned tb = (unsigned)(g * G);
            while (old_left) {
                const int n_here = (int)min(min(32u, old_left), (unsigned)(CK_BLOCK - old_idx));
                const unsigned word = lane < n_here ? A.T.pool[(int64_t)old_block * CK_BLOCK + old_idx + lane].x : 0xffffffffu;
                const int k = __popc(__ballot_sync(FULL, lane < n_here && (word & EVENT_BAR_MASK) < tb));    // (bars ascend: a prefix)
                if (k) {
                    const unsigned last = __shfl_sync(FULL, word, k - 1);
                    old_pos = (last & B200BT_EVENT_EXIT) ? 0 : ((last & B200BT_EVENT_SELL) ? -1 : 1);
                    old_ebar = (last & B200BT_EVENT_EXIT) ? -1 : (int)(last & EVENT_BAR_MASK);
                    old_idx += k; old_left -= (unsigned)k;
                    if (old_idx == CK_BLOCK && old_left) { old_block = A.T.next[old_block]; old_idx = 0; }
                }
                if (k < n_here) break;
            }
            if (m.pos == old_pos && (m.pos == 0 || m.entry_bar == old_ebar)) {
                // same state at the same bar: the rest of the recorded chain is this trajectory's; copy it behind the
                // re-scanned events (the chunk's end state, and with it every later chunk, stands as recorded)
                while (old_left) {
                    const int n_here = (int)min(min(32u, old_left), (unsigned)(CK_BLOCK - old_idx));
                    if (lane < n_here) ws->evq[(m.qhead + lane) & (SW_EVQ - 1)] = A.T.pool[(int64_t)old_block * CK_BLOCK + old_idx + lane];
                    m.qhead += (unsigned)n_here;
                    old_idx += n_here; old_left -= (unsigned)n_here;
                    if (old_idx == CK_BLOCK && old_left) { old_block = A.T.next[old_block]; old_idx = 0; }
                    __syncwarp();
                    while (m.qhead - qtail >= 32) flush(32);
                    __syncwarp();
                }
                spliced = true;
                break;
            }
        }
        const float* w = cur;
        int t0 = g * G;
#pragma unroll 1
        for (int v = 0; v < G / 64; ++v, w += 64, t0 += 64) {
            const float p0 = w[0], r0 = w[G];
            const float p1 = w[32], r1 = w[G + 32];
            const unsigned h0 = __ballot_sync(FULL, fires(m, p0, r0));
            const unsigned h1 = __ballot_sync(FULL, fires(m, p1, r1));
            if (h0 | h1) {
                if (h0) scan_window(p0, r0, w - lane, t0, ws, c, m, emit);
                scan_window(p1, r1, w - lane + 32, t0 + 32, ws, c, m, emit);
                while (m.qhead - qtail >= 32) {
                    __syncwarp();
                    flush(32);
                }
            }
        }
        __syncwarp();
        if (++cstage == SW_STAGES) { cstage = 0; cur -= (SW_STAGES - 1) * (2 * G); } else cur += 2 * G;
    }
    cp_async_wait<0>();
    if (lane == 0 && !spliced) {
        const int2 st = seg_state(m.pos, m.entry_bar);
        A.T.seg_out[seg] = st;
        if (T0 >= T1) A.T.seg_in[seg] = st;   // empty chunk: its assumed state is the state after the warm-up
    }
    if (!spliced && item.chunk == item.n_chunks - 1 && m.pos != 0) {
        // force-close at the last bar (:849-876)
        const float pl = __ldg(pr + (A.N - 1));
        const unsigned word = (unsigned)(A.N - 1) | B200BT_EVENT_EXIT | (m.pos > 0 ? B200BT_EVENT_SELL : 0u);
        if (lane == 0) ws->evq[m.qhead & (SW_EVQ - 1)] = make_uint2(word, __float_as_uint(pl));
        ++m.qhead;
    }
    __syncwarp();
    while (m.qhead != qtail) flush((int)min(32u, m.qhead - qtail));
    if (lane == 0) A.T.seg_count[seg] = dead ? SEG_LOST : m.qhead;
    __syncwarp();
    return spliced;      // REPAIR: the chunk's recorded end state stands
}

template <bool VEC16>
__global__ void __launch_bounds__(SW_WARPS * 32, 3)
chunk_scan_kernel(const ChunkScanArgs A) {   // by value, not __grid_constant__ (see sweep.cu)
    extern __shared__ __align__(16) unsigned char s_raw[];
    WarpShared* ws = reinterpret_cast<WarpShared*>(s_raw) + (threadIdx.x >> 5);
    const int sym = (int)(blockIdx.x % (unsigned)A.S);
    const int it = (int)(blockIdx.x / (unsigned)A.S) * SW_WARPS + (threadIdx.x >> 5);
    if (it >= A.n_items) return;
    chunk_scan_item<VEC16, false>(A, A.items[it], sym, ws);
}

// Verification and repair.  Two kernels share chunk_scan_item<REPAIR> (re-scan from the true state until the trajectory
// meets the recorded one, then splice the recorded chain on); neither needs a work list or anything read by the host.
//
// chunk_repair_kernel (critical path): one warp per (chunk, symbol), handed out by a counter.  The warp compares its chunk's
// assumed start state with the predecessor's recorded end state and re-scans on a mismatch.  All wrong chunks of a lane are
// repaired CONCURRENTLY, each trusting its predecessor's recorded end state -- which stands whenever the predecessor's own
// re-scan finds its way back to the recorded trajectory, i.e. almost always.  (A predecessor that is being rewritten at
// the same moment is a benign race on an aligned 8-byte word: whichever value is read becomes the chunk's published start
// state, and the boundary is checked again below and in lane_combine_kernel.)
template <bool VEC16>
__global__ void __launch_bounds__(SW_WARPS * 32, 3)
chunk_repair_kernel(const ChunkScanArgs A, unsigned* __restrict__ work) {
    extern __shared__ __align__(16) unsigned char s_raw[];
    WarpShared* ws = reinterpret_cast<WarpShared*>(s_raw) + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    const int64_t total = (int64_t)A.n_items * A.S;
    for (;;) {
        unsigned t = 0;
        if (lane == 0) t = atomicAdd(work, 1u);
        t = __shfl_sync(FULL, t, 0);
        if ((int64_t)t >= total) break;
        const int it = (int)(t / (unsigned)A.S), sym = (int)(t - (unsigned)it * (unsigned)A.S);
        const b200bt_chunk_item item = A.items[it];
        if (item.chunk == 0) continue;
        const int seg = sym * A.n_seg + item.segment;
        const int2 a = A.T.seg_in[seg], z = A.T.seg_out[seg - 1];
        if ((a.x != z.x || a.y != z.y) && A.T.seg_count[seg - 1] != SEG_LOST) chunk_scan_item<VEC16, true>(A, item, sym, ws);
    }
}

// lane_repair_kernel (beside the metrics kernels): one warp per (individual, symbol) lane walks the lane's boundaries in
// time order and re-scans where a chunk does not follow from its predecessor, checking the next boundary against the end
// state it has just produced -- so the lane is consistent when the warp leaves it, however many chunks in a row a re-scan
// runs through without meeting its recorded trajectory (lanes that hold one position across many chunks).  After
// chunk_repair_kernel only those cascades are left.  Individuals it touches are flagged in A.redo (metrics recomputed).
template <bool VEC16>
__global__ void __launch_bounds__(SW_WARPS * 32, 3)
lane_repair_kernel(const ChunkScanArgs A, const int pop, const int32_t* __restrict__ seg_base, unsigned* __restrict__ work) {
    extern __shared__ __align__(16) unsigned char s_raw[];
    WarpShared* ws = reinterpret_cast<WarpShared*>(s_raw) + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    const int lanes = pop * A.S;
    for (;;) {
        int t = 0;
        if (lane == 0) t = (int)atomicAdd(work, 1u);
        t = __shfl_sync(FULL, t, 0);
        if (t >= lanes) break;
        const int ind = t / A.S, sym = t - ind * A.S;
        const int K = A.n_chunks[ind];
        const int sb = seg_base[ind];
        const int base = sym * A.n_seg + sb;
        int2 prev = A.T.seg_out[base];
        bool usable = A.T.seg_count[base] != SEG_LOST;      // (a chunk that lost events to a full pool ends the walk: the lane is flagged later)
        for (int c = 1; c < K && usable; ++c) {
            const int2 a = A.T.seg_in[base + c];
            if (a.x != prev.x || a.y != prev.y) {
                b200bt_chunk_item item;
                item.individual = ind; item.chunk = c; item.segment = sb + c; item.n_chunks = K;
                if (A.redo && lane == 0) A.redo[ind] = 1;
                chunk_scan_item<VEC16, true>(A, item, sym, ws);      // (ends with a __syncwarp: its stores are visible to the warp)
            }
            prev = A.T.seg_out[base + c];
            usable = A.T.seg_count[base + c] != SEG_LOST;
        }
    }
}

// ---- thread-per-lane scan ---------------------------------------------------------------------------
// The warp-per-lane scan above spends a full warp on the scalar event chain of one lane.  With every lane cut
// into the SAME K time chunks there are pop x S x K independent machines -- enough to give each one a THREAD:
// a warp takes (warp-slot, chunk, symbol) work items, stages tiles of the price row and of the (at most
// LS_RSI_ROWS) RSI rows its 32 machines read through its own shared-memory ring (see "Tile movement"), and every
// thread steps its own machine through the tile, four bars per step.  The event path then runs in SIMT fashion
// for up to 32 lanes at once and all threads walk the same bars (no tail).  Events go to the same pool / segment
// tables as the warp scan, so verification, repair and the metrics kernels are shared.
#ifndef B200BT_LS_T
#define B200BT_LS_T 128
#endif
constexpr int LS_T = B200BT_LS_T;       // bars per tile
constexpr int LS_STRIDE = LS_T + 4;     // row stride in floats (16-byte aligned rows, rows 8 apart share banks)
#ifndef B200BT_LS_THREADS
#define B200BT_LS_THREADS 256
#endif
constexpr int LS_THREADS = B200BT_LS_THREADS;

constexpr int LS_ZONE = 32;             // bars per zone-map block

// Zone map: (min, max) of every 32-bar block ("coarse") and of every 4-bar group ("fine") of the price row and of each
// RSI row, NaNs ignored.  A machine whose thresholds lie outside a range cannot fire inside it: the scan skips a 32-bar
// block after four compares when no machine of the warp can fire in it, and inside a block it tests each 4-bar group
// against the group's precomputed range (two 8-byte loads, four compares) instead of folding the eight values itself.
// Layout: coarse [S][P + 1][zone_row_stride(N)] float2, then fine [S][P + 1][zone_fine_stride(N)] float2; row 0 = price;
// both strides keep rows 16-byte aligned and pad with (NaN, NaN) (every compare false).
__global__ void __launch_bounds__(256)
zone_map_kernel(const float* __restrict__ price, int64_t ld_price, const float* __restrict__ rsi, int64_t ld_rsi, int P,
                int64_t N, int64_t row_stride, int64_t fine_stride, float2* __restrict__ zones, float2* __restrict__ fine) {
    const int row = blockIdx.y % (P + 1), sym = blockIdx.y / (P + 1);
    const float* __restrict__ src = row == 0 ? price + (int64_t)sym * ld_price : rsi + ((int64_t)sym * P + row - 1) * ld_rsi;
    float2* __restrict__ dst = zones + ((int64_t)sym * (P + 1) + row) * row_stride;
    float2* __restrict__ fdst = fine + ((int64_t)sym * (P + 1) + row) * fine_stride;
    const int lane = threadIdx.x & 31;
    // (fine_stride covers whole 128-bar tiles and is >= 8 * row_stride - 8: one pass writes both)
    for (int64_t blk = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5); blk * (LS_ZONE / 4) < fine_stride || blk < row_stride;
         blk += (int64_t)gridDim.x * 8) {
        const int64_t t = blk * LS_ZONE + lane;
        const float v = t < N ? __ldg(src + t) : __int_as_float(0x7fc00000);
        float lo = v, hi = v;
#pragma unroll
        for (int m = 1; m < 4; m <<= 1) {
            lo = fminf(lo, __shfl_xor_sync(FULL, lo, m));
            hi = fmaxf(hi, __shfl_xor_sync(FULL, hi, m));
        }
        if ((lane & 3) == 0 && blk * (LS_ZONE / 4) + (lane >> 2) < fine_stride) fdst[blk * (LS_ZONE / 4) + (lane >> 2)] = make_float2(lo, hi);
#pragma unroll
        for (int m = 4; m < 32; m <<= 1) {
            lo = fminf(lo, __shfl_xor_sync(FULL, lo, m));
            hi = fmaxf(hi, __shfl_xor_sync(FULL, hi, m));
        }
        if (lane == 0 && blk < row_stride) dst[blk] = make_float2(lo, hi);
    }
}

struct LaneScanArgs {
    const float* price; int64_t ld_price;
    const float* rsi; int64_t ld_rsi;
    const float2* zones; int64_t n_zone_blocks;   // zone map (coarse part; n_zone_blocks = its row stride) or NULL
    const float2* fine; int64_t n_fine;           // 4-bar ranges and their row stride
    int P, S; int64_t N;
    const b200bt_individual* indiv; const int32_t* slots; int n_slots; int pop; int K; int warm;
    SegTables T;
    unsigned* work;      // work-item counter of the persistent scan (zero at launch)
    int* stalls;         // [0] tiles that did not arrive in time (their items go to the exact fallback), [1..8] the first one's details
    long long wait_cycles;   // bound of a tile wait in SM clocks (LS_WAIT_CYCLES; b200bt_sweep_scan_wait_cycles overrides, for tests)
};

// device-side tables the shared kernels expect: uniform K chunks per individual.  Work items are listed in dispatch
// order (`order`: individuals by predicted cost, a lane's chunks adjacent), so that the 32 chunks a warp of the
// thread-per-chunk metrics kernels folds hold similar numbers of records; segments stay indexed by individual.
__global__ void lane_tables_kernel(int pop, int K, const int32_t* __restrict__ order, b200bt_chunk_item* __restrict__ items,
                                   int32_t* __restrict__ seg_base, int32_t* __restrict__ n_chunks) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= pop * K) return;
    const int k = i / K, c = i - k * K;
    const int ind = order ? order[k] : k;
    b200bt_chunk_item it;
    it.individual = ind; it.chunk = c; it.n_chunks = K; it.segment = ind * K + c;
    items[i] = it;
    if (c == 0) { seg_base[ind] = ind * K; n_chunks[ind] = K; }
}

#ifndef B200BT_LS_MIN_BLOCKS
#define B200BT_LS_MIN_BLOCKS 3      // 85 registers: at 4 CTAs/SM (64) the scan loop spilled 18 words and ran 3 % slower
#endif
#ifndef B200BT_LS_STAGES
#define B200BT_LS_STAGES 2
#endif
#ifndef B200BT_LS_UNROLL
#define B200BT_LS_UNROLL 2
#endif
constexpr int LS_STAGES = B200BT_LS_STAGES;   // tiles in flight per warp (ring depth)
constexpr int LS_UNROLL = B200BT_LS_UNROLL;   // 4-bar groups per iteration of the scan loop
constexpr int LS_WARPS = LS_THREADS / 32;
constexpr int LS_RSI_ROWS = 2;                // distinct RSI rows the 32 machines of a warp may read (host packing)
constexpr int LS_ROWS = 1 + LS_RSI_ROWS;      // staged rows per warp: price + its RSI rows

static_assert(LS_ZONE == ZONE_BLOCK && LS_T == ZONE_TILE, "zone map layout (common.cuh) follows the scan's tile");

// Tile movement.  The 32 machines of a warp read the price row and (the host packs them so) at most LS_RSI_ROWS RSI rows.
// Every WARP owns a private ring of LS_STAGES shared-memory stages, each holding one 128-bar tile of those rows plus the
// tile's zone ranges; a stage is filled by bulk async copies (cp.async.bulk, one per row, issued by LS_ROWS lanes,
// completion counted on the stage's mbarrier) LS_STAGES - 1 tiles ahead of the scan and refilled by the warp itself the
// moment it has scanned it.  No warp ever waits for another one -- ncu on the round-1 form (one tile of all P + 1 rows per
// CTA, two CTA barriers per tile) showed a third of the warp time parked at those barriers behind the CTA's busiest warp
// and 18 % of the instructions computing cp.async addresses -- and the bytes moved per machine stay what they were,
// because a CTA-wide tile staged P + 1 rows for 256 machines and a warp stages 3 for 32.
// One work item: the 32 machines of warp-slot `wslot` (thread slots wslot * 32 ...) on symbol `sym`, chunk `c`.
constexpr long long LS_WAIT_CYCLES = 40ll * 1000 * 1000;     // ~20 ms at 1.9 GHz; a tile normally lands within microseconds

// the 32 machines of (warp-slot, symbol, chunk) are not scanned: their chunk is marked as having lost its events, which sends
// the chunk to the repair pass or the lane to the exact fallback
__device__ __forceinline__ void lane_scan_give_up(const LaneScanArgs& A, const int wslot, const int sym, const int c) {
    const int k = wslot * 32 + (int)(threadIdx.x & 31);
    const int slot = k < A.n_slots ? (A.slots ? A.slots[k] : (k < A.pop ? k : -1)) : -1;
    if (slot < 0) return;
    mark_lost(A.T, sym * (A.pop * A.K) + slot * A.K + c);
}

// -> false: a tile of this item did not arrive (see the wait below); the warp must not take another item
template <bool ZONES>
__device__ __forceinline__ bool lane_scan_item(const LaneScanArgs& A, const bool vec16, const int wslot, const int sym, const int c,
                                               float* const wtile, float2* const wzone, unsigned long long* const full,
                                               float (*ls_mul)[LS_THREADS], const void* (*ls_src_w)[3], int& ring_stage, unsigned& ring_parity) {
    constexpr int ZB = LS_T / LS_ZONE;                  // zone blocks per tile
    constexpr int FG = LS_T / 4;                        // 4-bar groups per tile
    constexpr int ZR = ZB + FG;                         // float2 per staged row: coarse ranges, then fine ranges
    const int lane = threadIdx.x & 31;
    const int k = wslot * 32 + lane;
    const int slot = k < A.n_slots ? (A.slots ? A.slots[k] : (k < A.pop ? k : -1)) : -1;
    const bool active = slot >= 0;
    const int ind = active ? slot : 0;
    const b200bt_individual iv = A.indiv[ind];
    // the screening multipliers are needed on events only: shared memory, [multiplier][thread] (conflict-free),
    // side-major so that the side selects an address instead of a value: long hi_c lo_c hi_d lo_d, short ...
    const float os_f = iv.rsi_lo, ob_f = iv.rsi_hi;
    {
        ScanConst sc;
        init_scan_const(sc, iv);
        float* m = &ls_mul[0][threadIdx.x];
        m[0 * LS_THREADS] = sc.hiL_c; m[1 * LS_THREADS] = sc.loL_c; m[2 * LS_THREADS] = sc.hiL_d; m[3 * LS_THREADS] = sc.loL_d;
        m[4 * LS_THREADS] = sc.hiS_c; m[5 * LS_THREADS] = sc.loS_c; m[6 * LS_THREADS] = sc.hiS_d; m[7 * LS_THREADS] = sc.loS_d;
    }
    __syncwarp();
    // The ring's barriers are initialised ONCE per warp (lane_scan_kernel) and their phases roll on from item to item: every
    // copy of the previous item has landed and been waited for, so the ring continues at (ring_stage, ring_parity).
    // (Invalidating and re-initialising them at every item lost a tile about once in 10^4 launches: DESIGN.md §3.1.)

    const int n = (int)A.N;
    const int T0 = (int)chunk_begin(A.N, c, A.K);       // first recorded bar (multiple of SW_GROUP, hence of LS_T)
    const int T1 = (int)chunk_begin(A.N, c + 1, A.K);   // end (exclusive)
    int s0 = (c == 0) ? 0 : T0 - A.warm;
    if (s0 < 0) s0 = 0;
    s0 &= ~(LS_T - 1);
    const int tl_begin = s0 / LS_T, n_tiles = (T1 + LS_T - 1) / LS_T - tl_begin;
    const int seg = sym * (A.pop * A.K) + ind * A.K + c;

    // the warp's distinct RSI rows: staged row 1 + j holds the j-th of them (in lane order of first use)
    const unsigned amask = __ballot_sync(FULL, active);
    if (amask == 0u) return true;                       // an empty warp (padding of the last CTA)
    const unsigned peers = __match_any_sync(FULL, active ? iv.rsi_row : -1 - lane);
    const int leader = __ffs(peers) - 1;
    const unsigned heads = __ballot_sync(FULL, active && lane == leader);
    const int n_rsi = __popc(heads);
    const int my_row = 1 + __popc(heads & ((1u << leader) - 1u));       // staged row this machine reads
    if (n_rsi > LS_RSI_ROWS) {
        // not packed for this schedule: the lanes are flagged and re-run by the caller's exact fallback (fused kernel)
        if (active) mark_lost(A.T, seg);
        return true;
    }
    // lane L <= n_rsi issues the copies of staged row L (0 = price)
    const unsigned src_lane = __fns(heads, 0, lane);                    // lane of the (lane)-th head (1-based), or ~0u
    const int row_of_lane = __shfl_sync(FULL, iv.rsi_row, src_lane < 32u ? (int)src_lane : 0);
    const bool issuer = lane <= n_rsi;
    const int zrow = (lane == 0 || !issuer) ? 0 : 1 + row_of_lane;      // row of the zone map (0 = price)
    // source rows of the warp's staged rows: a small table in shared memory (read by the issuing lanes only: three
    // 64-bit pointers per thread would not fit the register budget of the scan loop)
    if (issuer) {
        ls_src_w[lane][0] = (lane == 0) ? A.price + (int64_t)sym * A.ld_price : A.rsi + ((int64_t)sym * A.P + row_of_lane) * A.ld_rsi;
        ls_src_w[lane][1] = ZONES ? A.zones + ((int64_t)sym * (A.P + 1) + zrow) * A.n_zone_blocks : nullptr;   // (n_zone_blocks = row stride)
        ls_src_w[lane][2] = ZONES ? A.fine + ((int64_t)sym * (A.P + 1) + zrow) * A.n_fine : nullptr;
    }
    __syncwarp();
    const unsigned stage_bytes = (unsigned)(1 + n_rsi) * (LS_T * 4 + (ZONES ? ZR * 8 : 0));

    // fill stage `stage` of this warp's ring with tile `tl`
    auto issue = [&](int tl, int stage) {
        float* dst0 = wtile + (size_t)stage * LS_ROWS * LS_STRIDE;
        float2* zdst = wzone + (size_t)stage * LS_ROWS * ZR;
        const int t0 = tl * LS_T;
        if (vec16 && t0 + LS_T <= n) {
            if (lane == 0) mbar_arrive_expect_tx(&full[stage], stage_bytes);
            __syncwarp();
            if (issuer) {
                fence_proxy_async();      // the warp's reads of the stage (generic proxy) are ordered before the async writes
                bulk_g2s(dst0 + lane * LS_STRIDE, static_cast<const float*>(ls_src_w[lane][0]) + t0, LS_T * 4, &full[stage]);
                if (ZONES) {
                    bulk_g2s(zdst + lane * ZR, static_cast<const float2*>(ls_src_w[lane][1]) + (int64_t)tl * ZB, ZB * 8, &full[stage]);
                    bulk_g2s(zdst + lane * ZR + ZB, static_cast<const float2*>(ls_src_w[lane][2]) + (int64_t)tl * FG, FG * 8, &full[stage]);
                }
            }
        } else {
            const float qnan = __int_as_float(0x7fc00000);   // unaligned input or the ragged last tile: plain copies
            for (int r = 0; r <= n_rsi; ++r) {
                const float* src = static_cast<const float*>(ls_src_w[r][0]);
                for (int col = lane; col < LS_T; col += 32) dst0[r * LS_STRIDE + col] = (t0 + col < n) ? __ldg(src + t0 + col) : qnan;
                if (ZONES) {
                    const float2* zs = static_cast<const float2*>(ls_src_w[r][1]);
                    const float2* fs = static_cast<const float2*>(ls_src_w[r][2]);
                    if (lane < ZB) {
                        const int64_t zblk = (int64_t)tl * ZB + lane;
                        zdst[r * ZR + lane] = (zblk * LS_ZONE < n) ? zs[zblk] : make_float2(qnan, qnan);
                    }
                    zdst[r * ZR + ZB + lane] = fs[(int64_t)tl * FG + lane];        // (FG == 32; rows are padded to whole tiles)
                }
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(&full[stage]);     // (release: the stores above are visible after the wait)
        }
    };
    for (int it = 0; it < LS_STAGES && it < n_tiles; ++it) issue(tl_begin + it, (ring_stage + it) % LS_STAGES);

    // machine state (per thread)
    int pos = 0, entry_bar = 0;
    float e_px = 0.f, rlo = iv.rsi_lo, rhi = iv.rsi_hi, plo = -INFINITY, phi = INFINITY;
    // event sink: this thread's chunk owns a chain of pool blocks
    int cur_block = -1, fill = CK_BLOCK;
    unsigned count = 0;
    bool rec = false, dead = false;
    uint2* wptr = A.T.pool;
    auto record = [&](unsigned word, float p) {
        if (fill == CK_BLOCK && !dead) {
            const int b = pool_append(A.T, seg, cur_block);
            if (b < 0) dead = true;
            else { cur_block = b; fill = 0; wptr = A.T.pool + (int64_t)b * CK_BLOCK; }
        }
        if (!dead) { *wptr++ = make_uint2(word, __float_as_uint(p)); ++fill; }
        ++count;
    };

    // one bar of the state machine; same decisions as scan_window (sweep_dev.cuh).  Written as straight-line
    // selects: the threads of a warp that fire on the same bar (entries and exits alike) share one pass.
    auto step = [&](float p, float r, int t) {
        const bool rsi_hit = (r < rlo) | (r > rhi);
        if (!(rsi_hit | (p <= plo) | (p >= phi))) return;
        const bool flat = pos == 0, lng_open = pos > 0;
        bool ev = true;
        if (!flat && !rsi_hit) {
            // price trigger: definite outside the fp32 screening band, else the reference's float64 expression
            const float* m = &ls_mul[lng_open ? 2 : 6][threadIdx.x];
            const float hd = e_px * m[0], ld = e_px * m[LS_THREADS];
            if (!((p >= hd) || (p <= ld))) {
                const double ed = (double)e_px, pd = (double)p;
                const double q = lng_open ? __ddiv_rn(__dsub_rn(pd, ed), ed) : __ddiv_rn(__dsub_rn(ed, pd), ed);
                ev = (q >= A.indiv[ind].take_profit) || (q <= -A.indiv[ind].stop_loss);
            }
        }
        if (!ev) return;
        const bool lng = r < os_f;                        // entry side: long has priority (:784, :799)
        const unsigned word = flat ? ((unsigned)t | (lng ? 0u : B200BT_EVENT_SELL))
                                   : ((unsigned)t | B200BT_EVENT_EXIT | (lng_open ? B200BT_EVENT_SELL : 0u));
        pos = flat ? (lng ? 1 : -1) : 0;
        rlo = (flat && lng) ? -INFINITY : os_f;
        rhi = (flat && !lng) ? INFINITY : ob_f;
        const float* mc = &ls_mul[lng ? 0 : 4][threadIdx.x];
        phi = flat ? p * mc[0] : INFINITY;
        plo = flat ? p * mc[LS_THREADS] : -INFINITY;
        e_px = flat ? p : e_px;
        entry_bar = flat ? t : entry_bar;
        if (rec) record(word, p);
    };

    int stage = ring_stage;
    unsigned parity = ring_parity;
    for (int it = 0; it < n_tiles; ++it) {
        // A copy that never completes must not hang the GPU: the wait is bounded.  On a timeout the item is given up -- its
        // chunks are marked as having lost their events, so the repair pass re-scans them (or the lane takes the exact
        // fallback) -- and the warp never touches its ring again (copies may still be in flight into it): it goes on taking
        // items only to give them up as well (lane_scan_kernel), while the other warps scan theirs.
        // (wait_cycles < 0 is the test hook: the warp gives up at its (-wait_cycles)-th tile as if the tile had not arrived)
        const bool lost = A.wait_cycles < 0 ? (it + 1 == (int)-A.wait_cycles || !mbar_wait_bounded(&full[stage], parity, LS_WAIT_CYCLES))
                                            : !mbar_wait_bounded(&full[stage], parity, A.wait_cycles);
        if (__any_sync(FULL, lost)) {
            lane_scan_give_up(A, wslot, sym, c);
            if (lane == 0 && A.stalls && atomicAdd(A.stalls, 1) == 0) {
                A.stalls[1] = (int)blockIdx.x; A.stalls[2] = (int)(threadIdx.x >> 5); A.stalls[3] = wslot * 65536 + sym * 256 + c;
                A.stalls[4] = it; A.stalls[5] = n_tiles; A.stalls[6] = stage * 2 + (int)parity; A.stalls[7] = tl_begin; A.stalls[8] = n_rsi;
            }
            return false;
        }
        const int t0 = (tl_begin + it) * LS_T;
        if (active) {
            if (t0 == T0) { A.T.seg_in[seg] = seg_state(pos, entry_bar); rec = true; }
            const float4* __restrict__ pp = reinterpret_cast<const float4*>(wtile + (size_t)stage * LS_ROWS * LS_STRIDE);
            const float4* __restrict__ rr = reinterpret_cast<const float4*>(wtile + ((size_t)stage * LS_ROWS + my_row) * LS_STRIDE);
            const float2* __restrict__ zp = wzone + (size_t)stage * LS_ROWS * ZR;
            const float2* __restrict__ zr = zp + my_row * ZR;
#pragma unroll 1
            for (int zb = 0; zb < ZB; ++zb) {
                if (ZONES) {
                    // nothing can fire in a block whose (min, max) stay inside the machine's thresholds; the skip is
                    // taken when NO machine of the warp can fire (a warp-uniform branch: a machine that could skip alone
                    // would wait for its neighbours anyway, and the divergent form costs the re-convergence on top)
                    const float2 rz = zr[zb], pz = zp[zb];
                    if (!__any_sync(amask, (rz.x < rlo) | (rz.y > rhi) | (pz.x <= plo) | (pz.y >= phi))) continue;
                }
#pragma unroll LS_UNROLL
                for (int g = zb * (LS_ZONE / 4); g < (zb + 1) * (LS_ZONE / 4); ++g) {
                    bool hit;
                    if (ZONES) {
                        // the group's precomputed range decides whether any of its four bars can fire (tested against the
                        // machine's CURRENT thresholds: they move whenever it fires)
                        const float2 rm = zr[ZB + g], pm = zp[ZB + g];
                        hit = (rm.x < rlo) | (rm.y > rhi) | (pm.x <= plo) | (pm.y >= phi);
                        if (!hit) continue;
                    }
                    const float4 p = pp[g], r = rr[g];
                    if (!ZONES) {
                        // any bar of the four beyond a threshold?  (fminf / fmaxf drop NaNs, as the per-bar compares do)
                        const float r_min = fminf(fminf(r.x, r.y), fminf(r.z, r.w)), r_max = fmaxf(fmaxf(r.x, r.y), fmaxf(r.z, r.w));
                        const float p_min = fminf(fminf(p.x, p.y), fminf(p.z, p.w)), p_max = fmaxf(fmaxf(p.x, p.y), fmaxf(p.z, p.w));
                        hit = (r_min < rlo) | (r_max > rhi) | (p_min <= plo) | (p_max >= phi);
                    }
                    if (hit) {
                        const int t = t0 + g * 4;
                        step(p.x, r.x, t);
                        step(p.y, r.y, t + 1);
                        step(p.z, r.z, t + 2);
                        step(p.w, r.w, t + 3);
                    }
                }
            }
        }
        __syncwarp();      // every machine of the warp is done with the stage: refill it with the tile LS_STAGES ahead
        if (it + LS_STAGES < n_tiles) issue(tl_begin + it + LS_STAGES, stage);
        if (++stage == LS_STAGES) { stage = 0; parity ^= 1u; }
    }
    ring_stage = stage;
    ring_parity = parity;
    if (!active) return true;
    A.T.seg_out[seg] = seg_state(pos, entry_bar);
    if (c == A.K - 1 && pos != 0)   // force-close at the last bar (:849-876; the last chunk always records: T0 < N)
        record((unsigned)(n - 1) | B200BT_EVENT_EXIT | (pos > 0 ? B200BT_EVENT_SELL : 0u), __ldg(A.price + (int64_t)sym * A.ld_price + (n - 1)));
    A.T.seg_count[seg] = dead ? SEG_LOST : count;
    return true;
}

// Persistent form: the grid is one resident set of CTAs; every WARP takes work items -- (warp-slot, chunk, symbol), the
// most expensive warp-slots first -- from a global counter until none is left, so all warp slots of the GPU stay busy until
// the queue is empty and the last items to run are the cheapest ones (a static grid left the busiest CTAs running alone
// at the end while the rest of their SM sat idle).
template <bool ZONES>
__global__ void __launch_bounds__(LS_THREADS, B200BT_LS_MIN_BLOCKS)
lane_scan_kernel(const LaneScanArgs A, const bool vec16) {   // by value, not __grid_constant__ (see sweep.cu)
    // [LS_WARPS][LS_STAGES][LS_ROWS][LS_STRIDE] floats, then (ZONES) per warp and stage [LS_ROWS][LS_T / 32 + LS_T / 4] float2
    extern __shared__ __align__(16) float ls_tile[];
    __shared__ __align__(8) unsigned long long ls_full[LS_WARPS][LS_STAGES];   // "tile landed" (1 arrival + the copies' bytes)
    __shared__ float ls_mul[8][LS_THREADS];
    __shared__ const void* ls_src[LS_WARPS][LS_ROWS][3];
    constexpr int ZR = LS_T / LS_ZONE + LS_T / 4;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    float* const wtile = ls_tile + (size_t)warp * LS_STAGES * LS_ROWS * LS_STRIDE;
    float2* const wzone = reinterpret_cast<float2*>(ls_tile + (size_t)LS_WARPS * LS_STAGES * LS_ROWS * LS_STRIDE) + (size_t)warp * LS_STAGES * LS_ROWS * ZR;
    if (lane == 0) {
#pragma unroll
        for (int s = 0; s < LS_STAGES; ++s) mbar_init(&ls_full[warp][s], 1);
        mbar_fence_init();
        fence_proxy_async();
    }
    __syncwarp();
    int ring_stage = 0;            // the warp's position in its tile ring, carried from item to item
    unsigned ring_parity = 0;
    bool retired = false;          // a tile of this warp's ring did not arrive: the ring is not used again
    const int per_slot = A.K * A.S;
    const int n_items = (A.n_slots / 32) * per_slot;
    for (;;) {
        int item = 0;
        if (lane == 0) item = (int)atomicAdd(A.work, 1u);
        item = __shfl_sync(FULL, item, 0);
        if (item >= n_items) break;
        const int wslot = item / per_slot, rest = item - wslot * per_slot;
        const int c = rest / A.S, sym = rest - c * A.S;
        if (retired) { lane_scan_give_up(A, wslot, sym, c); continue; }     // (every item is either scanned or marked)
        retired = !lane_scan_item<ZONES>(A, vec16, wslot, sym, c, wtile, wzone, ls_full[warp], ls_mul, ls_src[warp], ring_stage, ring_parity);
        __syncwarp();
    }
}

// ---- metrics, chunk-parallel -------------------------------------------------------------------------
// The trade-record metrics are a fold over the lane's events in time order, but every piece of it is
// either a sum / max / xor (associative) or depends on the past only through three scalars: the equity
// and running equity peak at the chunk's start, and the index of the chunk's first record.  So:
//   chunk_sums_kernel    warp per (chunk, symbol): sum of record pnls and the largest prefix sum.
//   chunk_partial_kernel warp per (chunk, symbol): exclusive scan of those over the lane's earlier chunks
//                        -> starting equity / peak / record index, then the ordinary batch arithmetic
//                        (batch_core) over the chunk's own events into a ChunkPartial.
//   lane_combine_kernel  thread per (individual, symbol): verifies the boundaries, merges the partials
//                        (calendar days that straddle a chunk boundary are re-joined) and finalises.
struct ChunkPartial {
    double tot_profit, tot_loss, largest_p, largest_l, maxdd, first_sum, pivot, s1, s2, day_sum;
    long long sum_dur;
    unsigned long long hash;
    unsigned n_win, n_loss, n_days, count;
    int first_done, first_day, day_cur;
    unsigned n_neg;
    double npivot, ns1, ns2, pad;     // the chunk's finished negative days (DayAcc)
};
static_assert(sizeof(ChunkPartial) == 160, "ChunkPartial layout");

__device__ __forceinline__ unsigned seg_events(unsigned count) { return count == SEG_LOST ? 0u : count; }

// One step of a chunk's records: records 2l and 2l+1 of the step in lane l (event word w, price pf), and the record
// before 2l (lane l-1's second one; lane 0: the previous step's last record, or the entry the chunk starts in).
struct RecordPair {
    int cnt;                   // records in the step (1..64)
    int last;                  // lane holding the step's last record
    bool a0, a1;               // records 2l, 2l+1 exist
    unsigned w0, w1, w_prev;
    float pf0, pf1, p_prev;
};

// Cursor over the `count` records of segment `seg` in time order, 64 per step, two consecutive ones per lane (one 16-byte
// load: half the shuffles per record):  for (RecordPair r; next_pair(R, r); advance(R, r)) { ... }.  A chain that leaves
// the pool (a segment being re-scanned on the side stream) ends the walk.
struct RecordReader {
    const uint2* pool; const int* next; int pool_blocks;
    unsigned left; int b, off;
    unsigned w_carry; float p_carry;     // the record before the next step's first one
};

__device__ __forceinline__ RecordReader record_reader(const uint2* __restrict__ pool, const int* __restrict__ next, int pool_blocks,
                                                      const int* __restrict__ seg_first, int seg, unsigned count, int2 in,
                                                      const float* __restrict__ pr) {
    RecordReader R{pool, next, pool_blocks, count, count ? seg_first[seg] : -1, 0, 0u, 0.f};
    if (in.x != 0) {      // the entry record the chunk's first exit is priced against
        R.w_carry = (unsigned)in.y | (in.x < 0 ? B200BT_EVENT_SELL : 0u);
        R.p_carry = __ldg(pr + in.y);
    }
    if ((unsigned)R.b >= (unsigned)pool_blocks) R.left = 0;
    return R;
}

__device__ __forceinline__ bool next_pair(const RecordReader& R, RecordPair& r) {
    if (!R.left) return false;
    const int lane = threadIdx.x & 31;
    r.cnt = (int)min(64u, R.left);
    r.last = (r.cnt - 1) >> 1;
    r.a0 = 2 * lane < r.cnt; r.a1 = 2 * lane + 1 < r.cnt;
    uint4 ev = make_uint4(0u, 0u, 0u, 0u);
    if (r.a0) ev = *reinterpret_cast<const uint4*>(R.pool + (int64_t)R.b * CK_BLOCK + R.off + 2 * lane);   // (slot 2l+1 may be unused: in-block)
    r.w0 = ev.x; r.w1 = ev.z;
    r.pf0 = __uint_as_float(ev.y); r.pf1 = __uint_as_float(ev.w);
    r.p_prev = __shfl_up_sync(FULL, r.pf1, 1);
    r.w_prev = __shfl_up_sync(FULL, r.w1, 1);
    if (lane == 0) { r.p_prev = R.p_carry; r.w_prev = R.w_carry; }
    return true;
}

__device__ __forceinline__ void advance(RecordReader& R, const RecordPair& r) {
    R.w_carry = __shfl_sync(FULL, (r.cnt & 1) ? r.w0 : r.w1, r.last);
    R.p_carry = __shfl_sync(FULL, (r.cnt & 1) ? r.pf0 : r.pf1, r.last);
    R.left -= r.cnt;
    R.off += 64;
    if (R.off == CK_BLOCK && R.left) {
        R.b = R.next[R.b]; R.off = 0;
        if ((unsigned)R.b >= (unsigned)R.pool_blocks) R.left = 0;
    }
}

__global__ void __launch_bounds__(128)
chunk_sums_kernel(const float* __restrict__ price, int64_t ld_price, const b200bt_individual* __restrict__ indiv,
                  const b200bt_chunk_item* __restrict__ items, int n_items, int S, int n_seg,
                  const uint2* __restrict__ pool, const int* __restrict__ next, const int* __restrict__ seg_first,
                  const unsigned* __restrict__ seg_count, const int2* __restrict__ seg_in,
                  double* __restrict__ seg_sum, double* __restrict__ seg_max, const int* __restrict__ n_items_dev,
                  int pool_blocks) {
    const int lane = threadIdx.x & 31;
    const int sym = (int)(blockIdx.x % (unsigned)S);
    const int it = (int)(blockIdx.x / (unsigned)S) * 4 + (threadIdx.x >> 5);
    if (it >= (n_items_dev ? *n_items_dev : n_items)) return;
    const b200bt_chunk_item item = items[it];
    const int seg = sym * n_seg + item.segment;
    const double size = indiv[item.individual].position_size;
    const double fee1 = __dmul_rn(size, 0.001), fee2 = __dmul_rn(size, 0.002);
    double run = 0.0, best = -INFINITY;
    RecordReader R = record_reader(pool, next, pool_blocks, seg_first, seg, seg_events(seg_count[seg]), seg_in[seg],
                                   price + (int64_t)sym * ld_price);
    for (RecordPair r; next_pair(R, r); advance(R, r)) {
        int dur;
        const double pnl0 = record_pnl(r.a0, r.w0, r.pf0, r.w_prev, r.p_prev, size, fee1, fee2, dur);
        const double pnl1 = record_pnl(r.a1, r.w1, r.pf1, r.w0, r.pf0, size, fee1, fee2, dur);
        const double s2 = pnl0 + pnl1;
        double cs = s2;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const double up = shfl_up_d(cs, d);
            if (lane >= d) cs += up;
        }
        const double after0 = run + (cs - s2) + pnl0, after1 = run + cs;
        best = fmax(best, warp_max_d(fmax(r.a0 ? after0 : -INFINITY, r.a1 ? after1 : -INFINITY)));
        run += shfl_d(cs, 31);
    }
    if (lane == 0) { seg_sum[seg] = run; seg_max[seg] = best; }
}

#ifndef B200BT_M2_MIN_BLOCKS
#define B200BT_M2_MIN_BLOCKS 8
#endif
__global__ void __launch_bounds__(128, B200BT_M2_MIN_BLOCKS)
chunk_partial_kernel(const float* __restrict__ price, int64_t ld_price, const b200bt_individual* __restrict__ indiv,
                     const b200bt_chunk_item* __restrict__ items, int n_items, int S, int n_seg,
                     const uint2* __restrict__ pool, const int* __restrict__ next, const int* __restrict__ seg_first,
                     const unsigned* __restrict__ seg_count, const int2* __restrict__ seg_in,
                     const double* __restrict__ seg_sum, const double* __restrict__ seg_max,
                     const b200bt_sweep_config cfg, uint32_t* __restrict__ events, int64_t ev_cap,
                     ChunkPartial* __restrict__ partial, const int* __restrict__ n_items_dev, int pool_blocks) {
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const int sym = (int)(blockIdx.x % (unsigned)S);
    const int it = (int)(blockIdx.x / (unsigned)S) * 4 + wid;
    if (it >= (n_items_dev ? *n_items_dev : n_items)) return;
    const b200bt_chunk_item item = items[it];
    const int seg = sym * n_seg + item.segment;
    const int base = seg - item.chunk;
    const b200bt_individual iv = indiv[item.individual];

    // state at the chunk's start: equity, running peak, record index -- exclusive scan over earlier chunks
    double e0 = cfg.initial_capital, p0 = cfg.initial_capital;
    unsigned first_index = 0;
    for (int c0 = 0; c0 < item.chunk; c0 += 32) {
        const int c = c0 + lane;
        const bool in = c < item.chunk;
        const double s = in ? seg_sum[base + c] : 0.0;
        const double mx = in ? seg_max[base + c] : -INFINITY;
        const unsigned n = in ? seg_events(seg_count[base + c]) : 0u;
        double incl = s;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const double up = shfl_up_d(incl, d);
            if (lane >= d) incl += up;
        }
        const double start = e0 + (incl - s);            // equity at the start of chunk c
        p0 = fmax(p0, warp_max_d(start + mx));
        e0 += shfl_d(incl, 31);
        first_index += __reduce_add_sync(FULL, n);
    }

    // Order-dependent state (equity, peak, drawdown, calendar day) is warp-uniform and lives in registers; what
    // is a plain sum / max / xor over the records is accumulated PER LANE and reduced once at the end of the chunk.
    const double size = iv.position_size;
    const double fee1 = __dmul_rn(size, 0.001), fee2 = __dmul_rn(size, 0.002);
    double equity = e0, peak = p0, maxdd = 0.0;
    DayAcc da{0.0, 0.0, 0.0, 0u, 0};
    int day_valid = 0, day_cur = 0, first_done = 0, first_id = 0;
    double day_sum = 0.0, first_sum = 0.0;
    unsigned index = first_index;
    double l_gain = 0.0, l_loss = 0.0, l_maxp = 0.0, l_minl = 0.0;
    unsigned l_win = 0, l_los = 0;
    long long l_dur = 0;
    unsigned long long l_hash = 0ull;
    uint32_t* const ev_out = events ? events + ((int64_t)item.individual * S + sym) * ev_cap : nullptr;
    const unsigned minute0 = (unsigned)cfg.minute0, bar_minutes = (unsigned)cfg.bar_minutes;
    const unsigned gap_bar = cfg.gap_bar > 0 ? (unsigned)cfg.gap_bar : 0xffffffffu, gap_minutes = (unsigned)cfg.gap_minutes;
    auto day_of = [&](unsigned w) {   // calendar day of a record (a glued series jumps gap_minutes at gap_bar)
        const unsigned bar = w & 0x3fffffffu;
        return (int)((minute0 + bar * bar_minutes + (bar >= gap_bar ? gap_minutes : 0u)) / 1440u);
    };
    auto finish_day = [&](int id, double x) {     // the chunk's first day may continue the previous chunk's last one
        if (!first_done) { first_done = 1; first_id = id; first_sum = x; }
        else day_complete(da, x);
    };

    const unsigned count = seg_events(seg_count[seg]);
    RecordReader R = record_reader(pool, next, pool_blocks, seg_first, seg, count, seg_in[seg], price + (int64_t)sym * ld_price);
    for (RecordPair r; next_pair(R, r); advance(R, r)) {
        const int cnt = r.cnt, last_lane = r.last;
        const bool a0 = r.a0, a1 = r.a1;
        const unsigned w0 = r.w0, w1 = r.w1;
        const float pf0 = r.pf0, pf1 = r.pf1;
        int dur0, dur1;
        const double pnl0 = record_pnl(a0, w0, pf0, r.w_prev, r.p_prev, size, fee1, fee2, dur0);
        const double pnl1 = record_pnl(a1, w1, pf1, w0, pf0, size, fee1, fee2, dur1);
        if (pnl0 > 0.0) { l_gain += pnl0; ++l_win; l_maxp = fmax(l_maxp, pnl0); }
        else if (pnl0 < 0.0) { l_loss += pnl0; ++l_los; l_minl = fmin(l_minl, pnl0); }
        if (pnl1 > 0.0) { l_gain += pnl1; ++l_win; l_maxp = fmax(l_maxp, pnl1); }
        else if (pnl1 < 0.0) { l_loss += pnl1; ++l_los; l_minl = fmin(l_minl, pnl1); }
        l_dur += dur0 + dur1;
        const unsigned i0 = index + 2 * lane;
        if (a0) {
            l_hash ^= event_hash(i0, w0);
            if (ev_out && (int64_t)i0 < ev_cap) ev_out[i0] = w0;
        }
        if (a1) {
            l_hash ^= event_hash(i0 + 1, w1);
            if (ev_out && (int64_t)i0 + 1 < ev_cap) ev_out[i0 + 1] = w1;
        }

        // equity curve: inclusive scan of the lane sums, running peak, drawdown (cf. batch_core, sweep_dev.cuh)
        const double s2 = pnl0 + pnl1;
        double cs = s2;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const double up = shfl_up_d(cs, d);
            if (lane >= d) cs += up;
        }
        const double eq0 = equity + (cs - s2) + pnl0, eq1 = equity + cs;
        const double m2 = fmax(a0 ? eq0 : -INFINITY, a1 ? eq1 : -INFINITY);
        double pk0 = peak, pk1 = peak;
        if (__any_sync(FULL, m2 > peak)) {
            double pk = m2;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                const double up = shfl_up_d(pk, d);
                if (lane >= d) pk = fmax(pk, up);
            }
            double before = shfl_up_d(pk, 1);          // peak over the records of the lanes in front
            before = fmax(lane == 0 ? peak : before, peak);
            pk0 = fmax(before, eq0);
            pk1 = fmax(pk0, eq1);
            peak = fmax(peak, shfl_d(pk, 31));
        }
        {
            const double gap0 = __dsub_rn(pk0, eq0), gap1 = __dsub_rn(pk1, eq1);
            const double lim = maxdd * (1.0 - 1e-12);
            const bool c0 = a0 && gap0 > 0.0 && gap0 >= lim * pk0, c1 = a1 && gap1 > 0.0 && gap1 >= lim * pk1;
            if (__any_sync(FULL, c0 || c1))
                maxdd = fmax(maxdd, warp_max_d(fmax(c0 ? __ddiv_rn(gap0, pk0) : 0.0, c1 ? __ddiv_rn(gap1, pk1) : 0.0)));
        }
        const double batch_sum = shfl_d(cs, 31);
        equity += batch_sum;

        // calendar-day buckets
        const int d0 = a0 ? day_of(w0) : 0;
        const int d1 = a1 ? day_of(w1) : d0;
        const int first_day = __shfl_sync(FULL, d0, 0);
        const int last_day = __shfl_sync(FULL, d1, last_lane);
        if (first_day == last_day && (!day_valid || first_day == day_cur)) {
            day_sum = (day_valid ? day_sum : 0.0) + batch_sum;      // the whole step falls into the open day
        } else {
            // a record is a HEAD if it opens a day within the step; running day sum = segmented scan by heads.
            // As a function of the running sum it receives, a lane is either additive (no head) or constant.
            const bool merge_carry = day_valid && (first_day == day_cur);
            const int d_before = __shfl_up_sync(FULL, d1, 1);
            const bool head0 = a0 && (lane == 0 ? !merge_carry : d0 != d_before);
            const bool head1 = a1 && d1 != d0;
            double sg = head1 ? pnl1 : s2;
            bool flag = head0 || head1;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                const double up = shfl_up_d(sg, d);
                const int fup = __shfl_up_sync(FULL, (int)flag, d);
                if (lane >= d && !flag) { sg += up; flag = fup; }
            }
            // (the open day carried in is part of lane 0's chain when it continues)
            if (merge_carry && !flag) sg += day_sum;          // lanes whose chain reaches back to the step's start
            double carry_in = shfl_up_d(sg, 1);
            if (lane == 0) carry_in = merge_carry ? day_sum : 0.0;
            const double run0 = head0 ? pnl0 : carry_in + pnl0;     // running day sum after record 2l
            const double run1 = sg;                                  // ... after record 2l+1 (== run0 if inactive)
            // TAIL = last record of its day within the step, except the step's last record (its day stays open)
            const int d_after = __shfl_down_sync(FULL, d0, 1);
            const bool tail0 = a0 && (a1 ? head1 : false);
            const bool tail1 = a1 && lane < last_lane && d_after != d1;
            // (an unpaired last record 2l is the step's last record: its day stays open)
            unsigned t0m = __ballot_sync(FULL, tail0), t1m = __ballot_sync(FULL, tail1);
            if (day_valid && !merge_carry) finish_day(day_cur, day_sum);
            while (t0m | t1m) {
                const int j = __ffs(t0m | t1m) - 1;
                const unsigned bit = 1u << j;
                if (t0m & bit) finish_day(__shfl_sync(FULL, d0, j), shfl_d(run0, j));
                if (t1m & bit) finish_day(__shfl_sync(FULL, d1, j), shfl_d(run1, j));
                t0m &= ~bit; t1m &= ~bit;
            }
            day_sum = (cnt & 1) ? shfl_d(run0, last_lane) : shfl_d(run1, last_lane);
        }
        day_cur = last_day;
        day_valid = 1;

        index += cnt;
    }
    // per-lane accumulators -> chunk totals
    const double tot_profit = warp_sum_d(l_gain), tot_loss = warp_sum_d(l_loss);
    const double largest_p = warp_max_d(l_maxp), largest_l = warp_min_d(l_minl);
    const unsigned n_win = __reduce_add_sync(FULL, l_win), n_loss = __reduce_add_sync(FULL, l_los);
    long long sum_dur = l_dur;
    unsigned hlo = (unsigned)l_hash, hhi = (unsigned)(l_hash >> 32);
#pragma unroll
    for (int m = 16; m > 0; m >>= 1) sum_dur += __shfl_xor_sync(FULL, sum_dur, m);
    hlo = __reduce_xor_sync(FULL, hlo);
    hhi = __reduce_xor_sync(FULL, hhi);
    if (lane == 0) {
        ChunkPartial q;
        q.tot_profit = tot_profit; q.tot_loss = tot_loss; q.largest_p = largest_p; q.largest_l = largest_l;
        q.maxdd = maxdd; q.first_sum = first_sum; q.pivot = da.pivot; q.s1 = da.s1; q.s2 = da.s2; q.day_sum = day_sum;
        q.sum_dur = sum_dur; q.hash = ((unsigned long long)hhi << 32) | hlo;
        q.n_win = n_win; q.n_loss = n_loss; q.n_days = da.n_days; q.count = count;
        q.first_done = first_done; q.first_day = first_id; q.day_cur = day_cur;
        q.n_neg = da.n_neg; q.npivot = da.npivot; q.ns1 = da.ns1; q.ns2 = da.ns2; q.pad = 0.0;
        partial[seg] = q;
    }
}

// Work items (all chunks) of the individuals flagged in `redo`, for the recomputation after the overlapped repairs.
__global__ void fix_items_kernel(const b200bt_chunk_item* __restrict__ items, int n_items, const unsigned char* __restrict__ redo,
                                 b200bt_chunk_item* __restrict__ out, int* __restrict__ n_out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_items) return;
    const b200bt_chunk_item it = items[i];
    if (redo[it.individual]) out[atomicAdd(n_out, 1)] = it;
}

// Individuals with a lane the chunked evaluation could not settle (a boundary still inconsistent after the repair passes, a
// full event pool, a warp not packed for the thread-per-lane scan): listed on the device for the exact fallback.
__global__ void redo_list_kernel(int pop, int S, const unsigned char* __restrict__ invalid, int32_t* __restrict__ list,
                                 int* __restrict__ n_list, int* __restrict__ n_invalid_lanes) {
    const int ind = blockIdx.x * blockDim.x + threadIdx.x;
    if (ind >= pop) return;
    int bad = 0;
    for (int s = 0; s < S; ++s) bad += invalid[(int64_t)ind * S + s] ? 1 : 0;
    if (bad) {
        list[atomicAdd(n_list, 1)] = ind;
        atomicAdd(n_invalid_lanes, bad);
    }
}

__global__ void lane_combine_kernel(const b200bt_individual* __restrict__ indiv, int pop, int S,
                                    const int32_t* __restrict__ seg_base, const int32_t* __restrict__ n_chunks, int n_seg,
                                    const unsigned* __restrict__ seg_count, const int2* __restrict__ seg_in,
                                    const int2* __restrict__ seg_out, const ChunkPartial* __restrict__ partial,
                                    const b200bt_sweep_config cfg, b200bt_lane_stats* __restrict__ stats,
                                    unsigned char* __restrict__ invalid) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= (int64_t)pop * S) return;
    const int ind = (int)(t / S), sym = (int)(t % S);
    const int K = n_chunks[ind];
    const int base = sym * n_seg + seg_base[ind];
    bool ok = true;
    for (int c = 0; c < K; ++c) {
        const int2 a = seg_in[base + c];
        if (c == 0) ok = ok && (a.x == 0);
        else {
            const int2 z = seg_out[base + c - 1];
            ok = ok && (a.x == z.x) && (a.y == z.y);
        }
        ok = ok && (seg_count[base + c] != SEG_LOST);
    }
    invalid[t] = ok ? 0 : 1;
    if (!ok) return;
    WarpAcc a;
    init_acc(a, indiv[ind], cfg, nullptr);
    DayAcc da{0.0, 0.0, 0.0, 0u, 0};
    bool open = false;      // the lane's open (last, not yet finished) calendar day
    int open_day = 0;
    double open_sum = 0.0;
    for (int c = 0; c < K; ++c) {
        const ChunkPartial q = partial[base + c];
        if (q.count == 0) continue;
        a.n_events += q.count;
        a.n_win += q.n_win; a.n_loss += q.n_loss;
        a.tot_profit += q.tot_profit; a.tot_loss += q.tot_loss;
        a.largest_p = fmax(a.largest_p, q.largest_p); a.largest_l = fmin(a.largest_l, q.largest_l);
        a.maxdd = fmax(a.maxdd, q.maxdd);
        a.sum_dur += q.sum_dur;
        a.hash ^= q.hash;
        if (!q.first_done) {
            // the whole chunk lies in one calendar day, which stays open
            if (open && open_day == q.day_cur) open_sum += q.day_sum;
            else {
                if (open) day_complete(da, open_sum);
                open = true; open_day = q.day_cur; open_sum = q.day_sum;
            }
            continue;
        }
        double x = q.first_sum;
        if (open) {
            if (open_day == q.first_day) x += open_sum; else day_complete(da, open_sum);
        }
        day_complete(da, x);
        if (q.n_days) {
            // the chunk's own finished days, accumulated about its pivot: shift to the lane's pivot
            const double d = q.pivot - da.pivot, n = (double)q.n_days;
            da.s1 += q.s1 + n * d;
            da.s2 += q.s2 + 2.0 * d * q.s1 + n * d * d;
            da.n_days += q.n_days;
        }
        if (q.n_neg) {
            if (da.n_neg == 0) da.npivot = q.npivot;
            const double d = q.npivot - da.npivot, n = (double)q.n_neg;
            da.ns1 += q.ns1 + n * d;
            da.ns2 += q.ns2 + 2.0 * d * q.ns1 + n * d * d;
            da.n_neg += q.n_neg;
        }
        open = true; open_day = q.day_cur; open_sum = q.day_sum;
    }
    a.pivot = da.pivot; a.s1 = da.s1; a.s2 = da.s2; a.n_days = da.n_days; a.pivot_set = da.pivot_set;
    a.npivot = da.npivot; a.ns1 = da.ns1; a.ns2 = da.ns2; a.n_neg = da.n_neg;
    a.day_valid = open ? 1 : 0; a.day_sum = open_sum; a.day_cur = open_day;
    b200bt_lane_stats o;
    finalize_lane(a, cfg, o);
    stats[t] = o;
}

}  // namespace b200bt

using namespace b200bt;

namespace {

// Counters of one sweep, zeroed with the segment tables at entry.  The first four words are what the caller's
// overflow_host_or_null[0..3] receives.
struct SweepCounters {
    int overflow;              // [0] the event pool ran out of blocks
    int n_flagged;             // [1] (individual, symbol) lanes that went through the exact fallback
    unsigned alloc;            // [2] pool blocks handed out
    int scan_stalls[9];        // [3] tiles of lane_scan_kernel that did not arrive in time; [1..8] the first one's details
    unsigned repair_work[2];   // work counters of chunk_repair_kernel and lane_repair_kernel
    unsigned scan_work;        // work counter of lane_scan_kernel
    int n_fix, n_redo;         // items in fix_items, individuals in redo_list
};
static_assert(offsetof(SweepCounters, scan_stalls) == 3 * sizeof(int), "host flags: the first four words");

// Workspace of the time-chunked sweeps.  Every region starts 16-byte aligned (the base must be); the segment tables
// and the counters follow one another, so one memset clears them.
struct ChunkWorkspace {
    SegTables T;                           // pool, next [pool_blocks] (apart); seg_* [segs]; alloc, overflow -> ctr
    SweepCounters* ctr;
    ChunkPartial* partial;                 // [segs]
    double* seg_sum; double* seg_max;      // [segs] PnL sum and largest prefix sum of the chunk's records
    b200bt_chunk_item* fix_items;          // [n_seg] chunks of the individuals lane_repair_kernel touched; once their
    int32_t* redo_list;                    // metrics are recomputed the same memory holds [pop] individuals to re-run
    unsigned char* redo;                   // [pop] individuals lane_repair_kernel touched
    b200bt_chunk_item* items; int32_t* seg_base; int32_t* n_chunks;   // b200bt_sweep_tiled: lane tables [n_seg], [pop], [pop]
    int64_t bytes;                         // end of the last region
    size_t cleared;                        // bytes from seg_in to the end of the counters: they start at zero
};

template <class T>
void take(uintptr_t& at, T*& p, int64_t n) {
    at = (at + 15) & ~(uintptr_t)15;
    p = reinterpret_cast<T*>(at);
    at += (uintptr_t)n * sizeof(T);
}

// Lays the workspace out from `base` (nullptr: only `bytes` is wanted).  `tiled` adds the lane tables.
ChunkWorkspace carve(void* base, int pool_blocks, int64_t segs, int n_seg, int pop, bool tiled) {
    ChunkWorkspace w{};
    uintptr_t at = (uintptr_t)base;
    take(at, w.T.pool, (int64_t)pool_blocks * CK_BLOCK);
    take(at, w.T.seg_in, segs); take(at, w.T.seg_out, segs); take(at, w.T.seg_first, segs); take(at, w.T.seg_count, segs);
    take(at, w.ctr, 1);
    take(at, w.T.next, pool_blocks);
    take(at, w.partial, segs); take(at, w.seg_sum, segs); take(at, w.seg_max, segs);
    take(at, w.fix_items, n_seg);
    w.redo_list = reinterpret_cast<int32_t*>(w.fix_items);     // (pop <= n_seg)
    take(at, w.redo, pop);
    if (tiled) { take(at, w.items, n_seg); take(at, w.seg_base, pop); take(at, w.n_chunks, pop); }
    w.bytes = (int64_t)(at - (uintptr_t)base);
    w.cleared = (size_t)((char*)(w.ctr + 1) - (char*)w.T.seg_in);
    w.T.pool_blocks = pool_blocks; w.T.alloc = &w.ctr->alloc; w.T.overflow = &w.ctr->overflow;
    return w;
}

// rows the scan kernels may copy 16 bytes at a time
bool rows_vec16(const float* price, int64_t ld_price, const float* rsi, int64_t ld_rsi) {
    return (((uintptr_t)price | (uintptr_t)rsi) & 15) == 0 && ld_price % 4 == 0 && ld_rsi % 4 == 0;
}

ChunkScanArgs chunk_scan_args(const float* price, int64_t ld_price, const float* rsi, int64_t ld_rsi, int P, int S, int64_t N,
                              const b200bt_individual* indiv, const b200bt_chunk_item* items, int n_items, int n_seg, int warm,
                              const int32_t* n_chunks, const ChunkWorkspace& w) {
    ChunkScanArgs A;
    A.price = price; A.ld_price = ld_price; A.rsi = rsi; A.ld_rsi = ld_rsi; A.P = P; A.S = S; A.N = N;
    A.indiv = indiv; A.items = items; A.n_items = n_items; A.n_seg = n_seg; A.warm = warm;
    A.T = w.T; A.n_chunks = n_chunks; A.redo = nullptr;
    return A;
}

// second stream + events for the overlapped repair tail, one set per device
struct SideStream { cudaStream_t stream = nullptr; cudaEvent_t fork = nullptr, join = nullptr; };
int side_stream(SideStream** out) {
    static SideStream table[64];
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return cuda_status(e, "cudaGetDevice");
    B200BT_REQUIRE(dev >= 0 && dev < 64, B200BT_ELIMIT, "device ordinal %d out of range", dev);
    SideStream& s = table[dev];
    if (!s.stream) {
        int lo_p = 0, hi_p = 0;
        cudaDeviceGetStreamPriorityRange(&lo_p, &hi_p);   // highest priority: its few small kernels go first
        e = cudaStreamCreateWithPriority(&s.stream, cudaStreamNonBlocking, hi_p);
        if (e == cudaSuccess) e = cudaEventCreateWithFlags(&s.fork, cudaEventDisableTiming);
        if (e == cudaSuccess) e = cudaEventCreateWithFlags(&s.join, cudaEventDisableTiming);
        if (e != cudaSuccess) { s.stream = nullptr; return cuda_status(e, "side stream"); }
    }
    *out = &s;
    return B200BT_OK;
}

// Everything after the speculative scan: verify + repair -> chunk-parallel metrics.
//
// chunk_repair_kernel on the critical path makes almost every lane consistent; what it leaves is a handful of lanes whose
// trajectories do not meet the recorded ones inside a chunk (always in the market) and which have to be re-scanned chunk
// after chunk by a single warp each.  That is lane_repair_kernel, on another stream BESIDE the metrics kernels of all
// lanes; the individuals it touches are flagged and only their metrics are recomputed afterwards.
// max_repair_rounds: 0 = no repair (every inconsistent lane takes the exact fallback), 1 = chunk_repair_kernel only, >= 2 = both.
int finish_chunks(const ChunkScanArgs& A, const ChunkWorkspace& w, const bool vec16, const int32_t* seg_base, int pop,
                  int max_repair_rounds, const b200bt_sweep_config* cfg_host, b200bt_lane_stats* stats, uint32_t* events,
                  int64_t event_cap, unsigned char* lane_invalid, int* overflow_host_or_null, cudaStream_t st) {
    const int S = A.S, n_seg = A.n_seg, n_items = A.n_items;
    auto kern_fix = vec16 ? chunk_repair_kernel<true> : chunk_repair_kernel<false>;
    auto kern_walk = vec16 ? lane_repair_kernel<true> : lane_repair_kernel<false>;
    const size_t smem = sizeof(WarpShared) * SW_WARPS;
    cudaError_t e = cudaFuncSetAttribute(kern_fix, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(kern_walk, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return cuda_status(e, "sweep_chunked: cudaFuncSetAttribute");
    const int64_t lanes = (int64_t)pop * S;
    const int64_t mblocks = (int64_t)((n_items + 3) / 4) * S;
    B200BT_REQUIRE(mblocks < (1ll << 31), B200BT_ELIMIT, "sweep_chunked: too many work items");
    B200BT_REQUIRE(lanes < (1ll << 30), B200BT_ELIMIT, "sweep_chunked: too many lanes");

    // Both repair kernels run a persistent grid (3 CTAs per SM) whose warps take work from a counter (repair_work).
    int dev = 0, sms = 148;
    if (cudaGetDevice(&dev) == cudaSuccess) cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    const unsigned repair_grid = 3u * (unsigned)sms;
    // (the fix-up pass reuses the full-size grid with a device-side item count: CTAs beyond it leave at once)
    auto metrics = [&](const b200bt_chunk_item* its, const int* n_dev) -> int {
        chunk_sums_kernel<<<(unsigned)mblocks, 128, 0, st>>>(A.price, A.ld_price, A.indiv, its, n_items, S, n_seg, w.T.pool, w.T.next,
                                                              w.T.seg_first, w.T.seg_count, w.T.seg_in, w.seg_sum, w.seg_max, n_dev,
                                                              w.T.pool_blocks);
        B200BT_LAUNCH_CHECK("chunk_sums launch");
        chunk_partial_kernel<<<(unsigned)mblocks, 128, 0, st>>>(A.price, A.ld_price, A.indiv, its, n_items, S, n_seg, w.T.pool, w.T.next,
                                                                 w.T.seg_first, w.T.seg_count, w.T.seg_in, w.seg_sum, w.seg_max,
                                                                 *cfg_host, events, event_cap, w.partial, n_dev, w.T.pool_blocks);
        B200BT_LAUNCH_CHECK("chunk_partial launch");
        return B200BT_OK;
    };

    int rc = B200BT_OK;
    const bool tail = max_repair_rounds >= 2;
    if (max_repair_rounds >= 1) {
        kern_fix<<<repair_grid, SW_WARPS * 32, smem, st>>>(A, &w.ctr->repair_work[0]);
        B200BT_LAUNCH_CHECK("repair launch");
    }
    SideStream* side = nullptr;
    e = cudaMemsetAsync(w.redo, 0, (size_t)pop, st);
    if (e != cudaSuccess) return cuda_status(e, "sweep_chunked: memset");
    if (tail) {
        if ((rc = side_stream(&side))) return rc;
        e = cudaEventRecord(side->fork, st);
        if (e != cudaSuccess) return cuda_status(e, "sweep_chunked: fork");
    }
    if ((rc = metrics(A.items, nullptr))) return rc;
    if (tail) {
        e = cudaStreamWaitEvent(side->stream, side->fork, 0);
        if (e != cudaSuccess) return cuda_status(e, "sweep_chunked: side wait");
        ChunkScanArgs R = A;
        R.redo = w.redo;
        kern_walk<<<repair_grid, SW_WARPS * 32, smem, side->stream>>>(R, pop, seg_base, &w.ctr->repair_work[1]);
        B200BT_LAUNCH_CHECK("repair launch");
        e = cudaEventRecord(side->join, side->stream);
        if (e == cudaSuccess) e = cudaStreamWaitEvent(st, side->join, 0);
        if (e != cudaSuccess) return cuda_status(e, "sweep_chunked: join");
        fix_items_kernel<<<(n_items + 255) / 256, 256, 0, st>>>(A.items, n_items, w.redo, w.fix_items, &w.ctr->n_fix);
        B200BT_LAUNCH_CHECK("fix_items launch");
        if ((rc = metrics(w.fix_items, &w.ctr->n_fix))) return rc;
    }
    lane_combine_kernel<<<(unsigned)((lanes + 127) / 128), 128, 0, st>>>(A.indiv, pop, S, seg_base, A.n_chunks, n_seg, w.T.seg_count,
                                                                        w.T.seg_in, w.T.seg_out, w.partial, *cfg_host, stats,
                                                                        lane_invalid);
    B200BT_LAUNCH_CHECK("lane_combine launch");
    // exact fallback, driven from the device: the flagged individuals are listed and re-evaluated by the fused (serial)
    // kernel; with nothing flagged its warps leave at once
    redo_list_kernel<<<(pop + 127) / 128, 128, 0, st>>>(pop, S, lane_invalid, w.redo_list, &w.ctr->n_redo, &w.ctr->n_flagged);
    B200BT_LAUNCH_CHECK("redo_list launch");
    if ((rc = launch_sweep(A.price, A.ld_price, A.rsi, A.ld_rsi, A.P, S, A.N, A.indiv, w.redo_list, pop, &w.ctr->n_redo, cfg_host,
                           stats, events, event_cap, st)))
        return rc;
    if (overflow_host_or_null) {      // (read by the host after its next sync)
        e = cudaMemcpyAsync(overflow_host_or_null, w.ctr, 4 * sizeof(int), cudaMemcpyDeviceToHost, st);
        if (e != cudaSuccess) return cuda_status(e, "sweep_chunked: overflow readback");
    }
    if (trace_launches()) {
        int d[9];
        if (cudaMemcpy(d, w.ctr->scan_stalls, sizeof(d), cudaMemcpyDeviceToHost) == cudaSuccess && d[0])
            fprintf(stderr, "[b200bt] lane_scan: %d tile(s) timed out; first: block %d warp %d item(wslot,sym,c) %d,%d,%d tile %d of %d stage %d parity %d tl_begin %d rows %d\n",
                    d[0], d[1], d[2], d[3] >> 16, (d[3] >> 8) & 255, d[3] & 255, d[4], d[5], d[6] >> 1, d[6] & 1, d[7], d[8]);
    }
    return B200BT_OK;
}

int check_sweep_args(const char* who, const float* price, int64_t ld_price, const float* rsi, int64_t ld_rsi, int P, int S,
                     int64_t N, const b200bt_sweep_config* cfg_host, const uint32_t* events, int64_t event_cap) {
    B200BT_REQUIRE(price && rsi && cfg_host, B200BT_EINVAL, "%s: null pointer", who);
    B200BT_REQUIRE(S > 0 && N > 0 && P > 0, B200BT_EINVAL, "%s: bad sizes", who);
    B200BT_REQUIRE(ld_price >= N && ld_rsi >= N, B200BT_EINVAL, "%s: row stride shorter than N", who);
    B200BT_REQUIRE(N < (1ll << 30), B200BT_ELIMIT, "%s: N must be < 2^30 bars", who);
    B200BT_REQUIRE(cfg_host->bar_minutes > 0 && cfg_host->minute0 >= 0 && cfg_host->gap_minutes >= 0 &&
                       cfg_host->minute0 + N * (int64_t)cfg_host->bar_minutes + cfg_host->gap_minutes < (1ll << 32) - 1440,
                   B200BT_ELIMIT, "%s: minute0 + N*bar_minutes must stay below 2^32 minutes", who);
    B200BT_REQUIRE(events == nullptr || event_cap > 0, B200BT_EINVAL, "%s: event buffer without capacity", who);
    return B200BT_OK;
}

}  // namespace

extern "C" int64_t b200bt_sweep_chunked_workspace_bytes(int pool_blocks, int S, int n_seg) {
    return carve(nullptr, pool_blocks, (int64_t)S * n_seg, n_seg, n_seg, false).bytes;   // pop <= n_seg
}

extern "C" int b200bt_sweep_chunked(const float* price, int64_t ld_price, const float* rsi, int64_t ld_rsi, int P, int S,
                                    int64_t N, const b200bt_individual* indiv, const int32_t* order, int pop,
                                    const b200bt_chunk_item* items, int n_items, const int32_t* seg_base,
                                    const int32_t* n_chunks, int n_seg, int warm, int max_repair_rounds, int pool_blocks,
                                    void* workspace, int64_t workspace_bytes, const b200bt_sweep_config* cfg_host,
                                    b200bt_lane_stats* stats, uint32_t* events, int64_t event_cap,
                                    unsigned char* lane_invalid, int* overflow_host_or_null, b200bt_stream_t stream) {
    (void)order;
    B200BT_REQUIRE(indiv && items && seg_base && n_chunks && workspace && stats && lane_invalid, B200BT_EINVAL,
                   "sweep_chunked: null pointer");
    B200BT_REQUIRE(pop > 0 && n_items > 0 && n_seg > 0 && pool_blocks > 0 && warm >= 0, B200BT_EINVAL, "sweep_chunked: bad sizes");
    int rc = check_sweep_args("sweep_chunked", price, ld_price, rsi, ld_rsi, P, S, N, cfg_host, events, event_cap);
    if (rc) return rc;
    B200BT_REQUIRE(workspace_bytes >= b200bt_sweep_chunked_workspace_bytes(pool_blocks, S, n_seg), B200BT_EINVAL,
                   "sweep_chunked: workspace too small");
    B200BT_REQUIRE(((uintptr_t)workspace & 15) == 0, B200BT_EINVAL, "sweep_chunked: workspace must be 16-byte aligned");
    rc = check_device();
    if (rc) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    const int64_t segs = (int64_t)S * n_seg;
    B200BT_REQUIRE(pop <= n_seg, B200BT_EINVAL, "sweep_chunked: fewer segments than individuals");
    const ChunkWorkspace w = carve(workspace, pool_blocks, segs, n_seg, pop, false);
    cudaError_t e = cudaMemsetAsync(w.T.seg_in, 0, w.cleared, st);
    if (e != cudaSuccess) return cuda_status(e, "sweep_chunked: memset");

    const ChunkScanArgs A = chunk_scan_args(price, ld_price, rsi, ld_rsi, P, S, N, indiv, items, n_items, n_seg, warm, n_chunks, w);
    const bool vec16 = rows_vec16(price, ld_price, rsi, ld_rsi);
    auto kern = vec16 ? chunk_scan_kernel<true> : chunk_scan_kernel<false>;
    const size_t smem = sizeof(WarpShared) * SW_WARPS;
    e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return cuda_status(e, "sweep_chunked: cudaFuncSetAttribute");
    const int64_t blocks = (int64_t)((n_items + SW_WARPS - 1) / SW_WARPS) * S;
    B200BT_REQUIRE(blocks < (1ll << 31), B200BT_ELIMIT, "sweep_chunked: too many work items");
    kern<<<(unsigned)blocks, SW_WARPS * 32, smem, st>>>(A);
    B200BT_LAUNCH_CHECK("chunk_scan launch");
    return finish_chunks(A, w, vec16, seg_base, pop, max_repair_rounds, cfg_host, stats, events, event_cap, lane_invalid,
                         overflow_host_or_null, st);
}

extern "C" int64_t b200bt_zone_map_floats(int P, int S, int64_t N) {
    if (P <= 0 || S <= 0 || N <= 0) return 0;
    return (int64_t)S * (P + 1) * (zone_row_stride(N) + zone_fine_stride(N)) * 2;
}

extern "C" int b200bt_zone_map(const float* price, int64_t ld_price, const float* rsi, int64_t ld_rsi, int P, int S, int64_t N,
                               float* zones, b200bt_stream_t stream) {
    B200BT_REQUIRE(price && rsi && zones, B200BT_EINVAL, "zone_map: null pointer");
    B200BT_REQUIRE(P > 0 && S > 0 && N > 0 && ld_price >= N && ld_rsi >= N, B200BT_EINVAL, "zone_map: bad sizes");
    B200BT_REQUIRE(((uintptr_t)zones & 15) == 0, B200BT_EINVAL, "zone_map: output must be 16-byte aligned");
    int rc = check_device();
    if (rc) return rc;
    const int64_t stride = zone_row_stride(N), fstride = zone_fine_stride(N);
    const int64_t blocks = max(stride, fstride / (LS_ZONE / 4));
    const unsigned gx = (unsigned)min((int64_t)1024, (blocks + 7) / 8);
    float2* coarse = (float2*)zones;
    float2* fine = coarse + (int64_t)S * (P + 1) * stride;          // (16-byte aligned: stride is even)
    zone_map_kernel<<<dim3(gx, (unsigned)(S * (P + 1))), 256, 0, (cudaStream_t)stream>>>(price, ld_price, rsi, ld_rsi, P, N, stride, fstride,
                                                                                       coarse, fine);
    B200BT_LAUNCH_CHECK("zone_map launch");
    return B200BT_OK;
}

extern "C" int64_t b200bt_sweep_tiled_workspace_bytes(int pool_blocks, int S, int pop, int K) {
    const int64_t n_seg = (int64_t)pop * K;
    return carve(nullptr, pool_blocks, S * n_seg, (int)n_seg, pop, true).bytes;
}

// measurement hook: a pair of caller-owned CUDA events recorded around the scan kernel of the next b200bt_sweep_tiled calls
static cudaEvent_t g_scan_ev[2] = {nullptr, nullptr};
static long long g_wait_cycles = 0;
extern "C" int b200bt_sweep_scan_wait_cycles(int64_t cycles) {
    g_wait_cycles = cycles;
    return B200BT_OK;
}
extern "C" int b200bt_sweep_scan_timing(void* start_event, void* stop_event) {
    g_scan_ev[0] = (cudaEvent_t)start_event;
    g_scan_ev[1] = (cudaEvent_t)stop_event;
    return B200BT_OK;
}

extern "C" int b200bt_sweep_tiled(const float* price, int64_t ld_price, const float* rsi, int64_t ld_rsi, int P, int S,
                                  int64_t N, const float* zones_or_null, const b200bt_individual* indiv, const int32_t* slots,
                                  int n_slots, const int32_t* order, int pop, int K, int warm, int max_repair_rounds, int pool_blocks, void* workspace,
                                  int64_t workspace_bytes, const b200bt_sweep_config* cfg_host, b200bt_lane_stats* stats,
                                  uint32_t* events, int64_t event_cap, unsigned char* lane_invalid, int* overflow_host_or_null,
                                  b200bt_stream_t stream) {
    B200BT_REQUIRE(indiv && workspace && stats && lane_invalid, B200BT_EINVAL, "sweep_tiled: null pointer");
    B200BT_REQUIRE(pop > 0 && K > 0 && K <= 120 && pool_blocks > 0 && warm >= 0, B200BT_EINVAL, "sweep_tiled: bad sizes (1 <= K <= 120)");
    B200BT_REQUIRE(slots ? (n_slots > 0 && n_slots % 32 == 0) : true, B200BT_EINVAL, "sweep_tiled: n_slots must be a positive multiple of 32");
    if (!slots) n_slots = (pop + 31) & ~31;
    int rc = check_sweep_args("sweep_tiled", price, ld_price, rsi, ld_rsi, P, S, N, cfg_host, events, event_cap);
    if (rc) return rc;
    B200BT_REQUIRE((int64_t)pop * K * S < (1ll << 31), B200BT_ELIMIT, "sweep_tiled: too many chunks");
    B200BT_REQUIRE(K == 1 || N / K >= SW_GROUP, B200BT_EINVAL, "sweep_tiled: chunks shorter than %d bars", SW_GROUP);
    // shared-memory rings: one per warp, LS_STAGES tiles of LS_ROWS rows (+ their zone ranges): independent of P
    const size_t smem = (size_t)LS_WARPS * LS_STAGES * LS_ROWS * (LS_STRIDE * sizeof(float) + (zones_or_null ? (LS_T / LS_ZONE + LS_T / 4) * sizeof(float2) : 0));
    B200BT_REQUIRE(zones_or_null == nullptr || ((uintptr_t)zones_or_null & 15) == 0, B200BT_EINVAL, "sweep_tiled: zone map must be 16-byte aligned");
    B200BT_REQUIRE(workspace_bytes >= b200bt_sweep_tiled_workspace_bytes(pool_blocks, S, pop, K), B200BT_EINVAL,
                   "sweep_tiled: workspace too small");
    B200BT_REQUIRE(((uintptr_t)workspace & 15) == 0, B200BT_EINVAL, "sweep_tiled: workspace must be 16-byte aligned");
    rc = check_device();
    if (rc) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    const int n_seg = pop * K;
    const int64_t segs = (int64_t)S * n_seg;
    const ChunkWorkspace w = carve(workspace, pool_blocks, segs, n_seg, pop, true);
    cudaError_t e = cudaMemsetAsync(w.T.seg_in, 0, w.cleared, st);
    if (e != cudaSuccess) return cuda_status(e, "sweep_tiled: memset");
    lane_tables_kernel<<<(n_seg + 255) / 256, 256, 0, st>>>(pop, K, order, w.items, w.seg_base, w.n_chunks);
    B200BT_LAUNCH_CHECK("lane_tables launch");

    LaneScanArgs L;
    L.price = price; L.ld_price = ld_price; L.rsi = rsi; L.ld_rsi = ld_rsi; L.P = P; L.S = S; L.N = N;
    L.zones = (const float2*)zones_or_null; L.n_zone_blocks = zone_row_stride(N);    // (row stride of the zone map)
    L.fine = zones_or_null ? L.zones + (int64_t)S * (P + 1) * zone_row_stride(N) : nullptr; L.n_fine = zone_fine_stride(N);
    L.indiv = indiv; L.slots = slots; L.n_slots = n_slots; L.pop = pop; L.K = K; L.warm = warm;
    L.T = w.T;
    L.work = &w.ctr->scan_work;
    L.stalls = w.ctr->scan_stalls;
    L.wait_cycles = g_wait_cycles != 0 ? g_wait_cycles : LS_WAIT_CYCLES;
    const bool vec16 = rows_vec16(price, ld_price, rsi, ld_rsi);
    auto kern = zones_or_null ? lane_scan_kernel<true> : lane_scan_kernel<false>;
    e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
    if (e != cudaSuccess) return cuda_status(e, "sweep_tiled: cudaFuncSetAttribute");
    const int64_t n_items = (int64_t)(n_slots / 32) * K * S;
    B200BT_REQUIRE(n_items < (1ll << 30), B200BT_ELIMIT, "sweep_tiled: too many work items");
    // persistent grid: one resident set of CTAs (warps take work items from the counter), no more CTAs than items need
    int dev = 0, sms = 0, per_sm = 0;
    e = cudaGetDevice(&dev);
    if (e == cudaSuccess) e = cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    if (e == cudaSuccess) e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, LS_THREADS, smem);
    if (e != cudaSuccess) return cuda_status(e, "sweep_tiled: occupancy");
    int64_t blocks = (int64_t)sms * (per_sm > 0 ? per_sm : 1);
    if (blocks > (n_items + LS_WARPS - 1) / LS_WARPS) blocks = (n_items + LS_WARPS - 1) / LS_WARPS;
    if (g_scan_ev[0]) cudaEventRecord(g_scan_ev[0], st);
    kern<<<(unsigned)blocks, LS_THREADS, smem, st>>>(L, vec16);
    if (g_scan_ev[1]) cudaEventRecord(g_scan_ev[1], st);
    B200BT_LAUNCH_CHECK("lane_scan launch");

    const ChunkScanArgs A = chunk_scan_args(price, ld_price, rsi, ld_rsi, P, S, N, indiv, w.items, n_seg, n_seg, warm, w.n_chunks, w);
    return finish_chunks(A, w, vec16, w.seg_base, pop, max_repair_rounds, cfg_host, stats, events, event_cap, lane_invalid,
                         overflow_host_or_null, st);
}
