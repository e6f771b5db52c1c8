"""Population-fitness sweep: the GA hot path on the GPU.

Host side of `b200bt_sweep`, `b200bt_sweep_chunked` and `b200bt_sweep_tiled` (include/b200bt.h): three schedules of
the same computation, chosen by `PopulationSweep.plan`.  For every (individual, symbol) lane they evaluate what the
reference evaluates serially in Python:

    trades  = StrategyEvaluationSystem._simulate_trades(id, params, bars)   strategy_evaluation.py:746
    metrics = StrategyPerformanceMetrics.calculate_metrics(trades)          :32
    score   = StrategyEvaluationSystem._calculate_strategy_score(metrics)   :579

and reduces fitness(individual) = mean over symbols of score.  (The
composition simulate -> metrics -> score is the reference's own, see
cross_validate_strategy :682-691; the mean over symbols mirrors its mean over
folds, :1030-1060.)

PyTorch is used for device memory and streams only; all arithmetic happens in
the hand-written sm_100a kernels behind the C-ABI.
"""
from __future__ import annotations

import ctypes as C
import inspect
import os
from typing import Dict, Iterable, List, Optional, Sequence, Tuple

import numpy as np
import torch

from . import _lib
from .synth import EPOCH_2024_MINUTES

DEFAULT_GOALS = {  # config.json: evolution.optimization_goals
    "primary": "sharpe_ratio",
    "secondary": ["max_drawdown", "win_rate", "profit_factor"],
}


def _f32_up(x: float) -> np.float32:
    """Smallest float32 >= x."""
    f = np.float32(x)
    return f if float(f) >= x else np.nextafter(f, np.float32(np.inf))


def _f32_down(x: float) -> np.float32:
    """Largest float32 <= x."""
    f = np.float32(x)
    return f if float(f) <= x else np.nextafter(f, np.float32(-np.inf))


class MarketData:
    """Device-resident fp32 OHLCV, field-major SoA [5][S][N] (open, high, low, close, volume).
    `MarketData.from_close(close_dev, ...)` wraps device close prices alone (other fields zero).

    Mirrors the role of HistoricalDataManager.market_data_cache
    (backtesting/data_manager.py:218-220): load once, reuse across calls.

    From a PINNED host tensor only the close prices are uploaded at construction; open / high / low / volume are
    uploaded when first read (`materialise()` forces it), so the source must stay unchanged until then.
    """

    def __init__(self, ohlcv, symbols: Optional[Sequence[str]] = None,
                 minute0: int = EPOCH_2024_MINUTES, bar_minutes: int = 1,
                 device: Optional[torch.device] = None, pinned_source: bool = False):
        if not torch.cuda.is_available():
            raise RuntimeError("MarketData needs a CUDA device (sm_100); this engine has no CPU path")
        self.device = torch.device(device) if device is not None else torch.device("cuda", torch.cuda.current_device())
        if isinstance(ohlcv, torch.Tensor):
            host = ohlcv
        else:
            host = torch.from_numpy(np.ascontiguousarray(ohlcv, dtype=np.float32))
        if host.dim() != 3 or host.shape[0] != 5:
            raise ValueError("ohlcv must have shape [5][S][N] (open, high, low, close, volume)")
        self.S = int(host.shape[1])
        self.N = int(host.shape[2])
        self._pending_host = None       # pinned source whose open / high / low / volume rows are not on the device yet
        self._close_parts = []
        self.h2d_bytes = 0              # bytes this object has copied host -> device so far
        if host.is_cuda or not host.is_pinned():
            self._ohlcv = host.to(self.device, non_blocking=True).contiguous()
            self.h2d_bytes = 0 if host.is_cuda else host.numel() * 4
        else:
            # pinned host source: only the close prices (all the sweep and the RSI bank read) are uploaded now, in four
            # concurrent quarter copies (one 40 MB copy reaches ~24 GB/s here, four ~33 GB/s: tools/h2d_bandwidth.py);
            # open / high / low / volume follow on first use (the indicator kernels), so a GA generation does not move them
            host = host.contiguous()
            self._ohlcv = torch.empty(host.shape, dtype=torch.float32, device=self.device)
            cur = torch.cuda.current_stream(self.device)
            parts = min(4, self.S)
            lanes = [_copy_stream(self.device, 1 + i) for i in range(parts)]
            rows = [(i * self.S) // parts for i in range(parts + 1)]
            self._close_parts = []      # (row lo, row hi, stream) of the quarter copies the current stream has not joined yet
            for st, lo, hi in zip(lanes, rows[:-1], rows[1:]):
                st.wait_stream(cur)                                          # (allocation order)
                with torch.cuda.stream(st):
                    self._ohlcv[3, lo:hi].copy_(host[3, lo:hi], non_blocking=True)
                self._close_parts.append((lo, hi, st))
            self._pending_host = host
            self.h2d_bytes = self.S * self.N * 4
        self.symbols = list(symbols) if symbols is not None else [f"SYN{i:03d}USDT" for i in range(self.S)]
        self.minute0 = int(minute0)
        self.bar_minutes = int(bar_minutes)

    @classmethod
    def from_close(cls, close: torch.Tensor, minute0: int = EPOCH_2024_MINUTES, bar_minutes: int = 1,
                   symbols: Optional[Sequence[str]] = None) -> "MarketData":
        assert close.is_cuda and close.dtype == torch.float32 and close.dim() == 2
        ohlcv = torch.zeros((5,) + tuple(close.shape), dtype=torch.float32, device=close.device)
        ohlcv[3] = close
        return cls(ohlcv, symbols=symbols, minute0=minute0, bar_minutes=bar_minutes, device=close.device)

    def materialise(self) -> "MarketData":
        """Make all five fields device-resident now."""
        self._wait_others()
        return self

    def _wait_others(self) -> None:
        """Upload the fields that are still on the host (current stream)."""
        host = self._pending_host
        if host is not None:
            self._pending_host = None
            for f in (0, 1, 2, 4):
                self._ohlcv[f].copy_(host[f], non_blocking=True)
            self.h2d_bytes += 4 * self.S * self.N * 4

    @property
    def ohlcv(self) -> torch.Tensor:
        self._wait_others()
        return self._ohlcv

    def _join_close(self) -> None:
        """The current stream waits for the quarter copies of the close prices (once)."""
        if self._close_parts:
            cur = torch.cuda.current_stream(self.device)
            for _, _, st in self._close_parts:
                cur.wait_stream(st)
            self._close_parts = []

    @property
    def close(self) -> torch.Tensor:
        self._join_close()
        return self._ohlcv[3]

    @property
    def high(self) -> torch.Tensor:
        return self.ohlcv[1]

    @property
    def low(self) -> torch.Tensor:
        return self.ohlcv[2]

    @property
    def open(self) -> torch.Tensor:
        return self.ohlcv[0]

    @property
    def volume(self) -> torch.Tensor:
        return self.ohlcv[4]


_COPY_STREAMS: Dict[Tuple[int, int], "torch.cuda.Stream"] = {}


def _copy_stream(device: torch.device, which: int = 0) -> "torch.cuda.Stream":
    idx = device.index if device.index is not None else torch.cuda.current_device()
    if (idx, which) not in _COPY_STREAMS:
        _COPY_STREAMS[(idx, which)] = torch.cuda.Stream(device=device)
    return _COPY_STREAMS[(idx, which)]


def rsi_bank(close: torch.Tensor, periods: Sequence[int], fill: bool = True,
             out: Optional[torch.Tensor] = None, zones: Optional[torch.Tensor] = None, zones_symbols: int = 0,
             first_symbol: int = 0) -> torch.Tensor:
    """RSI for every window in `periods`: close [S][N] fp32 -> [S][P][N] fp32.

    ta.momentum.RSIIndicator semantics as used at binance_ml_strategy.py:112.
    `zones`: a sweep zone map (zone_map_floats(P, zones_symbols, N) floats) whose rows of the symbols
    [first_symbol, first_symbol + S) are written in the same pass (b200bt_rsi_bank_zones; needs fill=True).
    """
    assert close.is_cuda and close.dtype == torch.float32 and close.dim() == 2
    S, N = close.shape
    P = len(periods)
    if out is None:
        out = torch.empty((S, P, N), dtype=torch.float32, device=close.device)
    arr = (C.c_int * P)(*[int(p) for p in periods])
    with torch.cuda.device(close.device):
        if zones is not None:
            assert fill, "zone rows describe the NaN-filled bank"
            _lib.call("b200bt_rsi_bank_zones", close.data_ptr(), S, N, _lib.ld(close), arr, P, out.data_ptr(), zones.data_ptr(),
                      int(zones_symbols), int(first_symbol), _lib.current_stream())
        else:
            _lib.call("b200bt_rsi_bank", close.data_ptr(), S, N, _lib.ld(close), arr, P, 1 if fill else 0,
                      out.data_ptr(), _lib.current_stream())
    return out


def decode_population(population: List[Dict], period_row: Dict[int, int], n_timeframes: int = 1) -> np.ndarray:
    """List of GA parameter dicts -> packed b200bt_individual array (numpy structured).

    With `n_timeframes` > 1 the bank holds one block of len(period_row) rows per timeframe and the gene
    `rsi_timeframe` (an index into PopulationSweep.timeframes, default 0 = the base clock) selects the block."""
    dt = np.dtype([("rsi_row", "<i4"), ("rsi_lo", "<f4"), ("rsi_hi", "<f4"), ("reserved", "<i4"),
                   ("take_profit", "<f8"), ("stop_loss", "<f8"), ("position_size", "<f8")])
    assert dt.itemsize == C.sizeof(_lib.Individual)
    out = np.zeros(len(population), dtype=dt)
    g = lambda key, default: np.array([p.get(key, default) for p in population], dtype=np.float64)
    period = g("rsi_period", 14).astype(np.int64)
    rows = np.full(int(period.max()) + 2 if len(period) else 1, -1, dtype=np.int64)
    for w, r in period_row.items():
        if 0 <= w < len(rows):
            rows[w] = r
    row = rows[np.clip(period, 0, len(rows) - 1)]
    if len(period) and (period.min() < 0 or row.min() < 0):
        bad = int(period[(row < 0) | (period < 0)][0])
        raise KeyError(f"rsi_period {bad} is not in the RSI bank {sorted(period_row)}")
    if n_timeframes > 1:
        tf = g("rsi_timeframe", 0).astype(np.int64)
        if len(tf) and (tf.min() < 0 or tf.max() >= n_timeframes):
            raise KeyError(f"rsi_timeframe {int(tf[(tf < 0) | (tf >= n_timeframes)][0])} is not an index into the {n_timeframes} timeframes of the bank")
        row = row + tf * len(period_row)
    out["rsi_row"] = row
    # thresholds rounded towards the side that keeps `rsi < oversold` / `rsi > overbought` exact in fp32
    lo, hi = g("rsi_oversold", 30), g("rsi_overbought", 70)
    lo32, hi32 = lo.astype(np.float32), hi.astype(np.float32)
    out["rsi_lo"] = np.where(lo32.astype(np.float64) >= lo, lo32, np.nextafter(lo32, np.float32(np.inf)))
    out["rsi_hi"] = np.where(hi32.astype(np.float64) <= hi, hi32, np.nextafter(hi32, np.float32(-np.inf)))
    # strategy_evaluation.py:762-764, :773-774 (same float64 expressions)
    out["take_profit"] = g("take_profit", 3) / 100
    out["stop_loss"] = g("stop_loss", 2) / 100
    out["position_size"] = 10000 * (np.minimum(g("max_position_size", 5), 20) / 100)
    return out


def lane_cost(p: Dict) -> float:
    """Fraction of bars on which RSI(w) sits outside [oversold, overbought] under the model
    RSI(w) ~ N(50, 44/sqrt(w)): the lane's trade-event rate is proportional to it (measured on the
    synthetic 1-minute data: events ~= 0.27 * cost * bars).  Scheduling only; never affects results."""
    from math import erf, sqrt
    w = int(p.get("rsi_period", 14))
    sd = 44.0 / sqrt(max(w, 1))
    phi = lambda x: 0.5 * (1.0 + erf(x / sqrt(2.0)))
    return phi((float(p.get("rsi_oversold", 30)) - 50.0) / sd) + 1.0 - phi((float(p.get("rsi_overbought", 70)) - 50.0) / sd)


EVENTS_PER_COST_BAR = 0.27


def predicted_events(population: List[Dict], n_bars: int) -> np.ndarray:
    """Expected trade records per (individual, symbol) lane under the lane_cost model."""
    return EVENTS_PER_COST_BAR * lane_costs(population) * n_bars


def lane_costs(population: List[Dict]) -> np.ndarray:
    """lane_cost for a whole population (vectorised)."""
    from scipy.special import ndtr
    g = lambda key, default: np.array([float(p.get(key, default)) for p in population], dtype=np.float64)
    sd = 44.0 / np.sqrt(np.maximum(g("rsi_period", 14).astype(np.int64), 1))
    return ndtr((g("rsi_oversold", 30) - 50.0) / sd) + 1.0 - ndtr((g("rsi_overbought", 70) - 50.0) / sd)


_HASH_MULTIPLIERS = np.array([0x9E3779B97F4A7C15, 0xC2B2AE3D27D4EB4F, 0x165667B19E3779F9, 0x27D4EB2F165667C5,
                              0x85EBCA77C2B2AE63], dtype=np.uint64)


def _duplicate_classes(packed: np.ndarray):
    """(first index of each distinct record, class of every record), or None when all records are distinct.
    Records are compared through a 64-bit multiplicative hash of their 40 bytes (3x faster than sorting the structured
    array); a hash class is only trusted after every member is compared with its representative."""
    words = packed.view(np.uint64).reshape(len(packed), -1)
    with np.errstate(over="ignore"):
        key = (words * _HASH_MULTIPLIERS[:words.shape[1]]).sum(axis=1, dtype=np.uint64)
    uk, first, inverse = np.unique(key, return_index=True, return_inverse=True)
    if len(uk) == len(packed):
        return None
    inverse = inverse.reshape(-1)
    if not bool((packed[first][inverse] == packed).all()):       # a collision merged different records: exact path
        _, first, inverse = np.unique(packed, return_index=True, return_inverse=True)
        inverse = inverse.reshape(-1)
    return (first, inverse) if len(first) < len(packed) else None


def costs_from_packed(packed: np.ndarray, periods: Sequence[int], timeframes: Sequence[int] = (1,)) -> np.ndarray:
    """lane_cost of already decoded individuals (b200bt_individual records): no second pass over the dicts.  An RSI row
    of a k-times slower clock changes every k bars: its threshold crossings (events) are rarer by about sqrt(k)."""
    from scipy.special import ndtr
    P = len(periods)
    w = np.asarray(periods, dtype=np.float64)[packed["rsi_row"] % P]
    sd = 44.0 / np.sqrt(np.maximum(w, 1.0))
    c = ndtr((packed["rsi_lo"].astype(np.float64) - 50.0) / sd) + 1.0 - ndtr((packed["rsi_hi"].astype(np.float64) - 50.0) / sd)
    if len(timeframes) > 1:
        k = np.asarray(timeframes, dtype=np.float64)[packed["rsi_row"] // P] / float(timeframes[0])
        c = c / np.sqrt(k)
    return c


_SM_COUNT: Dict[int, int] = {}


def _sm_count(device) -> int:
    idx = torch.device(device).index
    idx = torch.cuda.current_device() if idx is None else idx
    if idx not in _SM_COUNT:
        _SM_COUNT[idx] = torch.cuda.get_device_properties(idx).multi_processor_count
    return _SM_COUNT[idx]


_PINNED_FLAGS = None
DEFERRED = torch.empty(0, dtype=torch.uint8)      # sentinel: the caller assigns plan.workspace (plan_batches)
_FLAG_SLOTS = 256


def _pinned_flags() -> torch.Tensor:
    """Pinned int32 [256][4]: per plan (slice) of a sweep, [0] = the event pool overflowed, [1] = lanes that went through
    the exact fallback, [2] = pool blocks handed out, [3] = scan tiles that timed out.  The kernels' flags are copied here asynchronously; the host looks at them only after a stream
    synchronisation it does anyway (page-locking memory is slow: one table shared by every plan)."""
    global _PINNED_FLAGS
    if _PINNED_FLAGS is None:
        _PINNED_FLAGS = torch.zeros((_FLAG_SLOTS, 4), dtype=torch.int32).pin_memory()
    return _PINNED_FLAGS


_NEXT_FLAG = [0]


def _flag_slot() -> torch.Tensor:
    i = _NEXT_FLAG[0] = (_NEXT_FLAG[0] + 1) % _FLAG_SLOTS
    return _pinned_flags()[i]


class _SweepPlan:
    """What both time-chunked plans hold besides their schedule: the event pool, the workspace, the lanes' fallback flags
    and a slot of the pinned flag table."""

    def _allocate(self, pred: np.ndarray, n_symbols: int, device, pool_scale: float, pool_blocks: Optional[int],
                  workspace: Optional[torch.Tensor], workspace_bytes) -> None:
        """`workspace_bytes(pool_blocks)` sizes the workspace; `workspace` may be shared between the plans of successive
        slices (DEFERRED: the caller assigns it)."""
        # every segment owns at least one block, and a repaired segment abandons its first chain
        self.pred_blocks = float(pred.sum()) * n_symbols / 256
        self.pool_blocks = int(pool_scale * self.pred_blocks) + 2 * self.n_seg * n_symbols + 1024
        if pool_blocks is not None:
            self.pool_blocks = int(pool_blocks)
        self.ws_bytes = int(workspace_bytes(self.pool_blocks))
        if workspace is not None and workspace.numel() >= self.ws_bytes:
            self.workspace = workspace
        else:
            self.workspace = None if workspace is DEFERRED else torch.empty(self.ws_bytes, dtype=torch.uint8, device=device)
        self.invalid = torch.zeros((self.pop, n_symbols), dtype=torch.uint8, device=device)
        self.overflow = _flag_slot()


class ChunkPlan(_SweepPlan):
    """Host-side plan of the time-chunked sweep for one population (device tensors inside)."""

    def __init__(self, population: List[Dict], n_bars: int, n_symbols: int, device, target_events: int = 16384,
                 warm: int = 8192, max_chunks: int = 64, pool_scale: float = 1.5, pool_blocks: Optional[int] = None,
                 max_repair_rounds: int = 8, lo: int = 0, workspace: Optional[torch.Tensor] = None,
                 pred: Optional[np.ndarray] = None):
        """`population` is the slice [lo, lo + len) of the caller's population (individual indices inside the
        plan are slice-relative); `workspace` may be shared between the plans of successive slices; `pred` =
        predicted_events(population, n_bars) when the caller already has it."""
        pop = len(population)
        self.lo, self.pop = int(lo), pop
        pred = predicted_events(population, n_bars) if pred is None else np.asarray(pred, dtype=np.float64)
        kmax = max(1, min(max_chunks, n_bars // max(8 * warm, 2048)))
        k = np.clip(np.ceil(pred / target_events), 1, kmax).astype(np.int32)
        self.n_chunks = k
        self.seg_base = np.concatenate([[0], np.cumsum(k)[:-1]]).astype(np.int32)
        self.n_seg = int(k.sum())
        self.order = np.argsort(-pred, kind="stable").astype(np.int32)      # (b200bt_sweep_chunked ignores it)
        items = np.zeros((self.n_seg, 4), dtype=np.int32)
        # most expensive work first (per-chunk cost), keeping one individual's chunks together
        per_chunk = pred / k
        row = 0
        for i in sorted(range(pop), key=lambda j: (-per_chunk[j], int(population[j].get("rsi_period", 14)))):
            for c in range(int(k[i])):
                items[row] = (i, c, k[i], self.seg_base[i] + c)
                row += 1
        self.warm = int(warm)
        self.max_repair_rounds = int(max_repair_rounds)
        self.items = torch.from_numpy(items).to(device)
        self.seg_base_dev = torch.from_numpy(self.seg_base).to(device)
        self.n_chunks_dev = torch.from_numpy(self.n_chunks).to(device)
        self.order_dev = torch.from_numpy(self.order).to(device)
        self._allocate(pred, n_symbols, device, pool_scale, pool_blocks, workspace,
                       lambda blocks: _lib.load().b200bt_sweep_chunked_workspace_bytes(blocks, n_symbols, self.n_seg))


class TilePlan(_SweepPlan):
    """Host-side plan of the thread-per-lane sweep (b200bt_sweep_tiled) for one population slice: every
    individual gets the same K time chunks, chosen so that the CTAs fill whole waves of the GPU."""

    THREADS = int(os.environ.get("B200BT_LS_THREADS", 256))     # individuals per CTA (csrc/sweep_chunked.cu LS_THREADS)
    CTAS_PER_SM = int(os.environ.get("B200BT_LS_CTAS", 3))     # resident CTAs of lane_scan_kernel per SM (__launch_bounds__(256, 3))
    WARM = 1536          # warm-up bars of a speculative chunk

    @classmethod
    def chunks_for(cls, pop: int, n_bars: int, n_symbols: int, device, warm: int = WARM, max_chunks: int = 64,
                   n_slots: Optional[int] = None) -> int:
        """About 2.5 work items per resident warp slot (the scan is persistent: warps take (warp-slot, chunk, symbol) items
        from a counter, the most expensive first; more chunks balance better but every chunk pays its warm-up and its share of
        the per-chunk metrics overhead), chunks at least 3 warm-ups long.  Measured on configs[1] (3 CTAs/SM): a plateau of
        7.15-7.25 ms for K = 26..30 and warm-ups of 1024..3072 bars; K = 34 +0.3 ms, K = 24 +0.15 ms.  A short warm-up is
        affordable because a mis-speculated chunk is re-scanned only until it meets its recorded trajectory again
        (chunk_scan_item, REPAIR): at 2048 bars ~10 % of the chunks start in the wrong state and take ~3500 bars each to come
        back (at 8192 bars: 2 % and ~7700 bars)."""
        kmax = max(1, min(max_chunks, n_bars // max(3 * warm, 2048)))
        slots = _sm_count(device) * cls.CTAS_PER_SM
        groups = -(-(n_slots if n_slots is not None else pop) // cls.THREADS) * n_symbols
        return min(kmax, max(1, round(2.5 * slots / groups)))

    def __init__(self, population: List[Dict], n_bars: int, n_symbols: int, device, warm: int = WARM,
                 max_chunks: int = 64, chunks: Optional[int] = None, pool_scale: float = 1.5,
                 pool_blocks: Optional[int] = None, max_repair_rounds: Optional[int] = None, lo: int = 0,
                 workspace: Optional[torch.Tensor] = None, order_by: str = "row_cost", pred: Optional[np.ndarray] = None,
                 rows: Optional[np.ndarray] = None):
        pop = len(population)
        self.lo, self.pop = int(lo), pop
        self.warm = int(warm)
        pred = predicted_events(population, n_bars) if pred is None else np.asarray(pred, dtype=np.float64)
        # thread slots: 32 consecutive slots = one warp, which stages its own tiles and may read two distinct RSI rows
        self.slots = pack_warps(population, pred, order_by, rows)
        if chunks is None:
            chunks = self.chunks_for(pop, n_bars, n_symbols, device, warm, max_chunks, n_slots=len(self.slots))
        self.K = int(chunks)
        # 0 = no repair, 1 = the bounded pass on the critical path, 2 = that and the unbounded pass beside the metrics
        self.max_repair_rounds = int(max_repair_rounds) if max_repair_rounds is not None else 2
        self.n_seg = pop * self.K
        self.order = np.ascontiguousarray(self.slots[self.slots >= 0])      # individuals in dispatch order
        self.slots_dev = torch.from_numpy(np.concatenate([self.slots, self.order])).to(device)     # [slots | order]
        self._allocate(pred, n_symbols, device, pool_scale, pool_blocks, workspace,
                       lambda blocks: _lib.load().b200bt_sweep_tiled_workspace_bytes(blocks, n_symbols, pop, self.K))


WARP_RSI_ROWS = 2       # distinct RSI rows the machines of one warp may read (csrc/sweep_chunked.cu LS_RSI_ROWS)


def pack_warps(population: List[Dict], pred: np.ndarray, order_by: str = "row_cost", rows: Optional[np.ndarray] = None) -> np.ndarray:
    """Thread slots of the thread-per-lane scan: int32[n_warps * 32], the individual each slot runs, -1 = empty.

    A warp stages the price row and the RSI rows of its own 32 machines, at most WARP_RSI_ROWS of them, and its cost is
    the UNION of its machines' events.  So individuals are sorted by (RSI row, predicted cost) -- neighbours read the same
    row and fire at similar rates on the same bars -- and cut into warps that never span more than WARP_RSI_ROWS rows (a
    row's tail shares a warp with the head of the next row; slots stay empty only where a third row would enter).  Warps
    are then dispatched most expensive first, so that the warps resident together (and the 8 of a CTA) cost the same.
    order_by = "identity" keeps the population order (testing: warps that break the row rule are re-run by the exact
    fallback), "row_thresholds" sorts a row by (oversold, overbought) instead of cost.  `rows`: the bank row of every
    individual when it is not a function of `rsi_period` alone (several timeframes)."""
    n = len(population)
    if order_by == "identity":
        out = np.full(-(-n // 32) * 32, -1, dtype=np.int32)
        out[:n] = np.arange(n, dtype=np.int32)
        return out
    g = lambda key, default: np.array([float(p.get(key, default)) for p in population], dtype=np.float64)
    row = g("rsi_period", 14).astype(np.int64) if rows is None else np.asarray(rows, dtype=np.int64)    # (bank row when given)
    pred = np.asarray(pred, dtype=np.float64)
    rows, inv = np.unique(row, return_inverse=True)
    mean_cost = np.bincount(inv, weights=pred) / np.maximum(np.bincount(inv), 1)
    if order_by == "row_thresholds":
        idx = np.lexsort((np.arange(n), -g("rsi_overbought", 70), g("rsi_oversold", 30), -mean_cost[inv]))
    else:
        idx = np.lexsort((np.arange(n), -pred, -mean_cost[inv]))          # rows by mean cost, inside a row by cost
    counts = np.bincount(inv, minlength=len(rows))[np.argsort(-mean_cost, kind="stable")]    # members per row, in dispatch order
    warps, fill, used, pos = [], 0, 0, 0
    cur = np.full(32, -1, dtype=np.int32)
    for cnt in counts:
        left = int(cnt)
        while left:
            if fill == 32 or (fill and used == WARP_RSI_ROWS):
                warps.append(cur)
                cur, fill, used = np.full(32, -1, dtype=np.int32), 0, 0
            take = min(32 - fill, left)
            cur[fill:fill + take] = idx[pos:pos + take]
            fill, used, pos, left = fill + take, used + 1, pos + take, left - take
    if fill:
        warps.append(cur)
    warps = np.stack(warps)
    cost = np.where(warps >= 0, pred[np.maximum(warps, 0)], 0.0).sum(axis=1)
    return np.ascontiguousarray(warps[np.argsort(-cost, kind="stable")]).reshape(-1)


def evaluation_order(population: List[Dict]) -> np.ndarray:
    """Order in which the kernel dispatches individuals: same RSI period adjacent (the
    warps of a CTA then read the same RSI stream), most expensive first.

    Cost model: a lane's work is dominated by its trade events, whose rate follows the
    fraction of time RSI(w) spends outside [oversold, overbought]; RSI(w) is roughly
    N(50, 44/sqrt(w)) on 1-minute data.  Only scheduling depends on this, never results.
    """
    period = np.array([int(p.get("rsi_period", 14)) for p in population], dtype=np.int64)
    return np.lexsort((np.arange(len(population)), -lane_costs(population), period)).astype(np.int32)


class PopulationSweep:
    """Evaluate a GA population against device-resident market data.

    `sweep.fitness_function` is a callable usable as GeneticAlgorithm's
    `fitness_function`; it carries a `.batch` attribute that evaluates the whole
    population in one kernel launch (see genetic_algorithm.GeneticAlgorithm).
    """

    def __init__(self, market: MarketData, rsi_periods: Iterable[int] = range(5, 31),
                 optimization_goals: Optional[Dict] = None, initial_capital: float = 10000.0,
                 event_cap: int = 0, mode: str = "auto", chunk_options: Optional[Dict] = None,
                 score_on_advanced: bool = False, timeframes: Sequence[int] = ()):
        """score_on_advanced: take the strategy score on calculate_advanced_metrics' dict (the composition of
        evaluate_strategy, strategy_evaluation.py:545-557: `expectancy`, `sortino_ratio`, ... exist as keys) instead of the
        plain calculate_metrics dict (cross_validate_strategy :683-691, the default).
        mode: "fused" (one warp per lane, serial in time), "chunked" (expensive lanes split into verified
        time chunks, one warp per chunk), "tiled" (every lane split into the same K verified chunks, one THREAD
        per chunk; csrc/sweep_chunked.cu) or "auto" (tiled from 131072 bars up, fused below)."""
        self._configure(market, sorted(set(int(p) for p in rsi_periods)), optimization_goals, initial_capital, event_cap,
                        mode, chunk_options, score_on_advanced)
        # timeframes (minutes per bar, the first one = the market's own clock): BASELINE configs[3] evaluates the RSI rule on
        # 1m / 5m / 15m indicators (recipe: services/market_monitor_service.py:219-301); the bank then holds one block of rows
        # per timeframe, each higher-timeframe RSI brought back to the base clock by "last completed bar", and the gene
        # `rsi_timeframe` (index into `timeframes`) selects the block
        self.timeframes = tuple(int(k) for k in timeframes) or (market.bar_minutes,)
        if self.timeframes[0] != market.bar_minutes or any(k % market.bar_minutes for k in self.timeframes):
            raise ValueError("timeframes must start with the market's own bar spacing and be multiples of it")
        self.bank = self._bank_behind_the_upload(market) if len(self.timeframes) == 1 else self._multi_timeframe_bank(market)

    def _configure(self, market: MarketData, periods: List[int], optimization_goals: Optional[Dict], initial_capital: float,
                   event_cap: int, mode: str, chunk_options: Optional[Dict], score_on_advanced: bool) -> None:
        self.market = market
        self.periods = periods
        self.period_row = {p: i for i, p in enumerate(self.periods)}
        goals = optimization_goals or DEFAULT_GOALS
        primary, mask = _lib.score_codes(goals, advanced=score_on_advanced)
        self.cfg = _lib.SweepConfig(initial_capital=float(initial_capital), minute0=market.minute0,
                                    bar_minutes=market.bar_minutes, primary=primary, secondary_mask=mask, variant=0)
        self.event_cap = int(event_cap)
        self.mode, self.chunk_min_bars, self.chunk_options = mode, 131072, dict(chunk_options or {})
        self._stats = self._events = None
        self._pop = 0
        self._pinned_in = self._pinned_out = None

    def _bank_behind_the_upload(self, market: MarketData) -> torch.Tensor:
        """RSI bank of the market.  While the close prices are still arriving in quarter copies (MarketData from a
        pinned host tensor), each quarter's rows are computed on that quarter's copy stream, so the bank is ready one
        quarter of its kernel time after the last byte instead of one whole kernel."""
        parts = market._close_parts
        P = len(self.periods)
        # the zone map of the bank (ranges of every 32-bar block and 4-bar group) comes out of the same pass
        zones = torch.empty(int(_lib.load().b200bt_zone_map_floats(P, market.S, market.N)), dtype=torch.float32, device=market.device)
        if not parts:
            bank = rsi_bank(market.close, self.periods, zones=zones, zones_symbols=market.S)
            self._zones = zones
            return bank
        bank = torch.empty((market.S, P, market.N), dtype=torch.float32, device=market.device)
        cur = torch.cuda.current_stream(market.device)
        for lo, hi, st in parts:
            st.wait_stream(cur)                        # (the allocations of the bank and of the zone map)
            with torch.cuda.stream(st):
                rsi_bank(market._ohlcv[3, lo:hi], self.periods, out=bank[lo:hi], zones=zones, zones_symbols=market.S, first_symbol=lo)
        market._join_close()                           # the current stream now waits for copies AND bank rows
        self._zones = zones
        return bank

    def _multi_timeframe_bank(self, market: MarketData) -> torch.Tensor:
        """[S][T * P][N] bank: block 0 = RSI of the base clock, block i = RSI of the clock-aligned timeframes[i]-minute bars
        (b200bt_resample), NaN policy applied on that clock like the reference's analyzer does per kline series, then aligned
        to the base clock with the value of the last COMPLETED higher-timeframe bar (b200bt_align: no look-ahead; NaN before
        the first completed bar, where no threshold compare is true)."""
        from . import indicators as ind
        P, T = len(self.periods), len(self.timeframes)
        bank = torch.empty((market.S, T * P, market.N), dtype=torch.float32, device=market.device)
        bank[:, :P] = rsi_bank(market.close, self.periods)
        for i, k in enumerate(self.timeframes[1:], start=1):
            hi = ind.resample(market, k)
            rows = rsi_bank(hi.close, self.periods)                                        # [S][P][M]
            aligned = ind.align_to_base(rows.view(market.S * P, hi.N), market, k)          # [S * P][N]
            bank[:, i * P:(i + 1) * P] = aligned.view(market.S, P, market.N)
            del hi, rows, aligned
        return bank

    @classmethod
    def from_bank(cls, market: MarketData, bank: torch.Tensor, periods, optimization_goals=None,
                  initial_capital: float = 10000.0, event_cap: int = 0, mode: str = "fused",
                  score_on_advanced: bool = False) -> "PopulationSweep":
        """Sweep over a caller-supplied RSI bank [S][P][N] (e.g. the 'rsi' field of the reference's
        market-data points) instead of one computed from the close prices."""
        self = cls.__new__(cls)
        self._configure(market, [int(p) for p in periods], optimization_goals, initial_capital, event_cap, mode, None,
                        score_on_advanced)
        self.timeframes = (market.bar_minutes,)
        assert bank.is_cuda and bank.dtype == torch.float32 and tuple(bank.shape) == (market.S, len(self.periods), market.N)
        self.bank = bank.contiguous()
        return self

    # -- device-side evaluation (inputs already resident) -------------------
    def evaluate_device(self, indiv_dev: torch.Tensor, order_dev: Optional[torch.Tensor], pop: int,
                        fitness_dev: torch.Tensor, plan: Optional["ChunkPlan"] = None) -> None:
        """Sweep + fitness reduction on the current stream.  With a ChunkPlan the time-chunked kernels
        run first and only lanes whose chunk boundaries failed verification go through the fused kernel."""
        self._inverse = None
        if plan is not None:
            plans = plan if isinstance(plan, (list, tuple)) else [plan]
            self._ensure_buffers(pop)
            self._last_plans = plans
            for pl in plans:
                (self._evaluate_tiled if isinstance(pl, TilePlan) else self._evaluate_chunked)(indiv_dev, pl)
            with torch.cuda.device(self.market.device):
                _lib.call("b200bt_fitness_reduce", self._stats.data_ptr(), pop, self.market.S, fitness_dev.data_ptr(),
                          _lib.current_stream())
            return
        m = self.market
        self._last_plans = []
        self._ensure_buffers(pop)
        with torch.cuda.device(m.device):
            st = _lib.current_stream()
            _lib.call("b200bt_sweep", m.close.data_ptr(), _lib.ld(m.close), self.bank.data_ptr(),
                      _lib.ld(self.bank), self.bank.shape[1], m.S, m.N, indiv_dev.data_ptr(),
                      _lib.ptr(order_dev), pop, C.byref(self.cfg), self._stats.data_ptr(),
                      _lib.ptr(self._events), self.event_cap, st)
            _lib.call("b200bt_fitness_reduce", self._stats.data_ptr(), pop, m.S, fitness_dev.data_ptr(), st)

    def _ensure_buffers(self, pop: int) -> None:
        m = self.market
        if self._stats is None or self._pop != pop:
            self._stats = torch.empty((pop, m.S, _lib.LANE_STATS_WORDS), dtype=torch.float64, device=m.device)
            self._events = (torch.zeros((pop, m.S, self.event_cap), dtype=torch.int32, device=m.device)
                            if self.event_cap else None)
            self._pop = pop

    def _evaluate_chunked(self, indiv_dev, plan: "ChunkPlan") -> None:
        """One slice [plan.lo, plan.lo + plan.pop) of the population through the chunked kernels; lanes whose
        chunk boundaries failed verification are re-evaluated by the fused kernel."""
        m = self.market
        lo, n = plan.lo, plan.pop
        stats = self._stats[lo:lo + n]
        events = self._events[lo:lo + n] if self._events is not None else None
        with torch.cuda.device(m.device):
            st = _lib.current_stream()
            _lib.call("b200bt_sweep_chunked", m.close.data_ptr(), _lib.ld(m.close), self.bank.data_ptr(), _lib.ld(self.bank),
                      self.bank.shape[1], m.S, m.N, indiv_dev.data_ptr() + lo * C.sizeof(_lib.Individual),
                      plan.order_dev.data_ptr(), n,
                      plan.items.data_ptr(), plan.n_seg, plan.seg_base_dev.data_ptr(), plan.n_chunks_dev.data_ptr(),
                      plan.n_seg, plan.warm, plan.max_repair_rounds, plan.pool_blocks, plan.workspace.data_ptr(), plan.workspace.numel(),
                      C.byref(self.cfg), stats.data_ptr(), _lib.ptr(events), self.event_cap,
                      plan.invalid.data_ptr(), plan.overflow.data_ptr(), st)

    def _evaluate_tiled(self, indiv_dev, plan: "TilePlan") -> None:
        """One slice of the population through the thread-per-lane kernels (same verification / fallback)."""
        m = self.market
        lo, n = plan.lo, plan.pop
        stats = self._stats[lo:lo + n]
        events = self._events[lo:lo + n] if self._events is not None else None
        with torch.cuda.device(m.device):
            st = _lib.current_stream()
            _lib.call("b200bt_sweep_tiled", m.close.data_ptr(), _lib.ld(m.close), self.bank.data_ptr(), _lib.ld(self.bank),
                      self.bank.shape[1], m.S, m.N, _lib.ptr(self._zones_if_amortised()),
                      indiv_dev.data_ptr() + lo * C.sizeof(_lib.Individual),
                      plan.slots_dev.data_ptr(), len(plan.slots), plan.slots_dev.data_ptr() + 4 * len(plan.slots), n, plan.K, plan.warm,
                      plan.max_repair_rounds, plan.pool_blocks,
                      plan.workspace.data_ptr(), plan.workspace.numel(), C.byref(self.cfg), stats.data_ptr(),
                      _lib.ptr(events), self.event_cap, plan.invalid.data_ptr(), plan.overflow.data_ptr(), st)

    # Lanes the time-chunked kernels flagged (a boundary still inconsistent after the repair passes, a full event pool, a warp
    # not packed for the thread-per-lane scan) are re-evaluated by the fused kernel ON THE DEVICE, inside b200bt_sweep_chunked /
    # b200bt_sweep_tiled: an evaluation reads nothing back.  These two look at the flags of the last evaluation afterwards.
    def _sync_flags(self):
        torch.cuda.current_stream(self.market.device).synchronize()
        return [pl.overflow for pl in (getattr(self, "_last_plans", None) or [])]

    @property
    def last_invalid_lanes(self) -> int:
        """(individual, symbol) lanes of the last evaluation that went through the exact fallback."""
        return int(sum(int(f[1]) for f in self._sync_flags()))

    @property
    def last_scan_stalls(self) -> int:
        """Tiles of the last thread-per-lane scan whose bulk copy did not complete in time (their chunks were re-scanned by the
        repair pass or their lanes re-run by the exact fallback; 0 in normal operation)."""
        return int(sum(int(f[3]) for f in self._sync_flags()))

    @property
    def last_pool_overflow(self) -> bool:
        """The event pool of the last evaluation was too small (its lanes were re-run exactly; the next plan is larger)."""
        return any(bool(f[0]) for f in self._sync_flags())

    def set_gap(self, gap_bar: int, gap_minutes: int) -> None:
        """Declare the series as two pieces glued at `gap_bar`, the second one `gap_minutes` later on the calendar
        (training folds of cross_validate_strategy): only the daily buckets of the metrics see it."""
        self.cfg.gap_bar, self.cfg.gap_minutes = int(gap_bar), int(gap_minutes)

    def zone_map(self) -> torch.Tensor:
        """(min, max) per 32-bar block of the price rows and of the RSI bank (b200bt_zone_map), built on first use."""
        if getattr(self, "_zones", None) is None:
            m = self.market
            n = int(_lib.load().b200bt_zone_map_floats(self.bank.shape[1], m.S, m.N))
            z = torch.empty(n, dtype=torch.float32, device=m.device)
            with torch.cuda.device(m.device):
                _lib.call("b200bt_zone_map", m.close.data_ptr(), _lib.ld(m.close), self.bank.data_ptr(), _lib.ld(self.bank),
                          self.bank.shape[1], m.S, m.N, z.data_ptr(), _lib.current_stream())
            self._zones = z
        return self._zones

    use_zones = True

    def _zones_if_amortised(self) -> Optional[torch.Tensor]:
        """The zone map costs about as much as it saves in ONE sweep (0.8 ms against ~0.2 ms at C2): it is built
        when this bank is swept a second time (a GA sweeps it every generation), not for a one-off evaluation."""
        self._tiled_sweeps = getattr(self, "_tiled_sweeps", 0) + 1
        if not self.use_zones or (self._tiled_sweeps < 2 and getattr(self, "_zones", None) is None):
            return None
        return self.zone_map()

    def plan(self, population: List[Dict], pred: Optional[np.ndarray] = None, rows: Optional[np.ndarray] = None) -> Optional[List]:
        """The kernel path `evaluate` takes for this population under self.mode: None = fused kernel, else the
        list of TilePlan / ChunkPlan slices to pass to evaluate_device(plan=...).  `pred`: predicted_events of the
        population when the caller already has it (evaluate derives it from the decoded records)."""
        long_enough = self.market.N >= self.chunk_min_bars
        tiled = self.mode == "tiled"
        if self.mode == "auto" and long_enough:
            # thread-per-lane needs many machines: enough chunks per lane, or enough lanes (tools/mode_crossover.py:
            # at 200k bars the warp-per-chunk path is faster below ~2000 individuals x 10 symbols)
            k = TilePlan.chunks_for(len(population), self.market.N, self.market.S, self.market.device,
                                    self.chunk_options.get("warm", TilePlan.WARM), self.chunk_options.get("max_chunks", 64))
            tiled = k >= 16 or len(population) * self.market.S * k >= 100_000
        if not (tiled or self.mode == "chunked" or (self.mode == "auto" and long_enough)):
            return None
        options = dict(self.chunk_options)
        if not tiled and self.mode == "auto":
            options.setdefault("target_events", 8192)
        # Event-pool sizing learns from the previous sweep of this bank: the cost model behind `pred` is calibrated on random
        # populations, while the populations a GA evolves write several times more records.  The pool is scaled by the
        # measured blocks-per-predicted-block ratio (never below the model), and by 4x more whenever it still overflowed.
        if getattr(self, "_last_plans", None):
            flags = self._sync_flags()
            used = sum(int(f[2]) - 2 * pl.n_seg * self.market.S for f, pl in zip(flags, self._last_plans))
            predicted = sum(pl.pred_blocks for pl in self._last_plans)
            if any(bool(f[0]) for f in flags):
                self._pool_factor = 4.0 * max(getattr(self, "_pool_factor", 1.0), 1.0)
                options.pop("pool_blocks", None)
            elif predicted > 0:
                self._pool_factor = max(1.0, 1.2 * used / predicted)
        if getattr(self, "_pool_factor", 1.0) > 1.0:
            options["pool_scale"] = getattr(self, "_pool_factor") * options.get("pool_scale", 1.5)
        if tiled and rows is None and len(self.timeframes) > 1:
            rows = decode_population(population, self.period_row, len(self.timeframes))["rsi_row"]
        return self.plan_batches(population, tiled=tiled, pred=pred, rows=rows, **options)

    def plan_tiles(self, population: List[Dict], **kw) -> "TilePlan":
        return TilePlan(population, self.market.N, self.market.S, self.market.device, **kw)

    def plan_chunks(self, population: List[Dict], **kw) -> "ChunkPlan":
        return ChunkPlan(population, self.market.N, self.market.S, self.market.device, **kw)

    def plan_batches(self, population: List[Dict], max_pool_bytes: int = 8 << 30, tiled: bool = False,
                     pred: Optional[np.ndarray] = None, rows: Optional[np.ndarray] = None, **kw) -> List:
        """Plans for contiguous slices of the population whose event pools each stay below `max_pool_bytes`
        and share one workspace: large populations (BASELINE configs[4]: 10 000 x 50 symbols) record more
        events than fit in HBM at once, so they go through the chunked kernels slice by slice."""
        cls = TilePlan if tiled else ChunkPlan
        accepted = inspect.signature(cls.__init__).parameters     # chunk_options may carry the other path's knobs
        kw = {k: v for k, v in kw.items() if k in accepted}
        if pred is None:
            pred = predicted_events(population, self.market.N)
        rows_of = (lambda lo, hi: {"rows": None if rows is None else rows[lo:hi]}) if tiled else (lambda lo, hi: {})
        if kw.get("pool_blocks") is not None:
            return [cls(population, self.market.N, self.market.S, self.market.device, pred=pred, **rows_of(0, None), **kw)]
        pool_bytes = pred * (self.market.S * 8 * kw.get("pool_scale", 1.5))
        if float(pool_bytes.sum()) <= max_pool_bytes:
            return [cls(population, self.market.N, self.market.S, self.market.device, pred=pred, **rows_of(0, None), **kw)]
        cuts, acc = [0], 0.0
        for i, b in enumerate(pool_bytes):
            if acc + b > max_pool_bytes and i > cuts[-1]:
                cuts.append(i)
                acc = 0.0
            acc += b
        cuts.append(len(population))
        plans = [cls(population[lo:hi], self.market.N, self.market.S, self.market.device, lo=lo, workspace=DEFERRED,
                     pred=pred[lo:hi], **rows_of(lo, hi), **kw) for lo, hi in zip(cuts[:-1], cuts[1:])]
        shared = torch.empty(max(pl.ws_bytes for pl in plans), dtype=torch.uint8, device=self.market.device)
        for pl in plans:
            pl.workspace = shared        # the slices run one after the other on the same stream
        return sorted(plans, key=lambda pl: pl.lo)

    # -- host-facing evaluation --------------------------------------------
    def evaluate(self, population: List[Dict]) -> np.ndarray:
        """fitness (float64[pop]) of a list of parameter dicts; H2D of the decoded
        population and D2H of the fitness vector happen inside this call."""
        if not population:
            return np.zeros(0, dtype=np.float64)
        dev = self.market.device
        packed = decode_population(population, self.period_row, len(self.timeframes))
        # individuals that decode to the same kernel parameters (the reference rule reads 6 of the 18 genes,
        # and elitism / crossover copy individuals) are evaluated once
        expand = None
        dup = _duplicate_classes(packed)
        if dup is not None:
            first, inverse = dup
            keep = np.sort(first)                       # unique individuals in population order
            rank = np.empty(len(first), dtype=np.int64)
            rank[np.argsort(first)] = np.arange(len(first))
            expand = rank[inverse.reshape(-1)]
            packed = np.ascontiguousarray(packed[keep])
            population = [population[i] for i in keep]
        self.last_unique = len(population)
        pop = len(population)
        pred = EVENTS_PER_COST_BAR * costs_from_packed(packed, self.periods, self.timeframes) * self.market.N
        plan = self.plan(population, pred=pred, rows=packed["rsi_row"])
        if plan is None:       # the fused kernel dispatches in this order: same RSI period adjacent, most expensive first
            order = np.lexsort((np.arange(pop), -pred, packed["rsi_row"])).astype(np.int32)
        else:
            order = np.zeros(0, dtype=np.int32)
        nbytes = packed.nbytes
        if self._pinned_in is None or self._pinned_in.numel() < nbytes + order.nbytes:
            self._pinned_in = torch.empty(nbytes + order.nbytes, dtype=torch.uint8, pin_memory=True)
        if self._pinned_out is None or self._pinned_out.numel() < pop:
            self._pinned_out = torch.empty(pop, dtype=torch.float64, pin_memory=True)
        hin = self._pinned_in.numpy()
        hin[:nbytes] = packed.view(np.uint8)
        hin[nbytes:nbytes + order.nbytes] = order.view(np.uint8)
        staged = self._pinned_in[:nbytes + order.nbytes].to(dev, non_blocking=True)
        indiv_dev = staged[:nbytes]
        order_dev = staged[nbytes:].view(torch.int32) if order.size else None
        fit = torch.empty(pop, dtype=torch.float64, device=dev)
        self.evaluate_device(indiv_dev, order_dev, pop, fit, plan=plan)
        self._inverse = expand
        out = self._pinned_out[:pop]
        out.copy_(fit, non_blocking=True)
        torch.cuda.current_stream(dev).synchronize()
        self.h2d_bytes = nbytes + order.nbytes
        self.d2h_bytes = pop * 8
        res = out.numpy().copy()
        return res if self._inverse is None else res[self._inverse]

    def lane_stats(self) -> Dict[str, np.ndarray]:
        """Per-lane metrics of the last evaluation: dict field -> [pop][S] array."""
        raw = self._stats.cpu().numpy()
        if getattr(self, "_inverse", None) is not None:
            raw = raw[self._inverse]
        out = {name: raw[:, :, i] for i, name in enumerate(_lib.LANE_STATS_FIELDS[:-1])}
        out["trade_hash"] = np.ascontiguousarray(raw[:, :, _lib.LANE_STATS_WORDS - 1]).view(np.uint64)
        return out

    def advanced_stats(self) -> Dict[str, np.ndarray]:
        """calculate_advanced_metrics (strategy_evaluation.py:231-319) for every lane of the last evaluation,
        [pop][S] arrays: the Sortino ingredients come out of the kernels' daily buckets, the rest is arithmetic on
        the lane stats (same expressions as the reference, including its fixed 10 000 in the recovery factor)."""
        st = self.lane_stats()
        with np.errstate(divide="ignore", invalid="ignore"):
            dd, net, n = st["max_drawdown"], st["net_profit"], st["n_records"]
            ret_pct = net / self.cfg.initial_capital * 100
            avg_p = np.where(st["n_wins"] > 0, st["total_profit"] / st["n_wins"], 0.0)
            avg_l = np.where(st["n_losses"] > 0, st["total_loss"] / st["n_losses"], 0.0)
            return {
                "calmar_ratio": np.where(dd > 0, (ret_pct / 100) / dd, np.inf),
                "sortino_ratio": st["sortino_ratio"],
                "recovery_factor": np.where(dd > 0, net / (dd * 10000), np.inf),
                "expectancy": np.where(n > 0, st["win_rate"] * avg_p - (1 - st["win_rate"]) * np.abs(avg_l), 0.0),
                "profit_per_day": st["mean_daily_pnl"],
            }

    def events(self) -> Optional[np.ndarray]:
        """First `event_cap` event words per lane, uint32 [pop][S][cap] (see B200BT_EVENT_*)."""
        if self._events is None:
            return None
        ev = self._events.cpu().numpy().view(np.uint32)
        return ev if getattr(self, "_inverse", None) is None else ev[self._inverse]

    @property
    def fitness_function(self):
        sweep = self

        def fitness(individual: Dict) -> float:
            return float(sweep.evaluate([individual])[0])

        fitness.batch = lambda population: [float(x) for x in sweep.evaluate(population)]
        return fitness
