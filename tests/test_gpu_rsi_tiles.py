"""The RSI bank and its zone map at the seams of the kernels' time tiles, against plain references.

rsi_bank_kernel writes 4096-bar tiles, the analyzer's RSI column 2048-bar tiles.  Random walks never hold the state a tile
inherits at its first bar far from a fresh start; runs of equal closes and runs of closes moving one way do.  RSI is the
ratio U / (U + D) of two Wilder averages, and a ratio does not forget its past when both terms shrink, so the bank must
carry the exact state across every seam.  The zone map (per 32-bar block and 4-bar group (min, max) of the price and bank
rows) is checked against a plain NumPy restatement of its layout, bit for bit, and the population sweep against the C
oracle fed the float64 bank on the inputs where a wrong bank or a wrong zone changes trades.
"""
import warnings

import numpy as np
import pandas as pd
import pytest

TILE = 4096          # bars per CTA of rsi_bank_kernel
AN_TILE = 2048       # bars per CTA of the analyzer kernels
ZONE_N = [1, 4, 31, 32, 33, 127, 128, 129, 4095, 4096, 4097, 262_177]
BANK_PERIODS = [1, 2, 5, 14, 30]
TINY = np.finfo(np.float64).tiny          # smallest normal float64


# ------------------------------------------------------------------------------------------------------------------
# plain references
# ------------------------------------------------------------------------------------------------------------------
def zone_strides(n):
    """(coarse, fine) row strides in float2 entries: whole 32-bar blocks rounded up to an even count, whole 128-bar
    tiles of 4-bar groups."""
    return ((n + 31) // 32 + 1) & ~1, ((n + 127) // 128) * 32


def _ranges(rows, width, stride):
    """rows [R][n] float32 -> [R][stride][2]: (min, max) of every `width`-bar group ignoring NaN (as fminf / fmaxf do),
    (NaN, NaN) for a group without a number and past the data."""
    R, n = rows.shape
    g = (n + width - 1) // width
    pad = np.full((R, g * width), np.nan, dtype=np.float32)
    pad[:, :n] = rows
    out = np.full((R, stride, 2), np.nan, dtype=np.float32)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore", RuntimeWarning)       # all-NaN groups
        out[:, :g, 0] = np.nanmin(pad.reshape(R, g, width), axis=2)
        out[:, :g, 1] = np.nanmax(pad.reshape(R, g, width), axis=2)
    return out


def zone_map_ref(price, bank):
    """price [S][N], bank [S][P][N] float32 -> the flat float32 zone map: coarse [S][P + 1][coarse stride] (min, max),
    then fine [S][P + 1][fine stride] (min, max); row 0 of every symbol is the price."""
    price, bank = np.asarray(price, dtype=np.float32), np.asarray(bank, dtype=np.float32)
    S, P, n = bank.shape
    zs, fs = zone_strides(n)
    rows = np.concatenate([price[:, None, :], bank], axis=1).reshape(S * (P + 1), n)
    return np.concatenate([_ranges(rows, 32, zs).ravel(), _ranges(rows, 4, fs).ravel()])


def _same_bits(got, want):
    got, want = np.asarray(got), np.asarray(want)
    assert got.shape == want.shape
    nan = np.isnan(want)
    bad = np.flatnonzero((np.isnan(got) != nan) | (~nan & (got != want)))
    return bad


def wilder_states(close32, w):
    """The oracle's two Wilder averages (U, D) of one fp32 close row, float64, no min_periods."""
    c = pd.Series(np.asarray(close32, dtype=np.float64))
    diff = c.diff(1)
    up = diff.where(diff > 0, 0.0)
    dn = -diff.where(diff < 0, 0.0)
    return (up.ewm(alpha=1 / w, adjust=False).mean().to_numpy(), dn.ewm(alpha=1 / w, adjust=False).mean().to_numpy())


def check_rsi_rows(got, close32, periods, name, fill=True):
    """got [P][N] against indicators_ref.rsi_bank, the bank's contract: at most a 2e-6 fraction of double-rounding ties,
    rtol 2e-7, atol 0, on every bar where the oracle's averages are normal numbers or zero; 100 wherever the oracle's D is
    exactly 0.  Bars where the oracle's U or D is subnormal (thousands of equal closes) carry no digits to compare and are
    left out; returns how many were, per period.

    The reference evaluates RSI as 100 - 100 / (1 + U / D).  Near 0 (a one-way run decays U to 1e-16 of D) that form
    resolves the value only to ~2.5e-14 absolute -- 1 + U / D rounds to 1 + k 2^-52 -- which is coarser than an fp32 ulp
    below RSI ~1e-6 and flips the fp32 rounding now and then up to ~1e-4.  On the bars where it rounds differently from the
    same float64 averages evaluated as 100 U / (U + D) (correct to a few float64 ulps), the latter is the reference."""
    from oracle import indicators_ref
    want = indicators_ref.rsi_bank(close32, periods, fill=fill)
    excluded, bad_total, size = [], 0, 0
    t = np.arange(len(close32))
    for i, w in enumerate(periods):
        U, D = wilder_states(close32, w)
        with np.errstate(all="ignore"):
            literal = np.where(D == 0, 100, 100 - (100 / (1 + U / D))).astype(np.float32)
            precise = np.where(D == 0, 100, 100.0 * U / (U + D)).astype(np.float32)
        ref = want[i].copy()
        defined = t >= w - 1
        assert np.array_equal(literal[defined], ref[defined], equal_nan=True), (name, w)   # the oracle's own arithmetic
        unresolved = defined & (literal != precise)
        ref[unresolved] = precise[unresolved]
        if fill and unresolved[min(w - 1, len(ref) - 1)]:
            ref[:w - 1] = precise[w - 1]                                                      # (its back-fill)
        sub = ((U > 0) & (U < TINY)) | ((D > 0) & (D < TINY))
        keep = ~sub
        excluded.append(int(sub.sum()))
        g, r = got[i][keep], ref[keep]
        assert np.array_equal(np.isnan(g), np.isnan(r)), (name, w, np.flatnonzero(np.isnan(g) != np.isnan(r))[:5])
        zero_d = (D == 0) & defined
        assert (got[i][zero_d] == 100.0).all(), (name, w, np.flatnonzero(got[i][zero_d] != 100.0)[:5])
        m = ~np.isnan(r)
        neq = np.flatnonzero(g[m] != r[m])
        bad_total += len(neq)
        size += int(m.sum())
        np.testing.assert_allclose(g[m], r[m], rtol=2e-7, atol=0,
                                   err_msg=f"{name} w={w}: first differing kept bars {np.flatnonzero(keep)[m][neq[:5]]}")
    assert bad_total <= int(2e-6 * size), (name, bad_total)
    return excluded


# ------------------------------------------------------------------------------------------------------------------
# inputs
# ------------------------------------------------------------------------------------------------------------------
def _walk(n, s=1):
    from ai_crypto_trader_b200 import synth
    return synth.synth_ohlcv(1, n, first_symbol=s)[3, 0].copy()


def _with_run(c, lo, hi, kind, step_ulps=3):
    """closes [lo, hi) made equal to close[lo - 1] ('flat') or moving by `step_ulps` fp32 ulps per bar ('up' / 'down');
    the series after the run continues from where the run ended."""
    c = c.copy()
    x = c[lo - 1]
    direction = {"flat": 0.0, "up": np.inf, "down": -np.inf}[kind]
    for t in range(lo, hi):
        for _ in range(step_ulps if kind != "flat" else 0):
            x = np.nextafter(x, np.float32(direction))
        c[t] = x
    if hi < len(c):
        c[hi:] = (c[hi:].astype(np.float64) - float(c[hi]) + float(c[hi - 1]) * 1.0001).astype(np.float32)
    return c


def _edge_case(name):
    """-> (closes [3][N] float32 with the run on the middle symbol only, periods, run length)."""
    L = 1400                                   # longer than the old warm-up halo of every period up to 30 (1248 bars)
    cases = {
        "flat_ends_before_seam": (TILE - 1 - L, TILE - 1, "flat", 2 * TILE + 77),
        "flat_ends_at_seam": (TILE - L, TILE, "flat", 2 * TILE + 77),
        "flat_ends_after_seam": (TILE - L, TILE + 300, "flat", 2 * TILE + 77),
        "flat_crosses_seam_ends_at_next": (TILE - L, 2 * TILE, "flat", 2 * TILE + 5),
        "up_run_crosses_seam": (TILE - L, TILE + 300, "up", 2 * TILE + 77),
        "down_run_crosses_seam": (TILE - L, TILE + 300, "down", 2 * TILE + 77),
        "flat_spans_three_tiles": (TILE - L, 3 * TILE + 100, "flat", 4 * TILE + 33),
        "down_spans_three_tiles": (TILE - L, 3 * TILE + 100, "down", 4 * TILE + 33),
        "flat_long_period": (1000, 1000 + 45_000, "flat", 12 * TILE + 3),
    }
    lo, hi, kind, n = cases[name]
    periods = BANK_PERIODS + ([1000] if name == "flat_long_period" else [])
    rows = np.stack([_walk(n, 2), _with_run(_walk(n, 1), lo, hi, kind), _walk(n, 3)])
    return rows, periods, hi - lo


EDGE_CASES = ["flat_ends_before_seam", "flat_ends_at_seam", "flat_ends_after_seam", "flat_crosses_seam_ends_at_next",
              "up_run_crosses_seam", "down_run_crosses_seam", "flat_spans_three_tiles", "down_spans_three_tiles",
              "flat_long_period"]


def _falling_with_upticks(n, upticks, ulps=2):
    """fp32 closes falling by `ulps` ulps every bar, one up-tick of 3 ulps at each bar of `upticks`: RSI(1) is 0 on every
    bar but those (and bar 0, which has no move: 100)."""
    c = np.empty(n, dtype=np.float32)
    x = np.float32(100.0)
    for t in range(n):
        if t in upticks:
            for _ in range(3):
                x = np.nextafter(x, np.float32(np.inf))
        elif t:
            for _ in range(ulps):
                x = np.nextafter(x, np.float32(-np.inf))
        c[t] = x
    return c


def _zone_closes(n):
    """[3][n]: a random walk, falling closes with isolated up-ticks next to the tile starts and at the last bar, and a
    flat run across the first seam."""
    a = _walk(n, 4)
    b = _falling_with_upticks(n, {t for t in (5, 60, TILE + 4, TILE + 61, 2 * TILE + 30, n - 1) if 0 < t < n})
    c = _with_run(_walk(n, 5), min(n - 1, 2600), min(n, TILE + 500), "flat") if n > 1 else _walk(n, 5)
    return np.stack([a, b, c])


# ------------------------------------------------------------------------------------------------------------------
# host-only
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n", ZONE_N)
def test_zone_map_reference_has_the_library_size(native_lib, n):
    for P, S in ((1, 1), (3, 2), (5, 3)):
        z = zone_map_ref(np.zeros((S, n), np.float32), np.zeros((S, P, n), np.float32))
        assert z.size == int(native_lib.b200bt_zone_map_floats(P, S, n)), (P, S, n)


def test_zone_map_reference_on_a_hand_example():
    price = np.arange(37, dtype=np.float32)[None]
    bank = np.full((1, 1, 37), np.nan, np.float32)
    bank[0, 0, 33] = 5.0
    z = zone_map_ref(price, bank)
    zs, fs = zone_strides(37)
    assert (zs, fs) == (2, 32)
    coarse = z[:2 * 2 * zs].reshape(2, zs, 2)
    fine = z[2 * 2 * zs:].reshape(2, fs, 2)
    assert coarse[0].tolist() == [[0, 31], [32, 36]]
    assert np.isnan(coarse[1, 0]).all() and coarse[1, 1].tolist() == [5, 5]
    assert fine[0, 9].tolist() == [36, 36] and np.isnan(fine[0, 10:]).all()
    assert np.isnan(fine[1, 7]).all() and fine[1, 8].tolist() == [5, 5]


# ------------------------------------------------------------------------------------------------------------------
# GPU
# ------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def cuda(native_lib):
    import torch
    assert torch.cuda.is_available(), "gpu-marked tests need a CUDA device"
    torch.cuda.set_device(0)
    return torch


def _zone_map_kernel(torch, close, bank):
    from ai_crypto_trader_b200 import _lib
    S, P, n = bank.shape
    z = torch.full((int(_lib.load().b200bt_zone_map_floats(P, S, n)),), 7.0, dtype=torch.float32, device="cuda")
    _lib.call("b200bt_zone_map", close.data_ptr(), _lib.ld(close), bank.data_ptr(), _lib.ld(bank), P, S, n, z.data_ptr(),
              _lib.current_stream())
    return z.cpu().numpy()


@pytest.mark.gpu
@pytest.mark.parametrize("periods", [[1], [1, 2, 14], [2, 5, 14, 30, 47]], ids=["w1", "w1_2_14", "w2_to_47"])
@pytest.mark.parametrize("n", ZONE_N)
def test_both_zone_writers_equal_the_plain_zone_map(cuda, n, periods):
    """b200bt_rsi_bank_zones (written in two symbol sub-ranges, as the upload pipeline does) and b200bt_zone_map, bit for
    bit against the NumPy zone map of the bank they describe, padding included."""
    torch = cuda
    from ai_crypto_trader_b200 import _lib
    from ai_crypto_trader_b200.sweep import rsi_bank
    closes = _zone_closes(n)
    S, P = closes.shape[0], len(periods)
    close = torch.from_numpy(closes).cuda()
    fused = torch.full((int(_lib.load().b200bt_zone_map_floats(P, S, n)),), 7.0, dtype=torch.float32, device="cuda")
    bank = torch.empty((S, P, n), dtype=torch.float32, device="cuda")
    rsi_bank(close[:1], periods, out=bank[:1], zones=fused, zones_symbols=S, first_symbol=0)
    rsi_bank(close[1:], periods, out=bank[1:], zones=fused, zones_symbols=S, first_symbol=1)
    assert torch.equal(bank, rsi_bank(close, periods))
    want = zone_map_ref(closes, bank.cpu().numpy())
    bad = _same_bits(fused.cpu().numpy(), want)
    assert bad.size == 0, ("rsi_bank_zones", bad[:8])
    bad = _same_bits(_zone_map_kernel(torch, close, bank), want)
    assert bad.size == 0, ("zone_map", bad[:8])


@pytest.mark.gpu
def test_sweep_zone_map_of_a_multi_timeframe_bank(cuda):
    """PopulationSweep.zone_map() over a 1m / 5m / 15m bank, whose higher-timeframe rows start with NaN."""
    from ai_crypto_trader_b200 import synth
    from ai_crypto_trader_b200.sweep import MarketData, PopulationSweep
    n = 3 * TILE + 45
    ohlcv = synth.synth_ohlcv(2, n, first_symbol=2)
    ohlcv[3, 1] = _falling_with_upticks(n, {7, TILE + 4, 2 * TILE + 100})
    market = MarketData(ohlcv, minute0=synth.EPOCH_2024_MINUTES + 7)
    sweep = PopulationSweep(market, rsi_periods=[1, 2, 14], timeframes=(1, 5, 15), mode="tiled")
    bank = sweep.bank.cpu().numpy()
    assert np.isnan(bank[:, 3:, 0]).all() and not np.isnan(bank[:, :3]).any()
    bad = _same_bits(sweep.zone_map().cpu().numpy(), zone_map_ref(ohlcv[3], bank))
    assert bad.size == 0, bad[:8]


@pytest.mark.gpu
@pytest.mark.parametrize("case", EDGE_CASES)
def test_rsi_bank_at_tile_seams_vs_float64_oracle(cuda, case):
    """b200bt_rsi_bank and b200bt_rsi_bank_zones on runs of equal closes and of one-way moves that cross 4096-bar
    seams, against indicators_ref.rsi_bank."""
    torch = cuda
    from ai_crypto_trader_b200 import _lib
    from ai_crypto_trader_b200.sweep import rsi_bank
    closes, periods, run = _edge_case(case)
    S, n = closes.shape
    close = torch.from_numpy(closes).cuda()
    got = rsi_bank(close, periods).cpu().numpy()
    zones = torch.empty(int(_lib.load().b200bt_zone_map_floats(len(periods), S, n)), dtype=torch.float32, device="cuda")
    got_z = rsi_bank(close, periods, zones=zones, zones_symbols=S).cpu().numpy()
    assert np.array_equal(got, got_z, equal_nan=True)
    assert _same_bits(zones.cpu().numpy(), zone_map_ref(closes, got)).size == 0
    nofill = rsi_bank(close, periods, fill=False).cpu().numpy()
    for s in range(S):
        excluded = check_rsi_rows(got[s], closes[s], periods, f"{case} symbol {s}")
        assert check_rsi_rows(nofill[s], closes[s], periods, f"{case} symbol {s} (no fill)", fill=False) == excluded
        ex = dict(zip(periods, excluded))
        if s != 1:
            assert not any(excluded), (case, s, ex)          # random walks never leave the normal numbers
        else:
            # RSI(1) is exact and RSI(1000) decays slowly; RSI(2) passes through the subnormals to exactly 0 on every
            # run (about 55 bars of them), the longer periods stay there only on runs long enough to get there
            assert ex[1] == 0 and ex.get(1000, 0) == 0 and 0 < ex[2] < 100, (case, ex)
            assert all(e <= run for e in excluded), (case, ex)
            if case == "flat_long_period":
                assert all(e > 20_000 for w, e in ex.items() if w in (5, 14, 30)), ex


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["flat_ends_after_seam", "down_run_crosses_seam", "flat_spans_three_tiles",
                                  "down_spans_three_tiles"])
@pytest.mark.parametrize("shift", [0, AN_TILE])
def test_analyzer_rsi_column_at_tile_seams(cuda, case, shift):
    """TechnicalAnalyzer's rsi column (2048-bar tiles) on the same runs, shifted so that they also cross the seams at odd
    multiples of 2048, against indicators_ref.rsi with the analyzer's NaN policy."""
    from ai_crypto_trader_b200.indicators import TechnicalAnalyzer
    from ai_crypto_trader_b200.sweep import MarketData
    closes, _, run = _edge_case(case)
    closes = np.ascontiguousarray(closes[:, shift:])
    S, n = closes.shape
    ohlcv = np.empty((5, S, n), dtype=np.float32)
    ohlcv[0:4] = closes[None]
    ohlcv[4] = 1.0
    ta = TechnicalAnalyzer(MarketData(ohlcv))
    got = ta.data["rsi"].cpu().numpy()
    for s in range(S):
        excluded = check_rsi_rows(got[s][None], closes[s], [14], f"{case}+{shift} symbol {s}")[0]
        assert excluded == 0 if s != 1 else excluded <= run, (case, s, excluded)


# ------------------------------------------------------------------------------------------------------------------
# sweeps
# ------------------------------------------------------------------------------------------------------------------
SWEEPS = [("fused", {}), ("tiled", dict(chunks=1)), ("tiled", dict(chunks=4, warm=512))]


def _sweep_vs_oracle(ohlcv, periods, population, cap=64):
    """Every sweep path against sim_oracle.lane fed the float64 bank; tiled sweeps run twice (the second one through the
    zone map).  -> the oracle's events per (individual, symbol)."""
    from ai_crypto_trader_b200.sweep import MarketData, PopulationSweep
    from oracle import indicators_ref, sim_oracle
    market = MarketData(ohlcv)
    S = ohlcv.shape[1]
    cfg = sim_oracle.config_of(market.minute0, 1)
    want = {}
    for s in range(S):
        bank = indicators_ref.rsi_bank(ohlcv[3, s], sorted(set(periods)))
        row = {w: i for i, w in enumerate(sorted(set(periods)))}
        for i, p in enumerate(population):
            want[i, s] = sim_oracle.lane(ohlcv[3, s], bank[row[p["rsi_period"]]], p, cfg, event_cap=cap)
    for mode, opts in SWEEPS:
        sweep = PopulationSweep(market, rsi_periods=periods, mode=mode, chunk_options=opts, event_cap=cap)
        for rnd in range(1 if mode == "fused" else 2):
            sweep.evaluate(population)
            stats, events = sweep.lane_stats(), sweep.events()
            for (i, s), (st, ev, _) in want.items():
                where = (mode, opts, rnd, i, s)
                assert int(stats["n_records"][i, s]) == int(st["n_records"]), where
                assert int(stats["trade_hash"][i, s]) == int(st["trade_hash"]), where
                assert np.array_equal(events[i, s, :len(ev)], ev), where
                assert stats["score"][i, s] == pytest.approx(float(st["score"]), rel=1e-9, abs=1e-11) or \
                    (np.isnan(stats["score"][i, s]) and np.isnan(st["score"])), where
    return {k: v[1] for k, v in want.items()}


@pytest.mark.gpu
def test_sweep_rsi1_exit_next_to_a_tile_start(cuda):
    """RSI(1) of closes falling by fp32 ulps is 0 except at one up-tick, 4 bars after the seam: a long position opened
    on RSI 0 must exit there.  The zone of that 32-bar block must hold the 100."""
    from ai_crypto_trader_b200 import _lib, synth
    n = 2 * TILE + 33
    ohlcv = synth.synth_ohlcv(1, n, first_symbol=1)
    ohlcv[3, 0] = _falling_with_upticks(n, {TILE + 4})
    population = synth.random_population(4, seed=11)
    for p, (lo, hi) in zip(population, [(30, 70), (20, 80), (50, 60), (5, 95)]):
        p.update(rsi_period=1, rsi_oversold=lo, rsi_overbought=hi, take_profit=10, stop_loss=5)
    ev = _sweep_vs_oracle(ohlcv, [1], population)
    for i in range(len(population)):
        bars = (ev[i, 0] & _lib.EVENT_BAR_MASK).tolist()
        assert TILE + 4 in bars, (i, bars)


@pytest.mark.gpu
def test_sweep_long_position_holds_through_a_flat_run_across_a_seam(cuda):
    """1040 equal closes, the last 300 past the seam: RSI(14) stays where the run started (about 46), so a long position
    opened before the run holds through it; an RSI restarted at the seam would read 100 and exit."""
    from ai_crypto_trader_b200 import _lib, synth
    from oracle import indicators_ref
    n = 2 * TILE + 33
    lo, hi = TILE - 576 - 40, TILE + 300
    ohlcv = synth.synth_ohlcv(1, n, first_symbol=1)
    ohlcv[3, 0] = _with_run(ohlcv[3, 0], lo, hi, "flat")
    r0 = float(indicators_ref.rsi_bank(ohlcv[3, 0], [14])[0][lo])
    assert 30 < r0 < 60, r0
    population = synth.random_population(3, seed=12)
    for p, d in zip(population, (0.5, 2.0, 5.0)):
        p.update(rsi_period=14, rsi_oversold=r0 + d, rsi_overbought=70, take_profit=50, stop_loss=50)
    ev = _sweep_vs_oracle(ohlcv, [14], population, cap=n)
    for i in range(len(population)):
        e = ev[i, 0]
        bars = e & _lib.EVENT_BAR_MASK
        before = e[bars < TILE]
        assert len(before) and not (before[-1] & (_lib.EVENT_EXIT | _lib.EVENT_SELL)), (i, "long across the seam")
        assert not ((bars >= TILE) & (bars < hi)).any(), (i, bars[(bars >= lo) & (bars < hi + 5)])
