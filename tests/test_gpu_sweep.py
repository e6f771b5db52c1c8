"""GPU parity of the indicator bank and the population sweep against the CPU oracle
(and, through the committed fixtures, against the reference's own code)."""
import numpy as np
import pytest

from conftest import unjson

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def torch_cuda(native_lib):
    import torch
    assert torch.cuda.is_available(), "gpu-marked tests need a CUDA device"
    torch.cuda.set_device(0)
    return torch


def _bank_mismatch(got, want):
    neq = got != want
    neq &= ~(np.isnan(got) & np.isnan(want))
    return int(neq.sum())


@pytest.mark.parametrize("n_bars", [1, 3, 29, 30, 31, 127, 128, 4095, 4096, 4097, 10000, 70001])
def test_rsi_bank_bitwise_vs_float64_oracle(torch_cuda, n_bars):
    torch = torch_cuda
    from ai_crypto_trader_b200 import synth
    from ai_crypto_trader_b200.sweep import rsi_bank
    from oracle import indicators_ref
    periods = [2, 5, 14, 30, 47]
    ohlcv = synth.synth_ohlcv(3, n_bars)
    got = rsi_bank(torch.from_numpy(ohlcv[3]).cuda(), periods).cpu().numpy()
    for s in range(3):
        want = indicators_ref.rsi_bank(ohlcv[3, s], periods)
        bad = _bank_mismatch(got[s], want)
        # fp64 evaluation rounded once to fp32: identical up to double-rounding ties (~1e-8 of values)
        assert bad <= max(0, int(2e-6 * want.size)), (n_bars, s, bad)
        np.testing.assert_allclose(got[s], want, rtol=2e-7, atol=0)


def test_rsi_bank_nan_mode_and_flat_series(torch_cuda):
    torch = torch_cuda
    from ai_crypto_trader_b200.sweep import rsi_bank
    from oracle import indicators_ref
    n = 500
    close = np.full((1, n), 123.25, dtype=np.float32)
    close[0, 200:] += np.linspace(0, 5, 300).astype(np.float32)   # flat, then strictly rising
    got = rsi_bank(torch.from_numpy(close).cuda(), [14], fill=False).cpu().numpy()[0]
    want = indicators_ref.rsi_bank(close[0], [14], fill=False)
    assert np.isnan(got[0, :13]).all() and not np.isnan(got[0, 13:]).any()
    assert _bank_mismatch(got, want) == 0
    assert (got[0, 13:200] == 100.0).all()   # no down moves -> 100 (ta: where(emadn == 0, 100, ...))


def test_sweep_matches_reference_fixtures(torch_cuda, sim_golden):
    """The kernel against records produced by the reference's own _simulate_trades /
    calculate_metrics / _calculate_strategy_score: bit-exact bars and sides, float64 metrics."""
    torch = torch_cuda
    from ai_crypto_trader_b200 import _lib
    from ai_crypto_trader_b200.sweep import MarketData, PopulationSweep
    meta, arrays = sim_golden
    syms = sorted({c["symbol"] for c in meta["cases"]})
    n = meta["n_bars"]
    ohlcv = np.zeros((5, len(syms), n), dtype=np.float32)
    for j, s in enumerate(syms):
        ohlcv[3, j] = arrays[f"close_{s}"]
    market = MarketData(ohlcv, minute0=meta["minute0"])
    sweep = PopulationSweep(market, rsi_periods=meta["periods"], optimization_goals=meta["goals"], event_cap=4096)
    # the bank the kernel consumes must be the fixture's bank
    bank = sweep.bank.cpu().numpy()
    names = []
    for c in meta["cases"]:
        if c["name"] not in names:
            names.append(c["name"])
    by_name = {c["name"]: c["params"] for c in meta["cases"]}
    for j, s in enumerate(syms):
        for name in names:
            period = by_name[name].get("rsi_period", 14)
            assert np.array_equal(bank[j, sweep.period_row[period]], arrays[f"rsi_{s}_{period}"]), (s, period)
    population = [dict(by_name[nm]) for nm in names]
    fitness = sweep.evaluate(population)
    stats = sweep.lane_stats()
    advanced = sweep.advanced_stats()
    events = sweep.events()
    for c in meta["cases"]:
        i, j, key = names.index(c["name"]), syms.index(c["symbol"]), c["key"]
        nrec = c["n_records"]
        for name, want in c["advanced"].items():      # the reference's calculate_advanced_metrics (:231-319)
            assert advanced[name][i, j] == pytest.approx(unjson(want), rel=1e-9, abs=1e-12), (key, name)
        assert int(stats["n_records"][i, j]) == nrec, key
        ev = events[i, j, :nrec]
        assert (ev & _lib.EVENT_BAR_MASK).tolist() == arrays[f"bar_{key}"].tolist(), key
        assert ((ev >> 31) == 1).tolist() == arrays[f"sell_{key}"].tolist(), key
        m = c["metrics"]
        for field, ref_name in (("total_profit", "total_profit"), ("total_loss", "total_loss"),
                                ("net_profit", "net_profit"), ("win_rate", "win_rate"),
                                ("max_drawdown", "max_drawdown"), ("sharpe_ratio", "sharpe_ratio"),
                                ("largest_profit", "largest_profit"), ("largest_loss", "largest_loss"),
                                ("profit_factor", "profit_factor")):
            assert stats[field][i, j] == pytest.approx(unjson(m[ref_name]), rel=1e-10, abs=1e-12), (key, field)
        assert stats["score"][i, j] == pytest.approx(unjson(c["score"]), rel=1e-9, abs=1e-12), key
        # equity curve end point: 1e-5 relative is the north-star tolerance; we hold 1e-12
        assert 10000.0 + stats["net_profit"][i, j] == pytest.approx(arrays[f"equity_{key}"][-1], rel=1e-12), key
    want_fit = [np.mean([unjson(c["score"]) for c in meta["cases"] if c["name"] == nm]) for nm in names]
    np.testing.assert_allclose(fitness, want_fit, rtol=1e-9, atol=1e-12)


def test_sweep_other_optimisation_goals_match_reference_scores(torch_cuda, sim_golden):
    """The kernels' score rule under other goal sets (any scalar key as the primary metric, `expectancy` as a secondary
    one, unknown keys) on the plain and on the advanced metrics dict: the reference's own scores (`alt_scores`)."""
    from ai_crypto_trader_b200.sweep import MarketData, PopulationSweep
    meta, arrays = sim_golden
    syms = sorted({c["symbol"] for c in meta["cases"]})
    ohlcv = np.zeros((5, len(syms), meta["n_bars"]), dtype=np.float32)
    for j, s in enumerate(syms):
        ohlcv[3, j] = arrays[f"close_{s}"]
    market = MarketData(ohlcv, minute0=meta["minute0"])
    names = list(dict.fromkeys(c["name"] for c in meta["cases"]))
    by_name = {c["name"]: c["params"] for c in meta["cases"]}
    population = [dict(by_name[nm]) for nm in names]
    for g, alt in enumerate(meta["alt_goals"]):
        sweep = PopulationSweep(market, rsi_periods=meta["periods"], optimization_goals=alt["goals"],
                                score_on_advanced=alt["advanced"])
        sweep.evaluate(population)
        score = sweep.lane_stats()["score"]
        for c in meta["cases"]:
            got, want = score[names.index(c["name"]), syms.index(c["symbol"])], unjson(c["alt_scores"][g])
            assert got == pytest.approx(want, rel=1e-9, abs=1e-12) or (np.isnan(got) and np.isnan(want)), (alt, c["key"], got, want)


@pytest.mark.parametrize("n_bars,pop,n_sym", [(1, 4, 1), (31, 8, 2), (33, 8, 1), (1000, 64, 3), (50001, 96, 2)])
def test_sweep_vs_c_oracle_random_populations(torch_cuda, n_bars, pop, n_sym):
    from ai_crypto_trader_b200 import _lib, synth
    from ai_crypto_trader_b200.sweep import MarketData, PopulationSweep
    from oracle import indicators_ref, sim_oracle
    ohlcv = synth.synth_ohlcv(n_sym, n_bars, first_symbol=5)
    market = MarketData(ohlcv)
    cap = 512
    sweep = PopulationSweep(market, event_cap=cap)
    population = synth.random_population(pop, seed=n_bars)
    # make a few lanes extreme: always in the market / leverage floats
    population[0].update(rsi_oversold=35, rsi_overbought=65, rsi_period=5, take_profit=1, stop_loss=1)
    population[1].update(take_profit=0.5, stop_loss=0.5)
    fitness = sweep.evaluate(population)
    stats, events = sweep.lane_stats(), sweep.events()
    cfg = sim_oracle.config_of(market.minute0, 1)
    scores = np.zeros((pop, n_sym))
    for s in range(n_sym):
        bank = indicators_ref.rsi_bank(ohlcv[3, s], sweep.periods)
        for i, p in enumerate(population):
            want, ev, _ = sim_oracle.lane(ohlcv[3, s], bank[sweep.period_row[p["rsi_period"]]], p, cfg, event_cap=cap)
            assert int(stats["n_records"][i, s]) == int(want["n_records"]), (i, s)
            assert int(stats["trade_hash"][i, s]) == int(want["trade_hash"]), (i, s)
            assert np.array_equal(events[i, s, :len(ev)], ev), (i, s)
            for f in ("n_wins", "n_losses", "n_days", "sum_duration_bars"):
                assert stats[f][i, s] == want[f], (i, s, f)
            for f in ("total_profit", "total_loss", "net_profit", "max_drawdown", "sharpe_ratio", "largest_profit",
                      "largest_loss", "win_rate", "profit_factor", "score", "sortino_ratio", "downside_deviation",
                      "mean_daily_pnl"):
                assert stats[f][i, s] == pytest.approx(float(want[f]), rel=1e-9, abs=1e-11), (i, s, f)
            assert stats["n_negative_days"][i, s] == want["n_negative_days"], (i, s)
            scores[i, s] = want["score"]
    np.testing.assert_allclose(fitness, scores.mean(axis=1), rtol=1e-9, atol=1e-11)


def test_simulate_trades_dropin_returns_reference_records(torch_cuda, sim_golden):
    """StrategyEvaluationSystem._simulate_trades (reference signature) -> the reference's own records."""
    from ai_crypto_trader_b200.strategy_evaluation import StrategyEvaluationSystem, StrategyPerformanceMetrics
    from oracle import simulate_ref
    meta, arrays = sim_golden
    ses = StrategyEvaluationSystem(config={"evolution": {"optimization_goals": meta["goals"]}})
    for c in meta["cases"][:6]:
        period = c["params"].get("rsi_period", 14)
        pts = simulate_ref.market_points(arrays[f"close_{c['symbol']}"], arrays[f"rsi_{c['symbol']}_{period}"],
                                         f"SYN{c['symbol']:03d}USDT", meta["minute0"])
        recs = ses._simulate_trades(c["name"], dict(c["params"]), pts)
        key = c["key"]
        assert len(recs) == c["n_records"]
        assert [r["side"] == "sell" for r in recs] == arrays[f"sell_{key}"].tolist()
        assert np.array_equal(np.array([r["pnl"] for r in recs]), arrays[f"pnl_{key}"])          # bit-identical float64
        assert np.array_equal(np.array([r["quantity"] for r in recs]), arrays[f"qty_{key}"])
        m = StrategyPerformanceMetrics.calculate_metrics(recs)
        for name, want in c["metrics"].items():
            assert float(m[name]) == unjson(want), (key, name)
        assert float(ses._calculate_strategy_score(m)) == unjson(c["score"])
    assert ses._simulate_trades("empty", {}, []) == []


def test_evolution_service_runs_ga_on_gpu(torch_cuda):
    import asyncio
    from ai_crypto_trader_b200 import synth
    from ai_crypto_trader_b200.evolution import StrategyEvolutionService
    from ai_crypto_trader_b200.sweep import MarketData
    market = MarketData(synth.synth_ohlcv(2, 30000))
    svc = StrategyEvolutionService(market, random_seed=42)
    svc.ga_population_size, svc.ga_generations = 24, 3
    cur = synth.random_population(1, seed=9)[0]
    best = asyncio.run(svc.optimize_with_genetic_algorithm(cur))
    assert best is not None and set(best) == set(svc.param_ranges)
    hist = svc.last_ga.get_generation_history()
    assert len(hist) == 4 and hist[-1]["best_fitness"] >= hist[0]["best_fitness"]
    # the GA's recorded fitness of the final population equals a fresh sweep of it
    again = svc.sweep.evaluate(svc.last_ga.population)
    np.testing.assert_array_equal(np.array(svc.last_ga.fitness_scores), again)
    assert svc.evolution_records[-1]["new_params"] == best


def _check_lanes_vs_oracle(sweep, population, ohlcv, cap):
    from oracle import indicators_ref, sim_oracle
    stats, events = sweep.lane_stats(), sweep.events()
    cfg = sim_oracle.config_of(sweep.market.minute0, 1)
    n_sym = ohlcv.shape[1]
    for s in range(n_sym):
        bank = indicators_ref.rsi_bank(ohlcv[3, s], sweep.periods)
        for i, p in enumerate(population):
            want, ev, _ = sim_oracle.lane(ohlcv[3, s], bank[sweep.period_row[p["rsi_period"]]], p, cfg, event_cap=cap)
            assert int(stats["n_records"][i, s]) == int(want["n_records"]), (i, s)
            assert int(stats["trade_hash"][i, s]) == int(want["trade_hash"]), (i, s)
            if events is not None:
                assert np.array_equal(events[i, s, :len(ev)], ev), (i, s)
            for f in ("n_wins", "n_losses", "n_days", "sum_duration_bars"):
                assert stats[f][i, s] == want[f], (i, s, f)
            for f in ("total_profit", "total_loss", "net_profit", "max_drawdown", "sharpe_ratio", "largest_profit",
                      "largest_loss", "win_rate", "profit_factor", "score", "sortino_ratio", "downside_deviation",
                      "mean_daily_pnl"):
                assert stats[f][i, s] == pytest.approx(float(want[f]), rel=1e-9, abs=1e-11), (i, s, f)
            assert stats["n_negative_days"][i, s] == want["n_negative_days"], (i, s)


@pytest.mark.parametrize("n_bars,opts", [
    (300_000, dict(target_events=1500, warm=4096)),          # many chunks, verified boundaries
    (70_001, dict(target_events=300, warm=0, max_chunks=64, max_repair_rounds=0)),  # no warm-up, no repair: fused fallback
    (150_000, dict(target_events=300, warm=0, max_chunks=64, max_repair_rounds=64)),  # no warm-up: repaired chunk by chunk
    (200_000, dict(target_events=2000, warm=2048, pool_blocks=8)),  # pool far too small -> flagged lanes re-run
])
def test_chunked_sweep_is_exact_and_self_repairing(torch_cuda, n_bars, opts):
    """Time-chunked sweep == serial reference semantics, whether or not the speculation holds."""
    from ai_crypto_trader_b200 import synth
    from ai_crypto_trader_b200.sweep import MarketData, PopulationSweep
    ohlcv = synth.synth_ohlcv(2, n_bars, first_symbol=1)
    market = MarketData(ohlcv)
    cap = 2048
    population = synth.random_population(40, seed=n_bars)
    population[0].update(rsi_oversold=35, rsi_overbought=65, rsi_period=5, take_profit=1, stop_loss=1)
    population[1].update(rsi_oversold=34, rsi_overbought=66, rsi_period=6, take_profit=10, stop_loss=5)
    chunked = PopulationSweep(market, event_cap=cap, mode="chunked", chunk_options=opts)
    fused = PopulationSweep(market, event_cap=cap, mode="fused")
    f_c = chunked.evaluate(population)
    f_f = fused.evaluate(population)
    plan = chunked.plan_chunks(population, **opts)
    assert plan.n_chunks.max() > 1, "the test population must exercise real chunking"
    if opts.get("max_repair_rounds", 8) == 0:
        assert chunked.last_invalid_lanes > 0          # the fallback path really ran
    if opts.get("max_repair_rounds", 8) == 64:
        assert chunked.last_invalid_lanes == 0         # every wrong boundary was repaired in place
    if "pool_blocks" in opts:
        assert chunked.last_pool_overflow and chunked.last_invalid_lanes > 0
    _check_lanes_vs_oracle(chunked, population, ohlcv, cap)
    np.testing.assert_array_equal(chunked.lane_stats()["trade_hash"], fused.lane_stats()["trade_hash"])
    np.testing.assert_allclose(f_c, f_f, rtol=1e-9, atol=1e-11)


def test_chunked_sweep_in_population_slices_with_duplicates(torch_cuda):
    """Large populations go through the chunked kernels slice by slice (shared workspace) and identical
    individuals are evaluated once: results are those of the plain fused sweep, in population order."""
    from ai_crypto_trader_b200 import synth
    from ai_crypto_trader_b200.sweep import MarketData, PopulationSweep
    n_bars = 180_000
    ohlcv = synth.synth_ohlcv(2, n_bars, first_symbol=2)
    market = MarketData(ohlcv)
    cap = 1024
    population = synth.random_population(48, seed=77)
    population[5].update(rsi_oversold=35, rsi_overbought=65, rsi_period=5, take_profit=1, stop_loss=1)
    population += [dict(population[5]), dict(population[0], macd_fast=9, ema_long=77), dict(population[5], atr_period=9)]
    opts = dict(target_events=1500, warm=2048, max_pool_bytes=200_000)
    chunked = PopulationSweep(market, event_cap=cap, mode="chunked", chunk_options=opts)
    fused = PopulationSweep(market, event_cap=cap, mode="fused")
    plans = chunked.plan_batches(population[:48], **opts)
    assert len(plans) > 2 and [p.lo for p in plans] == sorted(p.lo for p in plans)
    assert sum(p.pop for p in plans) == 48 and all(p.workspace.data_ptr() == plans[0].workspace.data_ptr() or
                                                  p.workspace.numel() <= max(q.workspace.numel() for q in plans) for p in plans)
    f_c = chunked.evaluate(population)
    assert chunked.last_unique == 48 and len(f_c) == 51
    f_f = fused.evaluate(population)
    assert fused.last_unique == 48
    np.testing.assert_allclose(f_c, f_f, rtol=1e-9, atol=1e-11)
    assert f_c[48] == f_c[5] and f_c[49] == f_c[0] and f_c[50] == f_c[5]
    sc, sf = chunked.lane_stats(), fused.lane_stats()
    assert sc["trade_hash"].shape == (51, 2)
    np.testing.assert_array_equal(sc["trade_hash"], sf["trade_hash"])
    np.testing.assert_array_equal(chunked.events(), fused.events())
    _check_lanes_vs_oracle(chunked, population, ohlcv, cap)


def test_scan_timing_hook_brackets_the_scan_kernel(torch_cuda):
    """b200bt_sweep_scan_timing: the library records the caller's two events around lane_scan_kernel on the launching stream
    (bench.py's roofline divides by that duration); NULL, NULL switches it off."""
    torch = torch_cuda
    from ai_crypto_trader_b200 import _lib, synth
    from ai_crypto_trader_b200.sweep import MarketData, PopulationSweep
    market = MarketData(synth.synth_ohlcv(2, 200_000, first_symbol=4))
    population = synth.random_population(128, seed=5)
    tiled = PopulationSweep(market, mode="tiled", chunk_options=dict(warm=1024, chunks=6))
    tiled.evaluate(population)
    e0, e1, a, b = (torch.cuda.Event(enable_timing=True) for _ in range(4))
    for e in (e0, e1):
        e.record()                                   # (makes torch create the cudaEvent_t)
    handle = lambda e: (e.cuda_event.value if hasattr(e.cuda_event, "value") else int(e.cuda_event))
    lib = _lib.load()
    try:
        assert lib.b200bt_sweep_scan_timing(handle(e0), handle(e1)) == 0
        a.record()
        tiled.evaluate(population)
        b.record()
    finally:
        lib.b200bt_sweep_scan_timing(None, None)
    torch.cuda.synchronize()
    scan_ms, sweep_ms = e0.elapsed_time(e1), a.elapsed_time(b)
    assert 0.0 < scan_ms < sweep_ms
    e1.record()                                      # hook off: the next sweep leaves the events alone
    torch.cuda.synchronize()
    t_before = e0.elapsed_time(e1)
    tiled.evaluate(population)
    torch.cuda.synchronize()
    assert e0.elapsed_time(e1) == t_before


def test_scan_tiles_that_do_not_arrive_are_redone_exactly(torch_cuda):
    """The scan's wait for a tile is bounded; a tile that does not arrive in time costs its work item, which is re-scanned by
    the repair pass or re-run by the exact fallback.  The test hook makes every warp give up at the third tile of an item."""
    from ai_crypto_trader_b200 import _lib, synth
    from ai_crypto_trader_b200.sweep import MarketData, PopulationSweep
    ohlcv = synth.synth_ohlcv(2, 200_000, first_symbol=2)
    market = MarketData(ohlcv)
    population = synth.random_population(200, seed=77)
    fused = PopulationSweep(market, mode="fused")
    f_f = fused.evaluate(population)
    tiled = PopulationSweep(market, mode="tiled", chunk_options=dict(warm=1024, chunks=6))
    lib = _lib.load()
    lib.b200bt_sweep_scan_wait_cycles(-3)
    try:
        f_t = tiled.evaluate(population)
        stalls, invalid = tiled.last_scan_stalls, tiled.last_invalid_lanes
        h_t = tiled.lane_stats()["trade_hash"].copy()
    finally:
        lib.b200bt_sweep_scan_wait_cycles(0)
    assert stalls > 0 and invalid > 0                     # the path really ran
    np.testing.assert_array_equal(h_t, fused.lane_stats()["trade_hash"])
    np.testing.assert_allclose(f_t, f_f, rtol=1e-9, atol=1e-11)
    f_t2 = tiled.evaluate(population)                     # and the default bound is back
    assert tiled.last_scan_stalls == 0
    np.testing.assert_allclose(f_t2, f_f, rtol=1e-9, atol=1e-11)


@pytest.mark.parametrize("n_bars,opts", [
    (300_000, dict(warm=4096)),                                        # wave-fitted K, verified boundaries
    (300_001, dict(warm=4096, chunks=7)),                              # ragged last tile
    (70_001, dict(warm=0, chunks=16, max_repair_rounds=0)),            # no warm-up, no repair: fused fallback
    (150_000, dict(warm=0, chunks=32, max_repair_rounds=64)),          # no warm-up: repaired chunk by chunk
    (200_000, dict(warm=2048, chunks=8, pool_blocks=8)),               # pool far too small -> flagged lanes re-run
    (5_000, dict(warm=512, chunks=1)),                                 # a single chunk
    (140_000, dict(warm=2048, chunks=6, order_by="identity")),         # population order: warps reading > 2 RSI rows are flagged and re-run
    (140_000, dict(warm=2048, chunks=6, order_by="row_thresholds")),   # the other packing
])
def test_tiled_sweep_is_exact_and_self_repairing(torch_cuda, n_bars, opts):
    """Thread-per-lane sweep == serial reference semantics, whether or not the speculation holds."""
    from ai_crypto_trader_b200 import synth
    from ai_crypto_trader_b200.sweep import MarketData, PopulationSweep
    ohlcv = synth.synth_ohlcv(2, n_bars, first_symbol=1)
    market = MarketData(ohlcv)
    cap = 2048
    population = synth.random_population(300, seed=n_bars)            # two CTAs per (symbol, chunk), one ragged
    population[0].update(rsi_oversold=35, rsi_overbought=65, rsi_period=5, take_profit=1, stop_loss=1)
    population[1].update(rsi_oversold=34, rsi_overbought=66, rsi_period=6, take_profit=10, stop_loss=5)
    population[2].update(rsi_oversold=60, rsi_overbought=40, rsi_period=10, take_profit=2, stop_loss=2)   # inverted
    tiled = PopulationSweep(market, event_cap=cap, mode="tiled", chunk_options=opts)
    fused = PopulationSweep(market, event_cap=cap, mode="fused")
    f_t = tiled.evaluate(population)
    f_f = fused.evaluate(population)
    hash_first = tiled.lane_stats()["trade_hash"].copy()
    first_invalid, first_overflow = tiled.last_invalid_lanes, tiled.last_pool_overflow
    f_t2 = tiled.evaluate(population)          # the second sweep of a bank goes through the zone map (block skipping)
    assert tiled._zones is not None
    np.testing.assert_allclose(f_t2, f_t, rtol=1e-12, atol=0)   # (lanes may switch between the chunked and the fused arithmetic)
    np.testing.assert_array_equal(tiled.lane_stats()["trade_hash"], hash_first)
    plan = tiled.plan_tiles(population, **opts)
    if "chunks" in opts:
        assert plan.K == opts["chunks"]
    if opts.get("max_repair_rounds", 8) == 0:
        assert first_invalid > 0                       # the fallback path really ran
    if opts.get("max_repair_rounds", 8) == 64:
        assert first_invalid == 0                      # every wrong boundary was repaired in place
    if opts.get("order_by") == "identity":
        assert first_invalid > 0                       # unpacked warps went through the exact fallback
    if "pool_blocks" in opts:
        assert first_overflow and first_invalid > 0    # (the second sweep planned a larger pool)
        assert not tiled.last_pool_overflow
    np.testing.assert_array_equal(tiled.lane_stats()["trade_hash"], fused.lane_stats()["trade_hash"])
    np.testing.assert_array_equal(tiled.lane_stats()["n_records"], fused.lane_stats()["n_records"])
    ev_t, ev_f, n_rec = tiled.events(), fused.events(), fused.lane_stats()["n_records"]
    live = np.arange(cap)[None, None, :] < n_rec[:, :, None]          # slots past a lane's last record are undefined
    np.testing.assert_array_equal(ev_t[live], ev_f[live])
    np.testing.assert_allclose(f_t, f_f, rtol=1e-9, atol=1e-11)
    _check_lanes_vs_oracle(tiled, population[:24], ohlcv, cap)


def test_evaluate_edge_populations(torch_cuda):
    """Empty population, one individual, one symbol, a series shorter than one tile -- through the default mode."""
    from ai_crypto_trader_b200 import synth
    from ai_crypto_trader_b200.sweep import MarketData, PopulationSweep
    from oracle import indicators_ref, sim_oracle
    for n_bars in (7, 200_001):
        ohlcv = synth.synth_ohlcv(1, n_bars, first_symbol=6)
        market = MarketData(ohlcv)
        sweep = PopulationSweep(market)
        assert sweep.evaluate([]).shape == (0,)
        one = synth.random_population(1, seed=n_bars)
        f = sweep.evaluate(one)
        bank = indicators_ref.rsi_bank(ohlcv[3, 0], sweep.periods)
        want, _, _ = sim_oracle.lane(ohlcv[3, 0], bank[sweep.period_row[one[0]["rsi_period"]]], one[0],
                                     sim_oracle.config_of(market.minute0, 1))
        assert f.shape == (1,) and f[0] == pytest.approx(float(want["score"]), rel=1e-9, abs=1e-12)
        assert int(sweep.lane_stats()["n_records"][0, 0]) == int(want["n_records"])


def test_multi_timeframe_bank_and_sweep(torch_cuda):
    """BASELINE configs[3]: RSI banks on 1m / 5m / 15m (device resample -> RSI -> align to the 1-minute clock), the gene
    `rsi_timeframe` selecting the block: bank rows against the pandas/NumPy restatement, lanes against the C oracle fed
    those rows -- through the fused kernel and through the thread-per-lane kernels (78 RSI rows)."""
    from ai_crypto_trader_b200 import synth
    from ai_crypto_trader_b200.sweep import MarketData, PopulationSweep
    from oracle import indicators_ref, sim_oracle
    import random
    S, N, POP = 2, 150_001, 200
    minute0 = synth.EPOCH_2024_MINUTES + 7                       # not aligned to the 5 / 15 minute grid
    ohlcv = synth.synth_ohlcv(S, N, first_symbol=4)
    market = MarketData(ohlcv, minute0=minute0)
    tfs = (1, 5, 15)
    population = synth.random_population(POP, seed=21)
    rnd = random.Random(5)
    for p in population:
        p["rsi_timeframe"] = rnd.randint(0, 2)
    population[0].update(rsi_oversold=35, rsi_overbought=65, rsi_period=5, take_profit=1, stop_loss=1, rsi_timeframe=2)
    cfg = sim_oracle.config_of(minute0, 1)
    want = None
    for mode, opts in (("fused", {}), ("tiled", dict(chunks=6, warm=4096))):
        sweep = PopulationSweep(market, timeframes=tfs, mode=mode, chunk_options=opts, event_cap=0)
        P = len(sweep.periods)
        assert tuple(sweep.bank.shape) == (S, 3 * P, N)
        if want is None:
            bank = sweep.bank.cpu().numpy()
            rows = {}
            for s in range(S):
                rows[s, 0] = indicators_ref.rsi_bank(ohlcv[3, s], sweep.periods)
                for i, k in enumerate(tfs[1:], start=1):
                    rows[s, i] = indicators_ref.rsi_rows_on_timeframe(ohlcv[3, s], minute0, k, sweep.periods)
                for i in range(3):
                    got, ref = bank[s, i * P:(i + 1) * P], rows[s, i]
                    assert np.array_equal(np.isnan(got), np.isnan(ref)), (s, i)
                    neq = (got != ref) & ~np.isnan(ref)
                    assert int(neq.sum()) <= max(2, int(2e-6 * ref.size)), (s, i, int(neq.sum()))   # double-rounding ties only
            want = np.zeros((POP, S), dtype=sim_oracle.STATS_DTYPE)
            for s in range(S):
                for i, p in enumerate(population):
                    r = rows[s, p["rsi_timeframe"]][sweep.period_row[p["rsi_period"]]]
                    want[i, s] = sim_oracle.lane(ohlcv[3, s], r, p, cfg)[0]
        for _ in range(2):
            fit = sweep.evaluate(population)
        st = sweep.lane_stats()
        assert np.array_equal(st["n_records"], want["n_records"]), mode
        assert np.array_equal(st["trade_hash"], want["trade_hash"]), mode
        np.testing.assert_allclose(st["score"], want["score"], rtol=1e-9, atol=1e-11, equal_nan=True)
        np.testing.assert_allclose(fit, want["score"].mean(axis=1), rtol=1e-9, atol=1e-11, equal_nan=True)
        if mode == "tiled":
            assert sweep.last_invalid_lanes == 0             # packed by bank row: no warp reads more than two rows
    assert len({int(r) for r in want["n_records"][:, 0]}) > 20


@pytest.mark.parametrize("n_bars", [5, 127, 4096, 8192, 70_001, 262_144 + 33])
def test_zone_rows_written_with_the_bank_equal_the_zone_map_kernel(torch_cuda, n_bars):
    """b200bt_rsi_bank_zones writes the (min, max) ranges of the bank while it computes it (rows of a sub-range of the
    symbols, as the upload pipeline does per quarter): bit-equal to b200bt_zone_map run on the finished bank, padding
    included."""
    torch = torch_cuda
    import ctypes as C
    from ai_crypto_trader_b200 import _lib, synth
    from ai_crypto_trader_b200.sweep import rsi_bank
    S, periods = 3, [1, 2, 5, 14, 30]
    P = len(periods)
    close = torch.from_numpy(synth.synth_ohlcv(S, n_bars, first_symbol=3)[3]).cuda()
    nz = int(_lib.load().b200bt_zone_map_floats(P, S, n_bars))
    fused = torch.full((nz,), 7.0, dtype=torch.float32, device="cuda")
    bank = torch.empty((S, P, n_bars), dtype=torch.float32, device="cuda")
    rsi_bank(close[:1], periods, out=bank[:1], zones=fused, zones_symbols=S, first_symbol=0)
    rsi_bank(close[1:], periods, out=bank[1:], zones=fused, zones_symbols=S, first_symbol=1)
    assert torch.equal(bank, rsi_bank(close, periods))
    want = torch.empty(nz, dtype=torch.float32, device="cuda")
    _lib.call("b200bt_zone_map", close.data_ptr(), _lib.ld(close), bank.data_ptr(), _lib.ld(bank), P, S, n_bars, want.data_ptr(),
              _lib.current_stream())
    a, b = fused.cpu().numpy(), want.cpu().numpy()
    assert np.array_equal(np.isnan(a), np.isnan(b))
    assert np.array_equal(a[~np.isnan(b)], b[~np.isnan(b)])
