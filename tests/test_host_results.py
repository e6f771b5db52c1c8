"""ResultAnalyzer drop-in against the reference's own outputs (tests/golden/ra_reference.json, produced by executing
backtesting/result_analyzer.py in make_golden.py), and the package entry points the reference's run_backtest.py CLI
calls."""
import json
import os
import sys
from pathlib import Path


from conftest import GOLDEN


def _strip(rs):
    return [dict(r, file_path=Path(r["file_path"]).name) for r in rs]


def test_result_analyzer_matches_reference_outputs(tmp_path):
    from ai_crypto_trader_b200.backtesting.result_analyzer import ResultAnalyzer
    ref = json.loads((GOLDEN / "ra_reference.json").read_text())
    for i, doc in enumerate(ref["documents"]):
        (tmp_path / f"result_{i:02d}.json").write_text(json.dumps(doc))
    (tmp_path / "broken.json").write_text("{not json")
    ra = ResultAnalyzer(str(tmp_path), plots_dir=str(tmp_path / "plots"))
    avail = sorted(ra.get_available_results(), key=lambda r: r["file_path"])
    assert _strip(avail) == ref["available"]                      # the broken file is skipped, file_path added
    for f in ref["filters"]:
        got = sorted(Path(r["file_path"]).name for r in ra.filter_results(**f["criteria"]))
        assert got == f["files"], f["criteria"]
    s = ra.generate_summary_report(avail)
    for k in ("strategies", "symbols", "intervals"):
        s[k] = sorted(s[k])
    s["best_result"], s["worst_result"] = _strip([s["best_result"]])[0], _strip([s["worst_result"]])[0]
    for r in s["results"]:
        r["file_path"] = Path(r["file_path"]).name
    assert s == ref["summary"]                                    # every number bit-equal (same float expressions)
    assert ra.generate_summary_report([]) == ref["summary_empty"] == {}
    assert ra.load_results(str(tmp_path / "does_not_exist.json")) == ref["load_missing"] == {}
    assert ra.load_results(str(tmp_path / "result_00.json")) == ref["load_first"]
    # compare_results: the table the reference charts (:338-361), written as CSV here; unknown metric / no results -> None
    path = ra.compare_results(avail, "sharpe_ratio")
    assert path and Path(path).exists()
    assert ra.compare_results(avail, "no_such_metric") is None and ra.compare_results([], "return_pct") is None
    rows = ra.comparison_table(avail)
    assert [r["return_pct"] for r in rows] == [r["return_pct"] for r in ref["summary"]["results"]]
    assert Path(ra.save_summary_report(s)).exists()


def test_cli_entry_points_on_the_dropin(tmp_path, monkeypatch):
    """What the reference's run_backtest.py calls for `list`, `analyze` and `backtest`, with `import backtesting` resolved
    to the drop-in and every object built with its default, working-directory-relative paths."""
    import asyncio
    import numpy as np
    import pandas as pd
    from datetime import datetime
    from ai_crypto_trader_b200 import synth
    import ai_crypto_trader_b200.backtesting as dropin
    for name in ("backtesting", "backtesting.backtest_engine", "backtesting.data_manager", "backtesting.result_analyzer",
                 "backtesting.strategy_tester"):
        monkeypatch.setitem(sys.modules, name, None)                # (removed again after the test)
    dropin.install_as_backtesting()
    from backtesting import BacktestEngine, ResultAnalyzer
    from backtesting.data_manager import HistoricalDataManager
    assert BacktestEngine is dropin.BacktestEngine and HistoricalDataManager is dropin.HistoricalDataManager
    monkeypatch.chdir(tmp_path)
    n = 3000
    d = synth.synth_symbol(0, n)
    idx = pd.date_range("2024-01-01", periods=n, freq="min")
    df = pd.DataFrame({k: d[k].astype(np.float64) for k in synth.FIELDS}, index=idx)
    dm = HistoricalDataManager()
    dm.save_market_data("SYNUSDC", "1m", df, datetime(2024, 1, 1), datetime(2024, 1, 3))
    # list
    dm = HistoricalDataManager()
    assert dm.available_symbols() == ["SYNUSDC"] and dm.available_intervals("SYNUSDC") == ["1m"]
    first, last = dm.get_data_range("SYNUSDC", "1m")
    assert (first.strftime("%Y-%m-%d"), last.strftime("%Y-%m-%d"), (last - first).days) == ("2024-01-01", "2024-01-03", 2)
    # analyze: result files in the reference's layout (backtesting/results/*.json)
    ref = json.loads((GOLDEN / "ra_reference.json").read_text())
    res = tmp_path / "backtesting" / "results"
    res.mkdir(parents=True, exist_ok=True)
    for i, doc in enumerate(ref["documents"]):
        (res / f"result_{i:02d}.json").write_text(json.dumps(doc))
    ra = ResultAnalyzer()
    results = ra.filter_results(symbol="BTCUSDC", interval=None)
    summary = ra.generate_summary_report(results)
    assert summary["total_results"] == 3 and summary["symbols"] == ["BTCUSDC"]
    assert Path(ra.save_summary_report(summary)).exists() and Path(ra.compare_results(results, "win_rate")).exists()
    picked = [r for r in (ra.load_results(str(res / "result_05.json")), ra.load_results(str(res / "missing.json"))) if r]
    summary = ra.generate_summary_report(picked)
    assert summary["total_results"] == 1 and summary["best_result"]["symbol"] == "ETHUSDC"
    assert ra.filter_results(symbol="NOPEUSDC", interval=None) == []
    # backtest: on a CUDA box the stats of the GPU path; without a device the reference's error convention
    # ({'error': ...} per (symbol, interval), backtest_engine.py:125) -- never a CPU fallback
    bt = asyncio.run(BacktestEngine().run_multiple_backtests(["SYNUSDC"], ["1m"], datetime(2024, 1, 1), datetime(2024, 1, 4), 10000.0))
    assert set(bt["SYNUSDC"]) == {"1m"}
    import torch
    if torch.cuda.is_available():
        assert bt["SYNUSDC"]["1m"]["initial_balance"] == 10000.0 and "total_trades" in bt["SYNUSDC"]["1m"]
    else:
        assert "error" in bt["SYNUSDC"]["1m"]


def test_sidecar_is_ignored_once_its_csv_changes(tmp_path):
    """ADVICE r1: a CSV rewritten after the sidecar was made must win; sub-minute bars must not collapse."""
    import numpy as np
    import pandas as pd
    from datetime import datetime
    from ai_crypto_trader_b200.backtesting import HistoricalDataManager
    dm = HistoricalDataManager(None, data_dir=str(tmp_path))
    n = 500
    idx = pd.date_range("2024-01-01", periods=n, freq="30s")            # two bars per minute
    rng = np.random.default_rng(0)
    df = pd.DataFrame({k: rng.uniform(10, 20, n) for k in ("open", "high", "low", "close", "volume")}, index=idx)
    a, b = datetime(2024, 1, 1), datetime(2024, 1, 2)
    path = dm.save_market_data("AAAUSDC", "30s", df, a, b)
    o1, m1 = dm.load_ohlcv32("AAAUSDC", "30s", a, b)
    assert o1.shape == (5, n) and (np.diff(m1) >= 0).all() and len(np.unique(m1)) == n // 2
    assert np.array_equal(o1[3], df["close"].to_numpy(dtype=np.float32))
    assert dm._sidecar_if_fresh(path) is not None
    # the fetcher rewrites the CSV (backtesting/data_manager.py:191-196): the stale sidecar must not shadow it
    df2 = df * 2.0
    df2.index.name = "timestamp"
    df2.to_csv(path)
    os.utime(path, ns=(path.stat().st_atime_ns, path.stat().st_mtime_ns + 5_000_000_000))
    assert dm._sidecar_if_fresh(path) is None
    dm.market_data_cache.clear()
    o2, _ = dm.load_ohlcv32("AAAUSDC", "30s", a, b)
    assert np.array_equal(o2[3], df2["close"].to_numpy(dtype=np.float32))
