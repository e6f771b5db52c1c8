"""BASELINE configs[0] on the GPU: StrategyTester / BacktestEngine vs the reference's own
StrategyTester run (tests/golden/bt_reference.*)."""
import asyncio
from datetime import datetime

import numpy as np
import pytest

from conftest import unjson
from test_oracle_bt import bt_frame, load_bt_golden

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def gpu(native_lib):
    import torch
    assert torch.cuda.is_available()
    torch.cuda.set_device(0)
    return torch


def _check_against_reference(st, case, arrays, df):
    name = case["name"]
    bar = {t.isoformat(): i for i, t in enumerate(df.index)}
    tr = st["trades"]
    assert len(tr) == case["n_trades"], name
    assert [bar[t["entry_time"]] for t in tr] == arrays[f"entry_bar_{name}"].tolist()      # bit-exact bars
    assert [bar[t["exit_time"]] for t in tr] == arrays[f"exit_bar_{name}"].tolist()
    code = {"Stop Loss": 1, "Take Profit": 2, "End of Test": 3}
    assert [code[t["exit_reason"]] for t in tr] == arrays[f"reason_{name}"].tolist()
    for k in ("entry_price", "quantity", "position_size", "pnl", "pnl_pct"):
        np.testing.assert_allclose(np.array([t[k] for t in tr], dtype=np.float64), arrays[f"{k}_{name}"], rtol=1e-12, atol=1e-12, err_msg=k)
    # equity curve: north-star tolerance 1e-5 relative; held to 1e-12
    np.testing.assert_allclose(np.array([p["equity"] for p in st["equity_curve"]]), arrays[f"eq_{name}"], rtol=1e-12)
    assert [bar[p["timestamp"]] for p in st["equity_curve"]] == arrays[f"eq_bar_{name}"].tolist()
    dd = np.array([[p["drawdown"], p["drawdown_pct"]] for p in st["drawdown_curve"]]).reshape(-1, 2)
    np.testing.assert_allclose(dd, arrays[f"dd_{name}"], rtol=1e-9, atol=1e-9)
    for k, want in case["stats"].items():
        assert float(st[k]) == pytest.approx(unjson(want), rel=1e-9, abs=1e-9), (name, k)


def test_strategy_tester_matches_reference(gpu, tmp_path):
    from ai_crypto_trader_b200.backtesting import HistoricalDataManager, StrategyTester
    meta, arrays = load_bt_golden()
    for case in meta:
        df = bt_frame(case)
        tester = StrategyTester(config={}, data_manager=HistoricalDataManager(None, data_dir=str(tmp_path / "data")),
                                results_dir=str(tmp_path / "res"), config_path=None)
        st = asyncio.run(tester.backtest_frame(df, "SYNUSDC"))
        c = tester.frame_constants
        assert c["signal"] == case["signal"] and c["strength"] == pytest.approx(unjson(case["strength"]), rel=1e-4, abs=1e-4)
        for k, want in case["constants"].items():
            if isinstance(want, str):
                assert c[k] == want
            else:
                assert c[k] == pytest.approx(unjson(want), rel=3e-5, abs=3e-6), (case["name"], k)
        _check_against_reference(st, case, arrays, df)


def test_backtest_engine_csv_store_roundtrip(gpu, tmp_path, monkeypatch):
    """run_backtest.py's path: CSV store -> BacktestEngine.run_multiple_backtests -> stats + summary."""
    from ai_crypto_trader_b200.backtesting import BacktestEngine
    meta, arrays = load_bt_golden()
    monkeypatch.chdir(tmp_path)
    eng = BacktestEngine(config_path=None, config={}, data_dir=str(tmp_path / "data"), results_dir=str(tmp_path / "results"))
    frames = {}
    for case, sym in zip(meta, ("AAAUSDC", "BBBUSDC", "CCCUSDC")):
        df = bt_frame(case)
        frames[sym] = (case, df)
        eng.data_manager.save_market_data(sym, "1m", df, df.index[0].to_pydatetime(), df.index[-1].to_pydatetime())
    start, end = datetime(2024, 1, 1), datetime(2024, 1, 4)
    res = asyncio.run(eng.run_multiple_backtests(list(frames), ["1m"], start, end))
    assert res["summary"]["total_results"] == 3
    for sym, (case, df) in frames.items():
        st = res[sym]["1m"]
        assert "error" not in st
        _check_against_reference(st, case, arrays, df)
    avail = eng.get_available_data()
    assert set(avail) == set(frames) and "1m" in avail["AAAUSDC"]["intervals"]
    # error convention: missing data -> {'error': ...}, never raises
    assert "error" in asyncio.run(eng.run_backtest("NOPEUSDC", "1m", start, end))
    # sidecar (f1): binary fp32 load equals the CSV parse
    o1, m1 = eng.data_manager.load_ohlcv32("AAAUSDC", "1m", start, end)
    dfc = eng.data_manager.load_market_data("AAAUSDC", "1m", start, end)
    assert np.array_equal(o1[3], dfc["close"].to_numpy(dtype=np.float32)) and len(m1) == len(dfc)
    # task queue surface
    async def q():
        tid = await eng.add_backtest_task("run_backtest", {"symbol": "BBBUSDC", "interval": "1m", "start_date": start.isoformat(), "end_date": end.isoformat()})
        await eng.process_task_queue(stop_when_empty=True)
        return tid
    assert asyncio.run(q()) == 1
