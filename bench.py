#!/usr/bin/env python
"""bench.py -- GA population-fitness sweep throughput (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W [--impl reference]

A "step" is one generation's fitness evaluation: the state-machine sweep over
every (individual x symbol) lane of the population plus the fitness reduction
(and, for N > 1, one NCCL all-gather of the fitness vector).  Workload at N=1 is
BASELINE.json configs[1]: population 1024, 10 symbols, 1M synthetic 1-minute
bars.  For N > 1 the population is sharded by individual, per-GPU work fixed
(weak scaling): global population = 1024*N, market data replicated.

Prints ONE JSON line (rank 0).  See DESIGN.md "Measurement" for every field.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

METRIC = "bar_strategy_evals_per_sec"
UNIT = "evals/s"
POP_PER_GPU = 1024
N_SYMBOLS = 10
N_BARS = 1_000_000
BYTES_PER_EVAL = 8  # SURVEY 8(d): price 4 B + RSI 4 B per (individual, symbol, bar), reference RSI rule
# ncu figures of the dominant kernel per launch on the configs[1] workload (pop 1024 x 10 x 1M, seed-42 population), from
# the committed `ncu --set full` capture named in "source"; "scan_share" = the kernel's share of the sweep's kernel time in
# the committed launch list of this bench command.  Valid for exactly that workload (the kernels are deterministic).
NCU_C2 = {
    "tiled": {"warp_inst": 3.2099e9, "threads_per_inst": 13.70, "dram_bytes": 4.613e9 + 1.032e9, "scan_share": 0.579,
              "issue_active_pct": 69.4, "alu_pipe_pct": 54.7,
              "source": "profiles/r2_lane_scan_ncu.txt (ncu --set full), profiles/r2_launches.csv (launch list of `bench.py --steps 2 --warmup 3 --skip-extras`)"},
}


def measured_hbm_peak():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        try:
            return float(json.loads(p.read_text())["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


_T0 = time.perf_counter()


_LAST_PHASE = [""]


def _phase(msg: str) -> None:
    """Progress marker on stderr (the JSON line is the only thing on stdout): where a run is, should it ever stall."""
    _LAST_PHASE[0] = msg
    print(f"[bench +{time.perf_counter() - _T0:7.1f}s] {msg}", file=sys.stderr, flush=True)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "20", "-i", str(self.index)],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), line.strip()))

    def stop(self, t0: float, t1: float):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        rows = [r for (t, r) in self.rows if t0 <= t <= t1] or [r for (_, r) in self.rows[-3:]]
        sm, smax, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in rows:
            f = [x.strip() for x in r.split(",")]
            try:
                sm.append(float(f[0])); smax.append(float(f[1]))
            except Exception:
                continue
            for name, val in zip(names, f[3:7]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(smax) if smax else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# --------------------------------------------------------------------------
# CPU arms.  `--impl reference` and the inline `cpu_baseline` leg use ONE recipe (same pool, same sample shape, the
# timer started after the pool is warm), so the two agree:
#   kind "reference": the reference's own _simulate_trades + calculate_metrics + _calculate_strategy_score, imported
#                     unmodified from oracle/_ref (placed there by oracle/make_ref.py in the build container; it
#                     travels to the GPU box with the snapshot, where /root/reference does not exist)
#   kind "port"     : the float64 Python restatement (oracle/simulate_ref.py) when oracle/_ref is not populated
# plus the same algorithm as compiled C (oracle/sim_oracle.c) under the same pool: the strong CPU baseline.
# --------------------------------------------------------------------------
_REF_STREAMS = []   # market-data dict lists, built in the parent before the fork (shared copy-on-write)
_REF_ARRAYS = []    # (close, rsi) fp32 rows of the same streams, for the C port
REF_BARS = 250_000
REF_LANES_PER_WORKER = 4


def _ref_kind() -> str:
    from oracle import make_ref
    return "reference" if make_ref.available() else "port"


def _ref_worker(job):
    stream, params, goals = job
    if stream < 0:                 # pool warm-up: import the modules, touch the data
        from oracle import make_ref, simulate_ref, sim_oracle   # noqa: F401
        if make_ref.available():
            make_ref.load()
        sim_oracle.lib()
        return 0.0, 0
    from oracle import make_ref
    if make_ref.available():
        ses, metrics_cls, _ = make_ref.load()
        ses.optimization_goals = goals
        recs = ses._simulate_trades("bench", dict(params), _REF_STREAMS[stream])
        m = metrics_cls.calculate_metrics(recs)
        return float(ses._calculate_strategy_score(m)), len(recs)
    from oracle import simulate_ref
    recs = simulate_ref.simulate_trades(params, _REF_STREAMS[stream])
    m = simulate_ref.calculate_metrics(recs)
    return float(simulate_ref.strategy_score(m, goals)), len(recs)


def _c_worker(job):
    stream, plist = job
    from oracle import sim_oracle
    from ai_crypto_trader_b200 import synth
    close, rsi = _REF_ARRAYS[stream]
    out = sim_oracle.lanes(close, rsi, plist, sim_oracle.config_of(synth.EPOCH_2024_MINUTES, 1))
    return float(out["score"].sum())


def reference_sample(n_bars: int, lanes: int):
    """Bounded sample of the workload: `lanes` individuals of the seed-42 population on n_bars bars of symbol 0, their
    rsi_period folded onto two streams (7, 14) so the prebuilt market-data dict lists stay small.  Returns the job list."""
    from ai_crypto_trader_b200 import synth
    from ai_crypto_trader_b200.sweep import DEFAULT_GOALS
    from oracle import indicators_ref, simulate_ref
    pop = synth.random_population(lanes, seed=42)
    close = synth.synth_symbol(0, n_bars)["close"]
    periods = [7, 14]
    bank = indicators_ref.rsi_bank(close, periods)
    _REF_STREAMS.clear()
    _REF_ARRAYS.clear()
    for row in bank:
        _REF_STREAMS.append(simulate_ref.market_points(close, row, "SYN000USDT", synth.EPOCH_2024_MINUTES))
        _REF_ARRAYS.append((close, row))
    return [(i % 2, dict(p, rsi_period=periods[i % 2]), DEFAULT_GOALS) for i, p in enumerate(pop)]


def run_cpu_pool(steps: int, warmup: int, c_port_steps: int = 0):
    """-> (per-step seconds of the Python arm, evals per step, cores, sample text, kind, C-port dict or None)."""
    import multiprocessing as mp
    cores = os.cpu_count() or 1
    use = max(1, min(cores, 64))
    lanes = use * REF_LANES_PER_WORKER
    jobs = reference_sample(REF_BARS, lanes)
    kind = _ref_kind()
    times, c_port = [], None
    with mp.get_context("fork").Pool(use) as pool:
        pool.map(_ref_worker, [(-1, None, None)] * (2 * use), chunksize=1)         # warm: imports done in every worker
        for it in range(warmup + steps):
            t0 = time.perf_counter()
            pool.map(_ref_worker, jobs, chunksize=1)
            dt = time.perf_counter() - t0
            if it >= warmup:
                times.append(dt)
        if c_port_steps:
            # the C port is ~200x faster per lane: full-length series, many more lanes, same pool
            from ai_crypto_trader_b200 import synth
            from oracle import indicators_ref
            close = synth.synth_symbol(0, N_BARS)["close"]
            _REF_ARRAYS.clear()
            _REF_ARRAYS.extend((close, row) for row in indicators_ref.rsi_bank(close, [7, 14]))
            pop = synth.random_population(use * 32, seed=42)
            cjobs = [(w % 2, pop[w * 32:(w + 1) * 32]) for w in range(use)]
    if c_port_steps:
        with mp.get_context("fork").Pool(use) as pool:        # (forked after the full-length rows exist)
            pool.map(_c_worker, cjobs, chunksize=1)
            t0 = time.perf_counter()
            for _ in range(c_port_steps):
                pool.map(_c_worker, cjobs, chunksize=1)
            dtc = (time.perf_counter() - t0) / c_port_steps
        c_port = {"value": N_BARS * len(pop) / dtc, "unit": UNIT, "cores": use,
                  "sample": f"{len(pop)} lanes x {N_BARS} bars per step, oracle/sim_oracle.c (-O2), {use} processes"}
    what = ("the reference's own _simulate_trades + calculate_metrics + _calculate_strategy_score (oracle/_ref, unmodified)"
            if kind == "reference" else "pure-Python float64 restatement of _simulate_trades + calculate_metrics + score (oracle/_ref not populated)")
    sample = (f"{lanes} lanes x {REF_BARS} bars of configs[1] per step ({REF_LANES_PER_WORKER} lanes per worker, {use} processes; {what}; "
              "market-data dicts prebuilt outside the timed region, pool warm before the timer starts)")
    return times, REF_BARS * lanes, use, sample, kind, c_port


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    times, evals_per_step, use, sample, kind, _ = run_cpu_pool(args.steps, args.warmup)
    total = sum(times)
    value = evals_per_step * len(times) / total
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * total / len(times), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": f"GA fitness sweep pop={POP_PER_GPU}x{args.gpus} symbols={N_SYMBOLS} bars={N_BARS} (bounded sample)",
                   "sample": sample},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": use, "kind": kind, "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def cpu_baseline_inline():
    """Rank-0, N=1 only: the CPU arms timed on the host cores on a bounded sample (same recipe as --impl reference)."""
    times, evals_per_step, use, sample, kind, c_port = run_cpu_pool(steps=2, warmup=1, c_port_steps=2)
    py = {"value": evals_per_step * len(times) / sum(times), "unit": UNIT, "cores": use, "kind": kind, "sample": sample}
    py["c_port_64core"] = c_port
    # BASELINE configs[0] (the reference's own CPU-runnable case): StrategyTester.backtest_strategy on 10 000 bars of one
    # symbol, restated in Python with the LLM stubbed (oracle/tester_ref.py), single process like the reference
    from oracle import tester_ref
    df = configs0_frame()
    t0 = time.perf_counter()
    st = tester_ref.backtest(df)
    py["configs0_backtest"] = {"cpu_ms": (time.perf_counter() - t0) * 1e3, "bars": len(df), "trades": int(st["total_trades"]),
                               "sample": "1 strategy x 1 symbol x 10 000 bars, oracle/tester_ref.py, 1 core"}
    # BASELINE configs[2] on the CPU (SURVEY 8(d)-iii): the reference's NumPy GBM loop + per-path drawdowns, float64, at
    # 10^5 paths x 1 000 steps (the full 10^6 x 10^4 would need an 80 GB array), one core like the reference
    import numpy as np
    from oracle import mc_ref
    ret = np.random.default_rng(7).normal(5e-4, 0.02, 60)
    mu, sigma = float(np.mean(ret) * 252), float(np.std(ret, ddof=1) * np.sqrt(252))
    t0 = time.perf_counter()
    fin, mdd = mc_ref.numpy_gbm_reference(100.0, mu, sigma, 1001, 100_000, seed=1)
    mc_ref.risk_statistics(fin, mdd, 100.0, 0.95)
    dt = time.perf_counter() - t0
    py["mc_gbm_numpy"] = {"path_steps_per_s": 100_000 * 1000 / dt, "seconds": dt, "cores": 1,
                          "sample": "100 000 paths x 1 000 steps, float64 (days, n) array stepped in time + drawdowns + percentiles (oracle/mc_ref.numpy_gbm_reference = monte_carlo_service.py:266-336)"}
    # GA operators on the host (SURVEY 8(d)-iv): the reference's own selection / crossover / mutation for one generation
    try:
        from oracle import make_ref
        from ai_crypto_trader_b200 import synth
        _, _, RefGA = make_ref.load()
        ga = RefGA(synth.param_ranges(), lambda ind: float(ind["rsi_period"]), population_size=POP_PER_GPU, generations=1, random_seed=42)
        ga.initialize_population()
        ga.evaluate_population()
        t0 = time.perf_counter()
        for _ in range(3):
            ga.evolve_generation()
            ga.evaluate_population()
        py["ga_operators_reference_ms"] = {"value": (time.perf_counter() - t0) / 3 * 1e3, "population": POP_PER_GPU,
                                           "sample": "services/genetic_algorithm.py evolve_generation (oracle/_ref, unmodified) with a trivial fitness, 1 core"}
    except Exception as e:      # oracle/_ref absent: the leg is skipped, never replaced
        py["ga_operators_reference_ms"] = {"unavailable": f"{type(e).__name__}: {e}"}
    return py


def _claim_stdout() -> int:
    """The JSON line must be the only thing on stdout, but libraries write there too (NCCL prints its version line to fd 1
    whatever NCCL_DEBUG_FILE says): file descriptor 1 is pointed at stderr for the rest of the process and the original
    is returned for the one os.write of the result."""
    try:
        sys.stdout.flush()
        real = os.dup(1)
        os.dup2(2, 1)
        return real
    except OSError:
        return 1                # (no such descriptor to duplicate: write the line to fd 1 as it is)


def _run_child(cmd, timeout_s, env=None):
    """(return code, stdout, stderr) of a child interpreter in its own session; on a timeout the whole process group it
    started (the child and its forked pool workers) is killed and TimeoutExpired raised."""
    import signal
    proc = subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, start_new_session=True, env=env)
    try:
        out, err = proc.communicate(timeout=timeout_s)
        return proc.returncode, out, err
    except subprocess.TimeoutExpired:
        try:
            os.killpg(proc.pid, signal.SIGKILL)
        except ProcessLookupError:
            pass
        proc.communicate()
        raise


def cpu_baseline_child(timeout_s: float = 420.0, attempts: int = 2):
    """cpu_baseline_inline() in a child interpreter (`bench.py --cpu-baseline-only` prints its dict as one JSON line)."""
    why = "not run"
    for attempt in range(attempts):
        try:
            rc, out, err = _run_child([sys.executable, os.path.abspath(__file__), "--cpu-baseline-only"], timeout_s)
            if rc == 0:
                return json.loads(out.strip().splitlines()[-1])
            why = f"exit code {rc}: {err.strip()[-300:]}"
        except subprocess.TimeoutExpired:
            why = f"no result within {timeout_s:.0f} s"
        except Exception as e:
            why = f"{type(e).__name__}: {e}"
        _phase(f"cpu_baseline attempt {attempt + 1} failed: {why}")
    return {"value": None, "unit": UNIT, "cores": 0, "kind": "reference", "sample": "", "unavailable": why}


def configs0_frame():
    """10 000 synthetic 1-minute bars ending in a sell-off (the constant technical signal then trades, as in the parity
    fixtures tests/golden/bt_reference.*)."""
    import numpy as np
    import pandas as pd
    from ai_crypto_trader_b200 import synth
    n = 10_000
    d = synth.synth_symbol(1, n)
    f = np.ones(n)
    f[-60:] = np.linspace(1.0, 0.90, 60)
    cols = {k: d[k].astype(np.float64) * (f if k in ("open", "high", "low", "close") else 1.0) for k in synth.FIELDS}
    return pd.DataFrame({k: v.astype(np.float32).astype(np.float64) for k, v in cols.items()},
                        index=pd.date_range("2024-01-01", periods=n, freq="min"))



# --------------------------------------------------------------------------
# parity of the timed population, and the rest of BASELINE.json's metric
# --------------------------------------------------------------------------
def parity_spot_check(sweep, my_pop, ohlcv, minute0, lanes=64):
    """`lanes` (individual, symbol) lanes of the population that was just timed, spread over the shard and the symbols:
    record count and trade hash (every entry / exit bar and side) bit-exact, score rel 1e-9, against oracle/sim_oracle.c
    fed the float64-pandas RSI row (oracle/indicators_ref.py)."""
    import numpy as np
    from oracle import indicators_ref, sim_oracle
    stats = sweep.lane_stats()
    S = ohlcv.shape[1]
    cfg = sim_oracle.config_of(minute0, 1)
    idx = np.unique(np.linspace(0, len(my_pop) - 1, lanes).astype(int))
    rows, bad = {}, 0
    for j, i in enumerate(idx):
        s = j % S
        w = int(my_pop[i]["rsi_period"])
        if (s, w) not in rows:
            rows[(s, w)] = indicators_ref.rsi_bank(ohlcv[3, s], [w])[0]
        want, _, _ = sim_oracle.lane(ohlcv[3, s], rows[(s, w)], my_pop[i], cfg)
        got_score, want_score = float(stats["score"][i, s]), float(want["score"])
        same_score = (got_score == want_score or (np.isnan(got_score) and np.isnan(want_score))
                      or abs(got_score - want_score) <= 1e-9 * max(1.0, abs(want_score)))
        if int(stats["n_records"][i, s]) != int(want["n_records"]) or int(stats["trade_hash"][i, s]) != int(want["trade_hash"]) or not same_score:
            bad += 1
    return {"lanes_checked": int(len(idx)), "mismatches": int(bad),
            "what": "n_records + trade_hash bit-exact, score rel 1e-9 vs oracle/sim_oracle.c on the timed population (rank 0 shard)"}


def run_extras(args, world, rank, dev, sweep, population, pop_local, timed_sweeps, barrier, evals_per_step_global, out=None):
    """Keys beside the headline, every rank taking part (same collectives in the same order):
      evolved_population_value  configs[1] throughput on the generation-3 population of a GA run (the GA drives the
                                trade-record count, the sweep's cost driver, up)
      ga_generation_s           configs[4]: population 10 000 x 50 symbols x 1M bars, individuals STRONG-sharded over the
                                N ranks, one all-gather per generation, GA operators included
      evolution_c4_s            configs[3]: 100 generations, population 4096, 20 symbols x 1M bars, RSI on 1m / 5m / 15m
      mc_c3_ms                  configs[2]: 1M GBM paths x 10 000 steps sharded over the N ranks incl. gather + statistics"""
    import numpy as np
    import torch
    import torch.distributed as dist
    from ai_crypto_trader_b200 import synth
    from ai_crypto_trader_b200.dist import ShardedFitness, gather_paths, shard_bounds
    from ai_crypto_trader_b200.genetic_algorithm import DeviceGeneticAlgorithm, GeneticAlgorithm
    from ai_crypto_trader_b200.monte_carlo import PathEngine, risk_statistics
    from ai_crypto_trader_b200.sweep import MarketData, PopulationSweep, decode_population
    out = {} if out is None else out          # (the caller's dict: legs that finished survive a later one that stalls)

    def wall(fn):
        """fn() between two barriers; seconds, max over ranks."""
        barrier()
        t0 = time.perf_counter()
        r = fn()
        barrier()
        t = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item()), r

    # ---- configs[1] on an evolved population ---------------------------------------------------------
    _phase("extras: evolved population (configs[1], generation 3)")
    fit = ShardedFitness(sweep.evaluate, device=dev)
    ga = GeneticAlgorithm(synth.param_ranges(), fit, population_size=len(population), generations=3, random_seed=42)
    ga.run(seeded_individuals=population)              # reference operators (host), fitness = the sharded sweep
    evolved = ga.population
    mine = evolved[rank * pop_local:(rank + 1) * pop_local]
    indiv = torch.from_numpy(decode_population(mine, sweep.period_row).view(np.uint8)).to(dev)
    ms_total, ms_k, _, _ = timed_sweeps(indiv, None, sweep.plan(mine))
    records = float(sweep.lane_stats()["n_records"].sum())
    out["evolved_population_value"] = {
        "value": evals_per_step_global * args.steps / (ms_total * 1e-3), "unit": UNIT, "ms_per_step": ms_total / args.steps,
        "generation": 3, "records_rank0": records,
        "note": "same workload and timing as `value`, population = generation 3 of GeneticAlgorithm(seed 42) started from the timed random population"}

    # ---- configs[4]: one GA generation at population 10 000 x 50 symbols x 1M bars --------------------
    _phase("extras: configs[4] generation")
    S5, POP5, GENS = 50, 10_000, 3
    close = np.stack([synth.synth_symbol(s, args.bars)["close"] for s in range(S5)])
    market5 = MarketData.from_close(torch.from_numpy(close).to(dev))
    del close
    sweep5 = PopulationSweep(market5, mode=args.mode)
    fit5 = ShardedFitness(sweep5.evaluate, device=dev)
    ga5 = DeviceGeneticAlgorithm(synth.param_ranges(), fit5, population_size=POP5, generations=GENS, random_seed=42)
    ga5.initialize_population()
    lo, hi, _ = shard_bounds(POP5, world, rank)
    ga5.evaluate_population()                          # untimed: workspace allocation, zone map (built on the second sweep)
    ga5.evaluate_population()
    gen_s, sweep_s = [], []
    for gen in range(GENS + 1):
        def one_generation():
            t0 = time.perf_counter()
            ga5.evaluate_population()                  # this rank's shard through the sweep + the all-gather
            torch.cuda.synchronize()
            t1 = time.perf_counter()
            ga5.evolve_generation(gen + 1)             # selection / crossover / mutation (device, Philox)
            torch.cuda.synchronize()
            return t1 - t0
        t, ts = wall(one_generation)
        gen_s.append(t)
        sweep_s.append(ts)
    out["ga_generation_s"] = {
        "random": gen_s[0], "gen3": gen_s[GENS], "per_generation": gen_s, "fitness_sweep_s_rank0": sweep_s,
        "population": POP5, "symbols": S5, "bars": args.bars, "individuals_per_rank": hi - lo,
        "what": "wall seconds of one generation = fitness of every individual (sharded sweep, one all-gather of 8 B per individual) + GA operators (DeviceGeneticAlgorithm), barrier on both sides, max over ranks",
        "scaling": "strong"}
    del ga5, fit5, sweep5, market5
    torch.cuda.empty_cache()

    # ---- configs[3]: the evolution loop, 100 generations, population 4096, 20 symbols, RSI on 1m / 5m / 15m -------------
    _phase("extras: configs[3] evolution loop")
    import importlib.util
    spec = importlib.util.spec_from_file_location("evolution_c4", str(ROOT / "tools" / "evolution_c4.py"))
    c4mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(c4mod)
    c4 = c4mod.run(generations=100, population=4096, symbols=20, bars=args.bars, device=dev)
    out["evolution_c4_s"] = {k: c4[k] for k in ("loop_s", "per_generation_s", "setup_s", "bank_rows", "operators", "best_fitness",
                                                "distinct_individuals_rank0", "evaluations_computed_rank0", "evaluations_nominal", "workload")}
    out["evolution_c4_s"]["scaling"] = "strong"
    out["evolution_c4_s"]["what"] = ("wall seconds of the whole loop (initial population + 100 generations: GA operators on the device, fitness = "
                                     "sharded sweep over the 78-row multi-timeframe bank, one all-gather per generation); max over ranks")
    torch.cuda.empty_cache()

    # ---- configs[2]: Monte-Carlo risk, 1M GBM paths x 10 000 steps, VaR + max drawdown ------------------
    _phase("extras: configs[2] Monte-Carlo")
    n_paths, steps = 1_000_000, 10_000
    eng = PathEngine()
    ret = np.random.default_rng(7).normal(5e-4, 0.02, 60)
    mu, sigma = float(np.mean(ret) * 252), float(np.std(ret, ddof=1) * np.sqrt(252))      # monte_carlo_service.py:243-244
    plo, phi, _ = shard_bounds(n_paths, world, rank)

    def mc_job():
        f, d, _ = eng.gbm(100.0, mu, sigma, 1 / 252, phi - plo, steps, 2024, path_offset=plo)
        f, d = gather_paths(f, d, n_paths)
        return risk_statistics(eng, f, d, 100.0, 0.95)
    mc_job()
    reps = 3
    t, st = wall(lambda: [mc_job() for _ in range(reps)][-1])
    out["mc_c3_ms"] = {"value": 1e3 * t / reps, "path_steps_per_s": n_paths * steps / (t / reps), "paths": n_paths, "steps": steps,
                       "var_pct": abs(st["var"]), "mdd_mean": st["mdd_mean"], "mu": mu, "sigma": sigma, "dt": 1 / 252, "scaling": "strong",
                       "what": "paths sharded by rank (Philox keyed by the global path index), one all-gather of finals + drawdowns, exact radix-select percentiles and moments on every rank; wall ms per run, max over ranks"}
    return out


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir: str, fitness, stats) -> None:
    """What the timed path hands its caller after its last step, one float64 .npy per array: the fitness vector [individual]
    and the lane stats [individual][symbol] of this rank's shard (trade_hash, a uint64, as its exact high and low 32-bit
    halves).  Every value written is finite: an array holding inf or nan (the reference's Sortino ratio is +inf when a lane
    has no downside deviation) is written with those entries as 0, and beside it <name>_nonfinite codes them as +1 (+inf),
    -1 (-inf) or 2 (nan), 0 elsewhere.  Above DUMP_LIMIT_BYTES in all, a fixed seeded sample of individuals is written,
    their indices in lane_index."""
    import numpy as np
    arrays = {"fitness": fitness}
    for name, a in stats.items():
        if name == "trade_hash":
            arrays["trade_hash_hi"], arrays["trade_hash_lo"] = a >> np.uint64(32), a & np.uint64(0xFFFFFFFF)
        else:
            arrays[name] = a
    for name, a in list(arrays.items()):
        a = np.asarray(a, dtype=np.float64)
        if not np.isfinite(a).all():
            arrays[name + "_nonfinite"] = np.where(np.isnan(a), 2.0, np.where(np.isinf(a), np.sign(a), 0.0))
            arrays[name] = np.where(np.isfinite(a), a, 0.0)
    pop = len(fitness)
    bytes_per_individual = 8 * (1 + sum(a.size // pop for a in arrays.values()))      # (+1: the lane_index entry)
    if pop * bytes_per_individual > DUMP_LIMIT_BYTES:
        idx = np.sort(np.random.default_rng(0).choice(pop, DUMP_LIMIT_BYTES // bytes_per_individual, replace=False))
        arrays = {name: a[idx] for name, a in arrays.items()}
        arrays["lane_index"] = idx
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.asarray(a, dtype=np.float64))


def _positive_int(text: str) -> int:
    n = int(text)
    if n < 1:
        raise argparse.ArgumentTypeError(f"must be at least 1, got {n}")
    return n


# --------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=_positive_int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--pop-per-gpu", type=int, default=POP_PER_GPU)
    ap.add_argument("--symbols", type=int, default=N_SYMBOLS)
    ap.add_argument("--bars", type=int, default=N_BARS)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--skip-extras", action="store_true", help="only the headline (configs[1]) legs")
    ap.add_argument("--cpu-baseline-only", action="store_true", help="(internal) print the cpu_baseline dict and exit")
    ap.add_argument("--reference-child", action="store_true", help="(internal) the worker of --impl reference")
    ap.add_argument("--mode", default="auto", choices=["auto", "fused", "chunked", "tiled"], help="sweep kernel path (auto = product default)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the fitness and lane stats of the last timed step as DIR/<name>.npy")
    args = ap.parse_args()
    if args.cpu_baseline_only:
        print(json.dumps(cpu_baseline_inline()), flush=True)
        return
    if args.impl == "reference":
        if args.reference_child or int(os.environ.get("RANK", "0")) != 0:
            run_reference_arm(args)
            return
        # the pool of forked workers runs in a child interpreter with a deadline (see cpu_baseline_child)
        why = "not run"
        for attempt in range(2):
            try:
                rc, out, err = _run_child([sys.executable, os.path.abspath(__file__), "--impl", "reference", "--reference-child", "--gpus", str(args.gpus),
                                           "--steps", str(args.steps), "--warmup", str(args.warmup)], 900, env=dict(os.environ, RANK="0"))
                if rc == 0 and out.strip():
                    print(out.strip().splitlines()[-1], flush=True)
                    return
                why = f"exit code {rc}: {err.strip()[-300:]}"
            except subprocess.TimeoutExpired:
                why = "no result within 900 s"
            _phase(f"reference arm attempt {attempt + 1} failed: {why}")
        print(json.dumps({"impl": "reference", "unavailable": why}), flush=True)
        return
    assert args.warmup >= 3 or os.environ.get("B200BT_ALLOW_SHORT_WARMUP"), "timing rules: warm-up >= 3"
    result_fd = _claim_stdout()
    # A stalled run must end with a traceback, not with the caller's patience: every thread's stack goes to stderr.
    import faulthandler
    faulthandler.dump_traceback_later(int(os.environ.get("B200BT_BENCH_WATCHDOG_S", 1500)), exit=True)
    # CPU baseline first (rank 0, N=1 only), in a child process of its own (a pool of forked workers; no CUDA in it) with a
    # deadline: a CPU leg that stalls costs the run its cpu_baseline key, not its result
    cpu_baseline = None
    if int(os.environ.get("WORLD_SIZE", "1")) == 1 and not args.no_cpu_baseline:
        _phase("cpu_baseline (child process)")
        cpu_baseline = cpu_baseline_child()

    import numpy as np
    import torch
    import torch.distributed as dist
    from ai_crypto_trader_b200 import _lib, synth
    from ai_crypto_trader_b200.sweep import MarketData, PopulationSweep, decode_population, evaluation_order

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    assert world == args.gpus, f"--gpus {args.gpus} but WORLD_SIZE={world} (launch with torch.distributed.run for N>1)"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")     # stdout carries the JSON line and nothing else
        dist.init_process_group("nccl", device_id=dev)

    pop_local, S, N = args.pop_per_gpu, args.symbols, args.bars
    pop_global = pop_local * world
    # synthetic market, identical on every rank (replicated), pinned on the host for the e2e leg
    ohlcv_host = torch.from_numpy(synth.synth_ohlcv(S, N)).pin_memory()
    market = MarketData(ohlcv_host)
    sweep = PopulationSweep(market, mode=args.mode)
    population = synth.random_population(pop_global, seed=42)
    my_pop = population[rank * pop_local:(rank + 1) * pop_local]
    packed = decode_population(my_pop, sweep.period_row)
    order = evaluation_order(my_pop)
    indiv_dev = torch.from_numpy(packed.view(np.uint8)).to(dev)
    order_dev = torch.from_numpy(order).to(dev)
    fit_local = torch.empty(pop_local, dtype=torch.float64, device=dev)
    fit_global = torch.empty(pop_global, dtype=torch.float64, device=dev)
    plan = sweep.plan(my_pop)          # the path sweep.evaluate() takes: None = fused kernel, else tile / chunk plans
    path = "fused" if plan is None else ("tiled" if type(plan[0]).__name__ == "TilePlan" else "chunked")
    path_kernels = {"fused": "sweep_kernel", "chunked": "chunk_scan_kernel + chunk_sums/partial/lane_combine",
                    "tiled": "lane_scan_kernel + chunk_sums/partial/lane_combine"}[path]
    # DRAM bytes (read + write) of the dominant kernel per launch on THIS workload, from the committed
    # `ncu --set full` captures (profiles/r1_tiled_final_ncu.txt, r1_chunk_scan_ncu.txt, r1_sweep_v2_ncu.txt);
    # null for any other workload size
    ncu_traffic = {"tiled": 5.222e9 + 1.006e9, "chunked": 45.6e9, "fused": 3.3e9}[path] \
        if (pop_local, S, N) == (POP_PER_GPU, N_SYMBOLS, N_BARS) else None

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed_sweeps(indiv, order_d, pl, sample_clocks=False):
        """W warm-up + K timed generations of this rank's shard (sweep + fitness reduce [+ all-gather]), device-resident.
        -> (ms for the K steps, max over ranks; mean ms of the sweep kernels alone; launches; clocks or None)"""
        def one():
            sweep.evaluate_device(indiv, order_d, pop_local, fit_local, plan=pl)
            if world > 1:
                dist.all_gather_into_tensor(fit_global, fit_local)
        for _ in range(args.warmup):
            one()
        barrier()
        sampler = ClockSampler(local_rank) if (sample_clocks and rank == 0) else None
        if sampler:
            sampler.start()
            time.sleep(0.25)
        barrier()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        k_ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
        # the dominant kernel (lane_scan_kernel) is bracketed by its own pair of events, recorded by the library on the
        # stream it launches on (b200bt_sweep_scan_timing); a first record() makes torch create the cudaEvent_t
        s_ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
        for a, b in s_ev:
            a.record(); b.record()
        handle = lambda e: (e.cuda_event.value if hasattr(e.cuda_event, "value") else int(e.cuda_event))
        lib = _lib.load()
        launches0 = _lib.launch_count()
        t_wall0 = time.time()
        ev0.record()
        for i in range(args.steps):
            # the sweep (scan, verify / repair, metrics, fitness reduction) is bracketed by its own events inside the
            # timed region; the all-gather follows
            lib.b200bt_sweep_scan_timing(handle(s_ev[i][0]), handle(s_ev[i][1]))
            k_ev[i][0].record()
            sweep.evaluate_device(indiv, order_d, pop_local, fit_local, plan=pl)
            k_ev[i][1].record()
            if world > 1:
                dist.all_gather_into_tensor(fit_global, fit_local)
        ev1.record()
        barrier()
        t_wall1 = time.time()
        n_launch = _lib.launch_count() - launches0
        t = torch.tensor([ev0.elapsed_time(ev1)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        lib.b200bt_sweep_scan_timing(None, None)
        ms_k = statistics.mean(a.elapsed_time(b) for a, b in k_ev)
        scan = [a.elapsed_time(b) for a, b in s_ev]
        timed_sweeps.scan_ms = statistics.mean(scan) if min(scan) > 1e-3 else None     # (None: the plan has no scan kernel)
        return float(t.item()), ms_k, n_launch, (sampler.stop(t_wall0, t_wall1) if sampler else None)

    # ---- device-resident leg ------------------------------------------------
    _phase("timed sweeps (device-resident)")
    ms_total, ms_kernel, launches, clocks = timed_sweeps(indiv_dev, order_dev, plan, sample_clocks=True)
    scan_ms_live = timed_sweeps.scan_ms
    evals_per_step_global = pop_global * S * N
    value = evals_per_step_global * args.steps / (ms_total * 1e-3)
    fit_random = fit_local.clone()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, fit_random.cpu().numpy(), sweep.lane_stats())

    # ---- parity spot check of the timed population (rank 0): 64 lanes against the C oracle ----
    parity = None
    _phase("parity spot check")
    if rank == 0:
        parity = parity_spot_check(sweep, my_pop, ohlcv_host.numpy(), market.minute0, lanes=64)

    # ---- end-to-end leg: host OHLCV + host population in, host fitness out ----
    def e2e_step():
        mk = MarketData(ohlcv_host)                      # H2D of the pinned OHLCV (5 fields)
        sw = PopulationSweep(mk, mode=args.mode)         # RSI bank on device
        f = sw.evaluate(my_pop)                          # H2D params, sweep, reduce, D2H fitness
        if world > 1:
            g = torch.from_numpy(f).to(dev)
            out = torch.empty(pop_global, dtype=torch.float64, device=dev)
            dist.all_gather_into_tensor(out, g)
            f = out.cpu().numpy()
        return f, sw.h2d_bytes + mk.h2d_bytes, sw.d2h_bytes    # (the sweep reads close prices: the other OHLCV fields stay on the host)

    e2e_steps = args.steps
    _phase("end-to-end leg")
    f_e2e, h2d, d2h = e2e_step()
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        f_e2e, h2d, d2h = e2e_step()
    barrier()
    e2e_s = time.perf_counter() - t0
    te = torch.tensor([e2e_s], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e_value = evals_per_step_global * e2e_steps / float(te.item())

    # sanity: the e2e result equals the device-resident result
    assert np.allclose(f_e2e[rank * pop_local:(rank + 1) * pop_local] if world > 1 else f_e2e,
                       fit_random.cpu().numpy(), rtol=1e-12, atol=0, equal_nan=True)

    # ---- the rest of the metric: evolved population, configs[4] generation wall time, configs[2] Monte-Carlo ----
    # (under a deadline: the headline above is complete at this point, and a leg beside it that stalls -- on any rank: the
    # legs are collective -- must not take the line with it; the thread is abandoned and the process leaves through os._exit)
    extras, abandoned = {}, False
    if not args.skip_extras:
        box = {}

        def _extras():
            torch.cuda.set_device(local_rank)
            run_extras(args, world, rank, dev, sweep, population, pop_local, timed_sweeps, barrier, evals_per_step_global, out=box.setdefault("partial", {}))
            box["out"] = box["partial"]
        th = threading.Thread(target=_extras, daemon=True)
        th.start()
        th.join(float(os.environ.get("B200BT_BENCH_EXTRAS_S", 600)))
        if th.is_alive() or "out" not in box:
            abandoned = True
            extras = dict(box.get("partial", {}))
            extras["extras_unavailable"] = f"the legs beside the headline did not finish within their deadline (last phase: {_LAST_PHASE[0]})"
            _phase("extras abandoned")
            faulthandler.dump_traceback(file=sys.stderr, all_threads=True)
        else:
            extras = box["out"]

    if rank == 0:
        peak, peak_src = measured_hbm_peak()
        lanes_evals = pop_local * S * N
        algorithmic_gbps = lanes_evals * BYTES_PER_EVAL / (ms_kernel * 1e-3) / 1e9
        # What binds the sweep is instruction issue, not HBM (profiles/: DRAM 10-15 % of peak, issue slots ~60 % busy,
        # the RSI rows are shared by every lane of a symbol so most of SURVEY 8(d)'s 8 B/eval never leaves L1/L2).
        # The roofline is therefore stated against the issue rate: warp-instructions of the dominant kernel per launch
        # (ncu, committed under profiles/, valid for exactly this workload) / its share of the live kernel time, against
        # 148 SMs x 4 schedulers x the SM clock sampled during the timed region.
        ncu = NCU_C2.get(path) if (pop_local, S, N) == (POP_PER_GPU, N_SYMBOLS, N_BARS) else None
        sm_mhz = (clocks or {}).get("sm_mhz") or 1965.0
        issue_peak = 148 * 4 * sm_mhz * 1e6 / 1e9                     # G warp-instructions / s
        roofline = {"bound": "issue", "kernel": path_kernels, "sweep_mode": path, "kernel_ms": ms_kernel,
                    "peak": issue_peak, "unit": "Ginst/s", "peak_source": f"148 SMs x 4 warp schedulers x {sm_mhz:.0f} MHz (sampled under load)",
                    "algorithmic_gbps": algorithmic_gbps, "bytes_per_eval": BYTES_PER_EVAL,
                    "hbm_peak_gbs": peak, "hbm_peak_source": peak_src}
        if ncu:
            scan_ms = scan_ms_live if scan_ms_live else ms_kernel * ncu["scan_share"]
            achieved = ncu["warp_inst"] / (scan_ms * 1e-3) / 1e9
            roofline.update({
                "achieved": achieved, "frac": achieved / issue_peak,
                "warp_inst_per_launch": ncu["warp_inst"], "warp_inst_per_eval": ncu["warp_inst"] / lanes_evals,
                "threads_per_inst": ncu["threads_per_inst"], "dominant_kernel_ms": scan_ms,
                "dominant_kernel_share_of_step": scan_ms / ms_kernel, "dominant_kernel_share_in_launch_list": ncu["scan_share"],
                "issue_active_pct_ncu": ncu["issue_active_pct"], "alu_pipe_pct_ncu": ncu["alu_pipe_pct"],
                "traffic": ncu["dram_bytes"], "traffic_unit": "DRAM bytes per launch of the dominant kernel (ncu dram__bytes_read.sum + dram__bytes_write.sum)",
                "dram_frac": ncu["dram_bytes"] / (scan_ms * 1e-3) / 1e9 / peak, "compulsory_bytes": (S * N * 4 + sweep.bank.numel() * 4),
                "source": ncu["source"],
                "note": "achieved = warp-instructions of lane_scan_kernel per launch (ncu, this workload) / its mean duration in the timed region (CUDA events recorded by the library around the kernel, on its stream); algorithmic_gbps = SURVEY 8(d)'s 8 B x evals / kernel time, a throughput figure, not a bound"})
        else:
            roofline.update({"achieved": None, "frac": None, "traffic": None,
                             "note": "no committed ncu capture for this workload size: only the algorithmic throughput is reported"})
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_total / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32 streams / f64 trade arithmetic", "data": "synthetic",
            "config": {"workload": f"GA fitness sweep (BASELINE configs[1] per GPU): population {pop_local}/GPU x {S} symbols x {N} 1-min bars, reference RSI rule",
                       "global_population": pop_global, "symbols": S, "bars": N, "parallelism": f"individuals sharded x{world}, market replicated, 1 all-gather/generation" if world > 1 else "single GPU",
                       "population": "GeneticAlgorithm.initialize_population draw, seed 42 (see evolved_population_value for generation 3)",
                       "l2_policy": "inputs larger than L2 (price+RSI bank = %.2f GB per GPU)" % ((S * N * 4 + sweep.bank.numel() * 4) / 1e9)},
            "roofline": roofline,
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                    "steps": e2e_steps, "path": "MarketData(pinned host OHLCV; close prices uploaded, the fields the sweep does not read stay on the host) -> PopulationSweep (RSI bank) -> evaluate(list of dicts) -> host fitness"},
            "gpu_launches": int(launches), "gpu_launches_per_step": launches / args.steps,
            "parity": parity,
            "clocks": clocks,
        }
        line.update(extras)
        if cpu_baseline is not None:
            if "configs0_backtest" in cpu_baseline and not abandoned:
                # the same configs[0] backtest through the GPU path (indicators, backtest_ref kernel, stats dict)
                import asyncio
                import tempfile
                from ai_crypto_trader_b200.backtesting import HistoricalDataManager, StrategyTester
                df0 = configs0_frame()
                with tempfile.TemporaryDirectory(prefix="b200bt_bench_") as scratch:      # (the source tree may be read-only)
                    tester = StrategyTester(config={}, data_manager=HistoricalDataManager(None, data_dir=os.path.join(scratch, "data")),
                                            results_dir=os.path.join(scratch, "results"), config_path=None)
                    asyncio.run(tester.backtest_frame(df0, "SYNUSDC"))
                    t0 = time.perf_counter()
                    st0 = asyncio.run(tester.backtest_frame(df0, "SYNUSDC"))
                    cpu_baseline["configs0_backtest"]["gpu_path_ms"] = (time.perf_counter() - t0) * 1e3
                cpu_baseline["configs0_backtest"]["gpu_trades"] = int(st0["total_trades"])
            line["cpu_baseline"] = cpu_baseline
        payload = (json.dumps(line) + "\n").encode()
        try:
            while payload:
                payload = payload[os.write(result_fd, payload):]
        except OSError:
            sys.__stdout__.write(payload.decode())
            sys.__stdout__.flush()
    _phase("done")
    faulthandler.cancel_dump_traceback_later()
    if abandoned:
        sys.stdout.flush()
        os._exit(0)          # (a thread is still inside a CUDA / NCCL call)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
