"""Recipe for oracle/_ref/: the reference's OWN hot-path modules, placed (not committed) next to the oracle so that the
CPU baseline legs of bench.py can time the real `_simulate_trades` / `calculate_metrics` / `_calculate_strategy_score`
(services/strategy_evaluation.py:746-878, :32-228, :579-633) and the real `GeneticAlgorithm` operators
(services/genetic_algorithm.py:135-252) on the GPU box, where /root/reference does not exist.

TEST / MEASUREMENT INFRASTRUCTURE.  oracle/_ref/ is git-ignored (no reference source enters the history) and NOT
gpurun-ignored, so it travels to the GPU box with the snapshot like the built .so files.  `__graft_entry__.build()` runs
this in the build container; on the GPU box the placed files are used as they are.  The modules are Python (the reference
has no compiled code), so "building" the reference is placing these files unmodified; `load()` imports them with
matplotlib stubbed (used for plots only) and with the cwd-relative paths the modules open at import time
(`logs/*.log`, `config.json`; strategy_evaluation.py:23,513) provided in a scratch directory.
"""
from __future__ import annotations

import os
import shutil
import sys
import types
from pathlib import Path

HERE = Path(__file__).resolve().parent
REF_DIR = HERE / "_ref"
REFERENCE_ROOT = Path(os.environ.get("B200BT_REFERENCE_ROOT", "/root/reference"))
FILES = ("services/strategy_evaluation.py", "services/genetic_algorithm.py", "config.json")


def place(force: bool = False) -> bool:
    """Copy FILES from the reference tree into oracle/_ref/ (build container).  -> True when oracle/_ref is complete."""
    if os.access(REFERENCE_ROOT / FILES[0], os.R_OK):     # (absent, or not readable by this user: nothing to place)
        for rel in FILES:
            dst = REF_DIR / rel
            if force or not dst.exists() or dst.stat().st_mtime < (REFERENCE_ROOT / rel).stat().st_mtime:
                dst.parent.mkdir(parents=True, exist_ok=True)
                shutil.copyfile(REFERENCE_ROOT / rel, dst)
    return available()


def available() -> bool:
    return all((REF_DIR / rel).exists() for rel in FILES)


_loaded = None


def load():
    """(StrategyEvaluationSystem instance, StrategyPerformanceMetrics class, GeneticAlgorithm class) of the reference,
    imported from oracle/_ref with its numeric code unmodified."""
    global _loaded
    if _loaded is not None:
        return _loaded
    if not available():
        raise RuntimeError("oracle/_ref is not populated (run oracle/make_ref.py where /root/reference exists)")
    import tempfile
    for name in ("matplotlib", "matplotlib.pyplot"):
        if name not in sys.modules:
            sys.modules[name] = types.ModuleType(name)
    sys.modules["matplotlib"].pyplot = sys.modules["matplotlib.pyplot"]
    scratch = Path(tempfile.mkdtemp(prefix="b200bt_ref_local_"))
    (scratch / "logs").mkdir()
    shutil.copy(REF_DIR / "config.json", scratch / "config.json")
    old = os.getcwd()
    os.chdir(scratch)                 # the modules open logs/*.log and config.json relative to the cwd
    sys.path.insert(0, str(REF_DIR))
    try:
        import importlib
        for m in ("services", "services.strategy_evaluation", "services.genetic_algorithm"):
            sys.modules.pop(m, None)
        se = importlib.import_module("services.strategy_evaluation")
        ga = importlib.import_module("services.genetic_algorithm")
        import logging
        logging.getLogger("strategy_evaluation").setLevel(logging.ERROR)    # (the per-call INFO lines go to a file)
        logging.getLogger("genetic_algorithm").setLevel(logging.ERROR)
        ses = se.StrategyEvaluationSystem("config.json")
    finally:
        sys.path.remove(str(REF_DIR))
        os.chdir(old)
    _loaded = (ses, se.StrategyPerformanceMetrics, ga.GeneticAlgorithm)
    return _loaded


if __name__ == "__main__":
    print("oracle/_ref complete:", place(force="--force" in sys.argv))
