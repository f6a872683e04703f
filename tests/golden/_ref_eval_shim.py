"""Import the reference's own evaluation utilities (src/util/metric.py, src/util/alignment.py) from /root/reference as
plain modules. Only usable where the reference checkout exists; used by make_eval_golden.py to produce the committed
fixture. metric.py imports pandas (for its MetricTracker), which must be installed."""
import importlib.util
import sys
from pathlib import Path

REF = Path("/root/reference")


def load_reference_eval_utils():
    if not REF.exists():
        raise RuntimeError("/root/reference is not available (fixtures are generated where the reference is checked out)")
    mods = {}
    for name in ("metric", "alignment"):
        spec = importlib.util.spec_from_file_location(f"refsrc_util_{name}", REF / "src" / "util" / f"{name}.py")
        m = importlib.util.module_from_spec(spec)
        sys.modules[spec.name] = m
        spec.loader.exec_module(m)
        mods[name] = m
    return mods
