"""Is the REAL reference stack importable on this box?  pinocchio (pin>=3.3.1) + nlopt (nlopt>=2.8.0) + the reference package
(baseline/_ref, the source directory named by DEX_RETARGETING_REFERENCE, or site-packages).  Used by tests/test_real_reference.py and by
`bench.py --impl reference`, which prefers the real thing (`kind: "reference"`) over the oracle's restated path (`"port"`)."""
import importlib
import os
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent


def probe():
    found = {}
    for name in ("pinocchio", "nlopt"):
        try:
            m = importlib.import_module(name)
            found[name] = getattr(m, "__version__", "unknown")
        except Exception:
            found[name] = None
    found["reference"] = None
    if found["pinocchio"] and found["nlopt"]:
        for cand in (os.environ.get("DEX_RETARGETING_REFERENCE"), ROOT / "baseline" / "_ref", None):
            if cand is not None and not (Path(cand) / "dex_retargeting").exists():
                continue
            if cand is not None:
                sys.path.insert(0, str(cand))
            try:
                importlib.import_module("dex_retargeting.seq_retarget")
                found["reference"] = str(cand) if cand is not None else "site-packages"
                break
            except Exception:
                if cand is not None:
                    sys.path.remove(str(cand))
    return found
