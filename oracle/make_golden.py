"""ORACLE (test infrastructure): regenerate ``tests/golden/reference_modules.npz``.

Runs the REFERENCE's own ``crossmodal`` package (imported, read-only and never copied, from a checkout
of brentyi/multimodalfilter named by the environment variable ``MMF_REFERENCE_DIR``) on CPU on top of
the oracle's ``torchfilter`` / ``fannypack`` shims, over the cases in ``oracle/golden_cases.py``.  The
reference is not part of this repository, so the outputs are committed as a small fixture; inputs and
parameters are re-derived from seeds where the fixture is checked.

What this pins: every row of SURVEY.md section 8a that has a ``ref:`` line range in the
reference repo itself (R3, R4, R5, R9, R10, R11, R12 -- architectures + fusion math, run by the
reference's code).  What it cannot pin: the torchfilter recursion underneath (R1, R2, R6, R7, R8),
which in this process is the oracle's own restatement -- PARITY UNPINNED there.

Usage:  MMF_REFERENCE_DIR=<checkout of the reference> python -m oracle.make_golden
"""
import importlib
import os
import sys
import warnings

import numpy as np

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REFERENCE = os.environ.get("MMF_REFERENCE_DIR", "")
OUT = os.path.join(REPO, "tests", "golden", "reference_modules.npz")


def reference_available() -> bool:
    """True when MMF_REFERENCE_DIR names a checkout of the reference (its ``crossmodal`` package)."""
    return bool(REFERENCE) and os.path.isdir(os.path.join(REFERENCE, "crossmodal"))


def reference_resolver():
    import oracle

    oracle.install_shims()
    if REFERENCE not in sys.path:
        sys.path.insert(1, REFERENCE)
    warnings.filterwarnings("ignore")  # torch.cholesky deprecation inside the reference
    modules = [
        importlib.import_module(m)
        for m in (
            "crossmodal.base_models",
            "crossmodal.push_models",
            "crossmodal.door_models",
            "crossmodal.push_models.dynamics",
            "crossmodal.door_models.dynamics",
        )
    ]

    def resolve(name):
        for mod in modules:
            if hasattr(mod, name):
                cls = getattr(mod, name)
                assert cls.__module__.startswith("crossmodal."), cls.__module__
                return cls
        raise KeyError(name)

    return resolve


def main():
    if not reference_available():
        raise SystemExit("MMF_REFERENCE_DIR does not name a checkout of the reference; the committed fixture stays as is")
    sys.path.insert(0, REPO)
    from oracle.golden_cases import run_all

    cases = run_all(reference_resolver(), device="cpu")
    os.makedirs(os.path.dirname(OUT), exist_ok=True)
    np.savez_compressed(OUT, **cases)
    size = os.path.getsize(OUT)
    print(f"wrote {OUT}: {len(cases)} arrays, {size / 1024:.1f} KiB")
    for key in sorted(cases):
        print(f"  {key:70s} {cases[key].shape}")


if __name__ == "__main__":
    main()
