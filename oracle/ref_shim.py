"""Import the LIVE reference as a checker.  TEST INFRASTRUCTURE ONLY.

The reference is a checkout of the original project (AIflowerQ/InvPref_KDD_2022, with its ``dataset/``) placed at
``oracle/_ref`` (git-ignored: its sources are not part of this repository) or named by ``INVPREF_REFERENCE_ROOT``.
Where it is absent the tests that use it skip, so nothing that must run everywhere (``-m gpu`` tests, ``smoke()``,
``bench.py``) may call this.  ``matplotlib`` / ``seaborn``, which the reference's ``utils.py:4-5`` imports, are
stubbed with empty modules where they are not installed (SURVEY.md §8c).
"""
from __future__ import annotations

import contextlib
import io
import os
import sys
import types

REF_ROOT = os.environ.get("INVPREF_REFERENCE_ROOT",
                          os.path.join(os.path.dirname(os.path.abspath(__file__)), "_ref"))


def available() -> bool:
    return os.path.isfile(os.path.join(REF_ROOT, "models.py"))


def load():
    """Returns the reference modules (models, train, functions, utils, dataloader, evaluate) imported under
    private names so they never shadow the product package's modules."""
    if not available():
        raise RuntimeError(f"reference checkout not found at {REF_ROOT}")
    for name in ("matplotlib", "matplotlib.pyplot", "seaborn"):
        if name not in sys.modules:
            try:
                __import__(name)
            except Exception:
                mod = types.ModuleType(name)
                sys.modules[name] = mod
    if "matplotlib" in sys.modules and "matplotlib.pyplot" in sys.modules:
        setattr(sys.modules["matplotlib"], "pyplot", sys.modules["matplotlib.pyplot"])
    saved = {k: sys.modules.get(k) for k in
             ("models", "train", "functions", "utils", "evaluate", "dataloader", "global_config")}
    sys.path.insert(0, REF_ROOT)
    try:
        for k in saved:
            sys.modules.pop(k, None)
        import importlib
        mods = {k: importlib.import_module(k) for k in ("functions", "utils", "models", "dataloader", "evaluate",
                                                        "train")}
    finally:
        sys.path.remove(REF_ROOT)
        for k in list(saved):
            cur = sys.modules.pop(k, None)
            if cur is not None:
                sys.modules["_invpref_ref_" + k] = cur
            if saved[k] is not None:
                sys.modules[k] = saved[k]
    return types.SimpleNamespace(**mods)


class NullEvaluator:
    """Stands in for the reference evaluators (evaluate.py:59-212), which are off the hot path."""

    def evaluate(self):
        return {"mse": 0.0, "rmse": 0.0, "mae": 0.0}


@contextlib.contextmanager
def quiet():
    with contextlib.redirect_stdout(io.StringIO()):
        yield
