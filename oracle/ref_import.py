"""Import the UNMODIFIED reference on CPU, for the golden-fixture generators only.

The reference is read from $NERF_REFERENCE, else from the git-ignored copy oracle/_ref/ (oracle/fetch_reference.py).
imageio / matplotlib are not installed and only used by I/O code paths, so empty module stubs
are registered first (SURVEY.md 8c).  No test, smoke() or bench.py calls this; it exists to pin
the oracle and to generate tests/golden/.
"""
import os
import sys
import types

REF = os.environ.get("NERF_REFERENCE", os.path.join(os.path.dirname(os.path.abspath(__file__)), "_ref"))


def available():
    return os.path.isfile(os.path.join(REF, "run_nerf.py"))


def load():
    for name in ("imageio", "matplotlib", "matplotlib.pyplot"):
        if name not in sys.modules:
            try:
                __import__(name)
            except Exception:
                sys.modules[name] = types.ModuleType(name)
    if REF not in sys.path:
        sys.path.insert(0, REF)
    import run_nerf            # noqa
    import run_nerf_helpers    # noqa
    return run_nerf, run_nerf_helpers
