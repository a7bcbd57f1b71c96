"""Copy the UNMODIFIED reference scripts (pure Python, no build step: there is no setup.py to pip-install) into the
git-ignored oracle/_ref/, so that oracle/gen_reference_runs.py can run them on any GPU host that has a copy of this repository.

    python oracle/fetch_reference.py <reference checkout>      # or NERF_REFERENCE=<reference checkout>

Nothing in the product, the tests or bench.py reads oracle/_ref/; the tests read what the generators stored in tests/golden/."""
import os
import shutil
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DST = os.path.join(ROOT, "oracle", "_ref")


def fetch(src, verbose=True):
    if not os.path.isfile(os.path.join(src, "run_nerf.py")):
        return False
    os.makedirs(DST, exist_ok=True)
    for f in sorted(os.listdir(src)):
        if f.endswith(".py"):
            shutil.copy2(os.path.join(src, f), os.path.join(DST, f))
    os.makedirs(os.path.join(DST, "configs"), exist_ok=True)
    for f in sorted(os.listdir(os.path.join(src, "configs"))):
        shutil.copy2(os.path.join(src, "configs", f), os.path.join(DST, "configs", f))
    if verbose:
        print("[fetch_reference] copied", sorted(os.listdir(DST)))
    return True


if __name__ == "__main__":
    src = sys.argv[1] if len(sys.argv) > 1 else os.environ.get("NERF_REFERENCE", "")
    sys.exit(0 if fetch(src) else 1)
