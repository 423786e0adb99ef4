"""Re-runs every golden generator in this directory against the UNMODIFIED reference (/root/reference under
oracle/ref_shims.py) and compares the regenerated arrays with the committed ones, bit for bit.  Build container only
(takes about ten minutes; the committed files are restored afterwards whatever the outcome).

    python tests/golden/check_reproducible.py            # all generators
    python tests/golden/check_reproducible.py make_golden_gn make_golden_misc
"""
import glob
import os
import shutil
import subprocess
import sys
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
GENERATORS = ["make_golden_misc", "make_golden_gn", "make_golden_io", "make_golden_chain", "make_golden_loss",
              "make_golden_next", "make_golden", "make_golden_dropin"]


def same(x, y):
    if x.shape != y.shape or x.dtype != y.dtype:
        return False
    return bool(np.array_equal(x, y, equal_nan=True) if x.dtype.kind in "fc" else np.array_equal(x, y))


def main():
    gens = sys.argv[1:] or GENERATORS
    backup = tempfile.mkdtemp(prefix="golden_backup_")
    files = sorted(glob.glob(os.path.join(HERE, "*.npz")))
    for f in files:
        shutil.copy2(f, backup)
    bad = total = 0
    try:
        for g in gens:
            r = subprocess.run([sys.executable, os.path.join(HERE, g + ".py")], capture_output=True, text=True)
            print(f"{g}: exit {r.returncode}")
            if r.returncode != 0:
                print(r.stderr[-2000:])
                bad += 1
        for f in files:
            old, new = np.load(os.path.join(backup, os.path.basename(f))), np.load(f)
            if set(old.files) != set(new.files):
                print("KEYS DIFFER", os.path.basename(f), sorted(set(old.files) ^ set(new.files)))
                bad += 1
            for k in sorted(set(old.files) & set(new.files)):
                total += 1
                if not same(old[k], new[k]):
                    bad += 1
                    print("DIFFERS", os.path.basename(f), k, old[k].shape, new[k].shape)
    finally:
        for f in files:
            shutil.copy2(os.path.join(backup, os.path.basename(f)), f)
        shutil.rmtree(backup, ignore_errors=True)
    print(f"{total} arrays compared, {bad} problems")
    return 1 if bad else 0


if __name__ == "__main__":
    sys.exit(main())
