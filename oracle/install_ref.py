"""Installs the UNMODIFIED reference (reczoo/FuxiCTR) under oracle/_ref/ for the tests and bench.py's
reference arms.  __graft_entry__.build() calls install(); `python oracle/install_ref.py [--force]` does
the same by hand.

The checkout is looked up in $FUXICTR_REFERENCE, then in a `reference/` directory beside this
repository, then in /root/reference.  Installed are the `fuxictr` package (what setup.py ships) and,
under extras/, what its own entry points read at run time: the five in-scope `model_zoo` directories
(config/*.yaml + src/), `demo/` (example3 = BASELINE config C1) and the `data/tiny_*` fixtures those
YAMLs point at.  The package is imported as is; baseline/refenv.py stubs its three import-time-only
dependencies (SURVEY.md 8c).

oracle/_ref/ is git-ignored: it is built from the checkout, never committed.  Without a checkout an
existing install is kept, and without either the reference-backed tests skip.
"""
import os
import shutil
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
DST = os.path.join(HERE, "_ref")
STAMP = os.path.join(DST, "INSTALLED")
ZOO = ["DeepFM", "DCNv2", "DLRM", "DIN", "xDeepFM"]
DATA = ["tiny_npz", "tiny_parquet", "tiny_seq", "tiny_csv"]


def find_reference():
    for cand in (os.environ.get("FUXICTR_REFERENCE"), os.path.join(os.path.dirname(ROOT), "reference"),
                 "/root/reference"):
        if cand and os.path.isdir(os.path.join(cand, "fuxictr")) and os.path.isdir(os.path.join(cand, "model_zoo")):
            return cand
    return None


def installed():
    return os.path.exists(STAMP)


def install(force=False):
    """Returns the install directory, or None when there is neither an install nor a checkout."""
    if installed() and not force:
        return DST
    src = find_reference()
    if src is None:
        return DST if installed() else None
    tmp = DST + ".tmp"
    shutil.rmtree(tmp, ignore_errors=True)
    skip = shutil.ignore_patterns("__pycache__", "*.pyc")
    shutil.copytree(os.path.join(src, "fuxictr"), os.path.join(tmp, "fuxictr"), ignore=skip)
    extras = os.path.join(tmp, "extras")
    for name in ZOO:
        shutil.copytree(os.path.join(src, "model_zoo", name), os.path.join(extras, "model_zoo", name), ignore=skip)
    shutil.copytree(os.path.join(src, "demo"), os.path.join(extras, "demo"), ignore=skip)
    for name in DATA:
        shutil.copytree(os.path.join(src, "data", name), os.path.join(extras, "data", name), ignore=skip)
    # the checkout may be read-only: the install belongs to whoever built it and can be rebuilt or removed
    for root, dirs, files in os.walk(tmp):
        os.chmod(root, 0o755)
        for f in files:
            os.chmod(os.path.join(root, f), 0o644)
    with open(os.path.join(tmp, "INSTALLED"), "w") as fd:
        fd.write(src + "\n")
    shutil.rmtree(DST, ignore_errors=True)
    os.rename(tmp, DST)
    return DST


if __name__ == "__main__":
    print(install(force="--force" in sys.argv) or "no FuxiCTR checkout found")
