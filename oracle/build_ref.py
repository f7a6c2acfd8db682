"""TEST / BENCH INFRASTRUCTURE -- installs the UNMODIFIED reference package into the git-ignored oracle/_ref/.

The reference (OpenDriveLab/ST-P3) is pure Python without a setup.py, so `pip install --target oracle/_ref <reference>`
has nothing to build; the equivalent install is a verbatim copy of its `stp3/` package directory (Python sources and
YAML configs only).  oracle/_ref/ is listed in .gitignore -- no reference source enters this repository's history.
Where the install exists, `bench.py --impl reference` and the `cpu_baseline` leg import it through
oracle/ref_loader.py and time the reference's own modules on the host cores (cpu_baseline.kind = "reference").  Run
by __graft_entry__.build() whenever the reference checkout (STP3_REFERENCE_SRC) is readable; without it the install
is left as it is and the benchmark times the op-for-op port instead."""
import os
import shutil
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SRC = os.environ.get("STP3_REFERENCE_SRC", "/root/reference")
DST = os.path.join(ROOT, "oracle", "_ref")


def build_ref(verbose=True) -> bool:
    pkg = os.path.join(SRC, "stp3")
    if not os.path.isdir(pkg):
        if verbose:
            print(f"build_ref: {pkg} not present: using the prebuilt {DST} if it exists")
        return os.path.isdir(os.path.join(DST, "stp3"))
    out = os.path.join(DST, "stp3")
    if os.path.isdir(out):
        shutil.rmtree(out)
    shutil.copytree(pkg, out, ignore=shutil.ignore_patterns("__pycache__", "*.pyc"))
    n = sum(len(f) for _, _, f in os.walk(out))
    if verbose:
        print(f"build_ref: installed the reference package ({n} files) into {out}")
    return True


if __name__ == "__main__":
    sys.exit(0 if build_ref() else 1)
