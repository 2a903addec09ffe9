"""Stages the reference's Python package for the CPU-timing arm: $GYM_PBN_REF/gym_PBN -> baseline/_ref/gym_PBN (git-ignored;
nothing is installed, nothing is modified).  GYM_PBN_REF names a checkout of the original gym-PBN-stac, the same variable
oracle/ref_loader.py reads.  Run by __graft_entry__.build(); a no-op when the variable is unset or the directory cannot be
read, so a build never depends on anything outside the repository."""
import os
import shutil
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
DST = ROOT / "baseline" / "_ref" / "gym_PBN"


def stage():
    ref = os.environ.get("GYM_PBN_REF")
    src = os.path.join(ref, "gym_PBN") if ref else None
    if not src or not os.path.isdir(src):  # os.path.isdir is False on any OSError (Path.is_dir raises on EACCES)
        return False
    if DST.exists():
        shutil.rmtree(DST)
    DST.parent.mkdir(parents=True, exist_ok=True)
    shutil.copytree(src, DST, ignore=shutil.ignore_patterns("__pycache__", "*.pyc", "*.xls", "*.pkl", "*.csv"))
    return True


if __name__ == "__main__":
    print("staged" if stage() else "nothing staged: set GYM_PBN_REF to a readable gym-PBN-stac checkout", file=sys.stderr)
