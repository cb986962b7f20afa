"""Install the UNMODIFIED reference package into the git-ignored ``oracle/_ref`` so that `bench.py --impl reference`
and the `cpu_baseline` leg can time the reference itself on the host cores, and the install() tests can rebind it.

    PTWT_REFERENCE_SRC=<reference checkout>/src python -m oracle.make_ref [--force]

The reference is pure Python and its build backend (`pdm-backend`) is not always installable, so the recipe copies
`src/ptwt` byte for byte into `oracle/_ref/ptwt` and records the file hashes; it is never committed.  PyWavelets may
be absent as well: the reference is then imported with the `pywt` / `more_itertools` shims of `oracle/shims` (filter
taps and level formulas only).  Without ``PTWT_REFERENCE_SRC`` nothing is installed and every user of the reference
falls back or skips.  Nothing in the product imports it.
"""
from __future__ import annotations

import hashlib
import importlib
import json
import shutil
import sys
from pathlib import Path

from oracle.ref_import import add_shims, reference_src

HERE = Path(__file__).resolve().parent
DST = HERE / "_ref" / "ptwt"


def make(force: bool = False) -> Path | None:
    if DST.exists() and not force:
        return DST
    src = reference_src()
    if src is None:
        return None
    if DST.exists():
        shutil.rmtree(DST)
    DST.parent.mkdir(parents=True, exist_ok=True)
    shutil.copytree(src / "ptwt", DST, ignore=shutil.ignore_patterns("__pycache__"))
    manifest = {str(p.relative_to(DST)): hashlib.sha256(p.read_bytes()).hexdigest() for p in sorted(DST.rglob("*.py"))}
    (DST.parent / "MANIFEST.json").write_text(json.dumps({"files": manifest}, indent=1))
    return DST


def import_ref():
    """The reference `ptwt` module from oracle/_ref (None when it was never installed there)."""
    if not (DST / "__init__.py").exists():
        return None
    add_shims()
    if str(DST.parent) not in sys.path:
        sys.path.insert(0, str(DST.parent))
    return importlib.import_module("ptwt")


if __name__ == "__main__":
    out = make(force="--force" in sys.argv)
    print(out if out else "PTWT_REFERENCE_SRC names no readable reference: nothing installed")
