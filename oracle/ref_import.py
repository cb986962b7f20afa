"""Import the UNMODIFIED reference (ptwt) from a checkout named by ``PTWT_REFERENCE_SRC`` (its ``src`` directory).
TEST INFRASTRUCTURE ONLY: the golden generators (oracle/make_golden*.py) and oracle/make_ref.py use it; the tests
compare against the fixtures those wrote under tests/golden and never need the reference itself."""
from __future__ import annotations

import importlib
import os
import sys
from pathlib import Path

SHIMS = Path(__file__).resolve().parent / "shims"


def reference_src() -> Path | None:
    """The reference's ``src`` directory, or None when it is not named or cannot be read."""
    src = os.environ.get("PTWT_REFERENCE_SRC")
    if not src:
        return None
    try:
        return Path(src) if (Path(src) / "ptwt" / "__init__.py").is_file() else None
    except OSError:
        return None


def reference_available() -> bool:
    return reference_src() is not None


def add_shims() -> None:
    """Put the pywt / more_itertools shims on sys.path for whichever of the two is not installed."""
    for mod in ("pywt", "more_itertools"):
        try:
            importlib.import_module(mod)
        except Exception:  # noqa: BLE001
            if str(SHIMS) not in sys.path:
                sys.path.insert(0, str(SHIMS))


def import_reference():
    """Returns the reference ``ptwt`` module (with the pywt / more_itertools shims if needed)."""
    src = reference_src()
    if src is None:
        raise RuntimeError("set PTWT_REFERENCE_SRC to the src directory of a readable reference checkout")
    add_shims()
    if str(src) not in sys.path:
        sys.path.insert(0, str(src))
    return importlib.import_module("ptwt")
