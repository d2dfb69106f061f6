"""Recipe for ``oracle/_ref/``: the unmodified reference package (VeOmni, pure Python) placed inside the tree.

``build()`` runs it. The source tree is ``$VEOMNI_SRC`` if set, else ``/root/reference`` (the location the fixture
generators under tests/golden/ read it from). Its ``veomni`` package is copied file by file, without bytecode, into
``oracle/_ref/veomni`` (git-ignored), replacing an earlier copy. When no readable source holds a ``veomni`` package nothing
is done, and the CPU tests that exercise the real package (tests/test_registry.py) skip. No GPU test reads ``oracle/_ref``.
"""
from __future__ import annotations

import os
import shutil
from pathlib import Path

REF_DIR = Path(__file__).resolve().parent / "_ref"
DEFAULT_SRC = "/root/reference"


def build_ref(verbose: bool = False) -> Path | None:
    """Copy the reference's ``veomni`` package into ``oracle/_ref``; return that directory, or None without a source."""
    src = Path(os.environ.get("VEOMNI_SRC") or DEFAULT_SRC) / "veomni"
    if not os.access(src / "__init__.py", os.R_OK):
        if verbose:
            print(f"[oracle.build_ref] no readable reference package at {src}: oracle/_ref not built")
        return None
    dst = REF_DIR / "veomni"
    if dst.exists():
        shutil.rmtree(dst)
    for f in sorted(src.rglob("*")):
        if "__pycache__" in f.parts or not f.is_file():
            continue
        out = dst / f.relative_to(src)
        out.parent.mkdir(parents=True, exist_ok=True)
        shutil.copyfile(f, out)  # contents only: the copy stays writable for the next rebuild
    if verbose:
        print(f"[oracle.build_ref] copied {src} -> {dst}")
    return REF_DIR
