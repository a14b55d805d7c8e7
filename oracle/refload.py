"""Loader for the UNMODIFIED reference (TEST INFRASTRUCTURE ONLY — never imported by the product).

Only usable where the reference tree exists: ``CSTR_REFERENCE_ROOT``, or a copy of it under the git-ignored ``oracle/_ref`` or
``baseline/_ref``.  The repository does not contain it.  It is used by
  * ``oracle/make_golden.py``   – to generate the committed fixtures under ``tests/golden/``;
  * ``tests/test_oracle_vs_reference.py`` – to pin the oracle restatement (skipped when absent);
  * ``oracle/run_reference_algos.py`` – reference TD3/SAC/BCQ/... on top of the GPU classes (staged for ``gpurun``).

What it does (SURVEY.md App. C, F3/F7):
  1. puts the stand-in ``gymnasium`` / ``matplotlib`` packages of ``oracle/shim`` on ``sys.path``
     (unless a real gymnasium is installed);
  2. ``twoseriescstr.py`` is imported straight from the reference root, unmodified;
  3. ``core/`` cannot be imported in place because ``core/__init__.py:16-18`` opens the missing
     ``core/version.txt`` and the tree is read-only, so ``core`` is *symlinked file by file* into
     a scratch directory outside the repo (``tempfile.mkdtemp``) next to a one-line ``version.txt``.
     No reference source is copied into this repository.
"""
from __future__ import annotations

import importlib
import os
import sys
import tempfile
from types import ModuleType
from typing import Optional

_HERE = os.path.dirname(os.path.abspath(__file__))
SHIM_DIR = os.path.join(_HERE, "shim")
_scratch: Optional[str] = None


def reference_root() -> Optional[str]:
    """``CSTR_REFERENCE_ROOT``, else a git-ignored copy of the reference tree in ``oracle/_ref`` or ``baseline/_ref``."""
    for root in (os.environ.get("CSTR_REFERENCE_ROOT"), os.path.join(_HERE, "_ref"), os.path.join(os.path.dirname(_HERE), "baseline", "_ref")):
        if root and os.path.isfile(os.path.join(root, "twoseriescstr.py")):
            return root
    return None


def available() -> bool:
    return reference_root() is not None


def install_shims() -> None:
    """Put the gymnasium/matplotlib stand-ins on sys.path if the real packages are missing."""
    need = []
    for name in ("gymnasium", "matplotlib"):
        try:
            importlib.import_module(name)
        except ImportError:
            need.append(name)
    if need and SHIM_DIR not in sys.path:
        sys.path.insert(0, SHIM_DIR)
        importlib.invalidate_caches()


def _mirror_core(root: str) -> str:
    """Symlink farm of <root>/core plus the missing version.txt, in a scratch dir."""
    global _scratch
    if _scratch is not None:
        return _scratch
    scratch = tempfile.mkdtemp(prefix="cstr_ref_")
    src_core = os.path.join(root, "core")
    for dirpath, dirnames, filenames in os.walk(src_core):
        dirnames[:] = [d for d in dirnames if d != "__pycache__"]
        rel = os.path.relpath(dirpath, root)
        os.makedirs(os.path.join(scratch, rel), exist_ok=True)
        for fn in filenames:
            if fn.endswith(".pyc"):
                continue
            os.symlink(os.path.join(dirpath, fn), os.path.join(scratch, rel, fn))
    with open(os.path.join(scratch, "core", "version.txt"), "w") as fh:
        fh.write("2.6.0\n")
    _scratch = scratch
    return scratch


def load_env_module() -> ModuleType:
    """Import the reference's ``twoseriescstr`` module unmodified."""
    root = reference_root()
    if root is None:
        raise RuntimeError("reference tree not available")
    install_shims()
    if root not in sys.path:
        sys.path.append(root)
    return importlib.import_module("twoseriescstr")


def load_core() -> ModuleType:
    """Import the reference's ``core`` package (SB3 fork) unmodified."""
    root = reference_root()
    if root is None:
        raise RuntimeError("reference tree not available")
    install_shims()
    scratch = _mirror_core(root)
    if scratch not in sys.path:
        sys.path.insert(0, scratch)
    return importlib.import_module("core")
