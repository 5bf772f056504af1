"""Staged copy of the reference, byte-compiled, under ``oracle/_ref/`` (never committed).

``stage()`` (called by ``build()``) compiles the reference's ``pink`` package and its
unittest files into sourceless ``.pyc`` modules under ``oracle/_ref/{pink,tests}``.  The
staged tree travels with the built tree to machines without a reference checkout. There
``scripts/run_reference_tests.py`` and ``scripts/make_reference_golden.py`` import the
reference from it, with ``oracle/refshim`` standing in for its third-party imports.

The reference checkout is ``$PINK_REFERENCE_DIR``, else ``reference_path`` of BASELINE.json.
Where neither is readable, ``stage()`` leaves an existing ``oracle/_ref/`` as it is.

Loaded as a pytest plugin (``-p oracle.ref_build``), it collects the staged ``test_*.pyc``
modules, which pytest by itself only looks for as ``.py`` files.
"""

import json
import os
import py_compile
import shutil

HERE = os.path.dirname(os.path.abspath(__file__))
STAGED = os.path.join(HERE, "_ref")
PACKAGES = ("pink", "tests")


def reference_dir():
    path = os.environ.get("PINK_REFERENCE_DIR")
    if not path:
        with open(os.path.join(HERE, "..", "BASELINE.json")) as fh:
            path = json.load(fh).get("reference_path", "")
    return path if path and os.access(os.path.join(path, "pink", "__init__.py"), os.R_OK) else None


def staged() -> bool:
    return all(os.path.isfile(os.path.join(STAGED, p, "__init__.pyc")) for p in PACKAGES)


def stage() -> bool:
    """(Re)compile the reference into ``oracle/_ref``; False when no reference is readable here."""
    src = reference_dir()
    if src is None:
        return False
    tmp = STAGED + ".tmp"
    shutil.rmtree(tmp, ignore_errors=True)
    for pkg in PACKAGES:
        for d, _, files in os.walk(os.path.join(src, pkg)):
            for f in sorted(files):
                if f.endswith(".py"):
                    rel = os.path.relpath(os.path.join(d, f), src)
                    py_compile.compile(os.path.join(d, f), cfile=os.path.join(tmp, rel + "c"), dfile=rel, doraise=True,
                                       invalidation_mode=py_compile.PycInvalidationMode.UNCHECKED_HASH)
    shutil.rmtree(STAGED, ignore_errors=True)
    os.rename(tmp, STAGED)
    return True


def pytest_collect_file(file_path, parent):
    if file_path.suffix == ".pyc" and file_path.name.startswith("test_") and file_path.is_relative_to(STAGED):
        import pytest

        return pytest.Module.from_parent(parent, path=file_path)
    return None
