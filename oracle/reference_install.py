"""Installs the unmodified reference package (stable-ts, pure Python) into oracle/_ref/ for the tests that drive its own
control plane (``Aligner`` / ``Refiner``) over this package's closures.  TEST INFRASTRUCTURE ONLY: oracle/_ref/ is not part of
the repository, and only the Aligner / Refiner tests of tests/test_boundary_reference_cpu.py and tests/test_gpu_boundary.py
import from it, removing it from the interpreter again afterwards.

The source is the stable-ts checkout named by $STABLE_TS_SRC (default: the checkout the oracle was pinned against).  Where it
is absent nothing is installed and those tests skip.
"""
import os
import shutil

SRC = os.environ.get("STABLE_TS_SRC", "/root/reference")
DEST = os.path.join(os.path.dirname(os.path.abspath(__file__)), "_ref")
PACKAGE = "stable_whisper"


def build() -> bool:
    """Copies the package's modules into oracle/_ref/ (what a pip --target install does for a pure-Python package) and
    byte-compiles them.  -> True when the package is installed."""
    src = os.path.join(SRC, PACKAGE)
    if not os.path.isfile(os.path.join(src, "__init__.py")):
        return path() is not None
    dest = os.path.join(DEST, PACKAGE)
    tmp = dest + ".tmp"
    shutil.rmtree(tmp, ignore_errors=True)
    shutil.copytree(src, tmp, ignore=shutil.ignore_patterns("__pycache__", "*.pyc"))
    shutil.rmtree(dest, ignore_errors=True)
    os.replace(tmp, dest)
    import compileall
    import warnings
    with warnings.catch_warnings():                 # the reference's own docstrings trip SyntaxWarnings; not ours to report
        warnings.simplefilter("ignore", SyntaxWarning)
        compileall.compile_dir(dest, quiet=1)
    return True


def path():
    """Import root of the installed package, or None."""
    return DEST if os.path.isfile(os.path.join(DEST, PACKAGE, "__init__.py")) else None
