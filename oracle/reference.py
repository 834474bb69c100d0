"""Installs the unmodified reference package (normflows 1.7.3; pure Python, needs only numpy and torch) into
oracle/_ref/normflows for the reference arms of bench.py (`reference_eager_b200`, `cpu_baseline`, `--impl reference`).

build() calls install().  oracle/_ref/ is not part of the repository: it is made from a checkout of the original
project (https://github.com/VincentStimper/normalizing-flows), taken from $NFB_REFERENCE or from the location it has in
the build environment.  The package is copied file for file, without its own `*_test.py` modules, so that a pytest run
from the repository root never collects them (collecting them would put the reference on sys.path ahead of this
package).  Where no checkout is found, an existing installation is kept as it is."""
import os
import shutil

DEST = os.path.join(os.path.dirname(os.path.abspath(__file__)), "_ref")
DEFAULT_SOURCE = "/root/reference"


def source():
    """The checkout holding the reference's normflows/ package, or None."""
    for d in (os.environ.get("NFB_REFERENCE"), DEFAULT_SOURCE):
        if d and os.path.isfile(os.path.join(d, "normflows", "__init__.py")):
            return d
    return None


def install():
    """Copy the reference package to oracle/_ref/normflows; -> True when an installation is present afterwards."""
    src = source()
    if src is not None:
        dst = os.path.join(DEST, "normflows")
        shutil.rmtree(dst, ignore_errors=True)
        shutil.copytree(os.path.join(src, "normflows"), dst,
                        ignore=shutil.ignore_patterns("__pycache__", "*.pyc", "*_test.py", "test_*.py"))
    return os.path.isfile(os.path.join(DEST, "normflows", "__init__.py"))
