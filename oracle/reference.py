"""An importable copy of the unmodified reference (rlabbe/filterpy 1.4.5 @ 3b51149) under
``oracle/_ref`` (git-ignored), for the reference arm of ``bench.py``.

``FILTERPY_REFERENCE`` names a source checkout of the reference.  ``install()`` pip-installs it
once into ``oracle/_ref``; without a checkout it does nothing and ``bench.py`` times the oracle
port instead.  The reference is pure Python: no build step, ``--no-deps`` because numpy / scipy
are already installed.
"""
import os
import shutil
import subprocess
import sys
import tempfile

ENV = "FILTERPY_REFERENCE"
DST = os.path.join(os.path.dirname(os.path.abspath(__file__)), "_ref")


def importable():
    """The ``sys.path`` entry of the installed copy, or None."""
    return DST if os.path.isdir(os.path.join(DST, "filterpy", "kalman")) else None


def install():
    """Never fatal: a failed install leaves ``bench.py`` on the oracle port."""
    src = os.environ.get(ENV)
    if importable() or not src or not os.path.isdir(os.path.join(src, "filterpy")):
        return
    tmp = tempfile.mkdtemp(prefix="ref_copy_")
    try:
        copy = os.path.join(tmp, "reference")
        shutil.copytree(src, copy, ignore=shutil.ignore_patterns(".git"))   # pip writes next to the sources
        subprocess.run([sys.executable, "-m", "pip", "install", "--no-index", "--no-build-isolation", "--no-deps",
                        "--target", DST, copy],
                       check=False, capture_output=True, timeout=600)
    except Exception:
        pass
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
