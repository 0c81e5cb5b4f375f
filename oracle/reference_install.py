"""Recipe for ``oracle/_ref``: the unmodified reference package (astooke/rlpyt, pure Python, so nothing is
compiled) copied from the reference checkout, ``RLPYT_REFERENCE`` or by default the one tests/golden/make_golden.py
reads.  bench.py's ``--impl reference`` arm and tests/test_gpu_runner_dropin.py import it from there.
``oracle/_ref`` is not tracked; where it was not built, the reference arm runs the oracle port instead and the
drop-in test skips."""
import os
import shutil

DEST = os.path.join(os.path.dirname(os.path.abspath(__file__)), "_ref")
SOURCE = os.environ.get("RLPYT_REFERENCE", "/root/reference")


def available():
    return os.path.isdir(os.path.join(DEST, "rlpyt"))


def install(src=None):
    """Copy ``<src>/rlpyt`` (default: SOURCE) to ``oracle/_ref/rlpyt`` once; returns whether the package is there
    afterwards.  Files are copied without their modes: the checkout may be read-only."""
    src = src or SOURCE
    pkg = os.path.join(src, "rlpyt")
    if available() or not src or not os.path.isdir(pkg):
        return available()
    tmp = os.path.join(DEST, "rlpyt.partial")
    shutil.rmtree(tmp, ignore_errors=True)
    for d, dirs, files in os.walk(pkg):
        dirs[:] = [x for x in dirs if x != "__pycache__"]
        out = os.path.join(tmp, os.path.relpath(d, pkg))
        os.makedirs(out, exist_ok=True)
        for f in files:
            if not f.endswith(".pyc"):
                shutil.copyfile(os.path.join(d, f), os.path.join(out, f))
    os.rename(tmp, os.path.join(DEST, "rlpyt"))
    return True
