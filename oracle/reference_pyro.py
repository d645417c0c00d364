"""Recipe for the unmodified reference Pyro (pyro-ppl 1.9.1) used by the binding tests and by the
CPU-baseline arm of bench.py.

``install()`` copies the ``pyro`` package of the reference source tree, unchanged, into ``oracle/_ref``
(git-ignored).  The tree is read from ``PYRO_REFERENCE_SRC`` or, when that variable is unset, from
``DEFAULT_SRC``, the reference's default checkout location; where neither exists nothing is installed, a
note says so, and the tests that need reference Pyro skip.  Pyro is pure Python, so a copy is a complete
install (``pyro.__version__`` falls back to ``version_prefix`` without the generated ``_version.py``); torch
and numpy are already importable, and its one other dependency, ``opt_einsum``, is replaced by the
stand-in under ``tests/golden/opt_einsum_standin`` (see ``pyro_b200.bind.add_reference_to_path``).
"""
import os
import shutil
import stat
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
DEST = os.path.join(HERE, "_ref")
ENV = "PYRO_REFERENCE_SRC"
DEFAULT_SRC = "/root/reference"


def install():
    """Install the reference into ``oracle/_ref`` once; returns True when it is there afterwards."""
    if os.path.isdir(os.path.join(DEST, "pyro")):
        return True
    src = os.environ.get(ENV)
    if src is None:
        if not os.path.isdir(os.path.join(DEFAULT_SRC, "pyro")):
            print("[pyro_b200] reference Pyro not installed (set %s to its source tree); "
                  "tests/test_bind_pyro.py will skip" % ENV, file=sys.stderr)
            return False
        src = DEFAULT_SRC
    elif not os.path.isdir(os.path.join(src, "pyro")):
        raise RuntimeError("%s=%s is not a Pyro source tree" % (ENV, src))
    # copy next to the destination and rename, so an interrupted copy never looks like an install
    tmp = DEST + ".partial"
    shutil.rmtree(tmp, ignore_errors=True)
    try:
        shutil.copytree(os.path.join(src, "pyro"), os.path.join(tmp, "pyro"),
                        ignore=shutil.ignore_patterns("__pycache__"))
        # the copy keeps the source's modes; a read-only copy could not be replaced or removed later
        for d, _, files in os.walk(tmp):
            for p in [d] + [os.path.join(d, f) for f in files]:
                os.chmod(p, os.stat(p).st_mode | stat.S_IWUSR)
        shutil.rmtree(DEST, ignore_errors=True)   # leftovers without a pyro package
        os.rename(tmp, DEST)
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    return True
