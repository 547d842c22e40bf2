"""ORACLE (test infrastructure only): the reference itself, materialised so it can travel.

The reference is a Python package with C code it generates and compiles at run
time (``aesara/link/c``).  ``/root/reference`` exists only in the build
container; the GPU box gets whatever lies in the repo directory.  ``materialise()``
therefore copies the *package directory* ``/root/reference/aesara`` — unmodified,
byte for byte — into ``oracle/_ref/aesara`` (git-ignored, so nothing of the
reference enters history; not gpurun-ignored, so it travels).  It is the
equivalent of ``pip install --target`` for a pure-Python package and is run by
``__graft_entry__.build()`` whenever ``/root/reference`` is present.

What uses it (and nothing else may):
  * ``tests/`` — ``aesara.function(..., mode="B200")`` against the reference's own
    C-linker (``Mode("cvm", "fast_run")``, ``aesara/link/vm.py:1057-1174``) in the
    same process, on the GPU box;
  * ``bench.py --impl reference`` / ``cpu_baseline`` — the reference C-linker timed on
    the host cores (``kind: "reference"``);
  * ``tests/golden/make_golden.py`` — fixture generation.

The product (``aesara_b200``) never looks here: it imports whatever ``aesara`` the
user has installed (or ``$AESARA_B200_REFERENCE``), exactly like any other Aesara
linker plugin.  ``activate()`` is how the checkers point that variable at the copy.
"""

from __future__ import annotations

import hashlib
import os
import shutil
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
REF_DIR = os.path.join(HERE, "_ref")
SOURCE = "/root/reference"


def _tree_stamp(root):
    """Cheap content stamp: relative path + size + mtime of every .py/.c/.h/.pyx file."""
    h = hashlib.sha256()
    for d, dirs, files in os.walk(root):
        dirs[:] = sorted(x for x in dirs if x != "__pycache__")
        for f in sorted(files):
            if f.endswith((".pyc", ".pyo")):
                continue
            p = os.path.join(d, f)
            st = os.stat(p)
            h.update(os.path.relpath(p, root).encode())
            h.update(str(st.st_size).encode())
    return h.hexdigest()


def materialise(force=False, verbose=True):
    """Copy /root/reference/aesara -> oracle/_ref/aesara if the source is present.
    Returns the directory that holds the ``aesara`` package, or None."""
    src = os.path.join(SOURCE, "aesara")
    dst = os.path.join(REF_DIR, "aesara")
    if not os.path.isdir(src):
        return REF_DIR if os.path.isdir(dst) else None
    stamp_file = os.path.join(REF_DIR, "stamp")
    stamp = _tree_stamp(src)
    if not force and os.path.isdir(dst) and os.path.exists(stamp_file):
        with open(stamp_file) as f:
            if f.read().strip() == stamp:
                return REF_DIR
    if os.path.isdir(dst):
        shutil.rmtree(dst)
    os.makedirs(REF_DIR, exist_ok=True)
    shutil.copytree(src, dst, ignore=shutil.ignore_patterns("__pycache__", "*.pyc", "*.pyo"))
    with open(stamp_file, "w") as f:
        f.write(stamp)
    if verbose:
        print(f"oracle/_ref: materialised the reference package from {src}", file=sys.stderr)
    return REF_DIR


def reference_dir():
    """Directory containing the reference ``aesara`` package: the copy ``materialise()`` made,
    else None.  Tests, ``smoke()`` and the benchmark read only that copy, never the source."""
    if os.path.isdir(os.path.join(REF_DIR, "aesara")):
        return REF_DIR
    return None


def compiledir():
    """Where the reference C-linker caches its compiled modules: next to the copy (so
    modules compiled in the build container travel and are reused when the key matches)."""
    d = os.path.join(REF_DIR, "compiledir")
    try:
        os.makedirs(d, exist_ok=True)
        return d
    except OSError:
        return None


def activate():
    """Point the plugin's front-end lookup (``aesara_b200.compat.bootstrap``) at the
    reference copy.  Must run before the first ``import aesara``.  Returns the directory
    or None when no reference is available (tests then skip)."""
    d = reference_dir()
    if d is None:
        return None
    os.environ.setdefault("AESARA_B200_REFERENCE", d)
    if d == REF_DIR:
        cd = compiledir()
        if cd:
            os.environ.setdefault("AESARA_B200_COMPILEDIR", cd)
    return d


if __name__ == "__main__":
    print(materialise(force="--force" in sys.argv))
