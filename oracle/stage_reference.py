"""Recipe that builds the UNMODIFIED reference into the git-ignored ``oracle/_ref/`` (test + benchmark infrastructure).

The reference (Rongjiehuang/FastDiff) is pure Python with no ``setup.py``: its "build" is Python bytecode.  Given a read-only
checkout of it (``FD_REFERENCE_ROOT``, else ``DEFAULT_SOURCE``), every module of the trees the sampling path and its callers import (``modules/ tasks/ utils/ vocoders/
data_gen/``) is compiled to a sourceless ``.pyc`` at the place of its ``.py`` under ``oracle/_ref/``, which Python imports like the
package itself.  No source file is copied; YAML configs and audio are not built, so what needs them (the task-level drop-in tests)
reads the checkout, whose path the build records in ``oracle/_ref/SOURCE``.  ``oracle/_ref/`` travels with a working tree to a machine without the checkout, where

  * ``bench.py --impl reference`` and the ``cpu_baseline`` leg time the reference's OWN ``sampling_given_noise_schedule`` /
    ``FastDiff.forward`` (``cpu_baseline.kind = "reference"``) instead of the oracle port,
  * ``tests/golden/make_golden.py --gpu`` records the reference's outputs on the GPU, and
  * the ``-m gpu`` vocoder-registry drop-in test runs the reference's registry code against the CUDA path.

Run by ``__graft_entry__.build()``; where no checkout is reachable, nothing happens.
"""
from __future__ import annotations

import os
import py_compile
import sys
import warnings

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DST = os.path.join(ROOT, "oracle", "_ref")
TREES = ("modules", "tasks", "utils", "vocoders", "data_gen")
DEFAULT_SOURCE = "/root/reference"          # where the read-only reference checkout is mounted when FD_REFERENCE_ROOT is unset


def stage(force: bool = False) -> str | None:
    """Compile the trees if a checkout of the reference is reachable; returns the built root or None."""
    src = os.path.abspath(os.environ.get("FD_REFERENCE_ROOT") or DEFAULT_SOURCE)
    if not os.path.isdir(os.path.join(src, "modules", "FastDiff")):
        return None
    for tree in TREES:
        for dirpath, _dirs, files in os.walk(os.path.join(src, tree)):
            rel = os.path.relpath(dirpath, src)
            for f in files:
                if not f.endswith(".py"):
                    continue
                s, d = os.path.join(dirpath, f), os.path.join(DST, rel, f + "c")
                if not force and os.path.exists(d) and os.path.getmtime(d) >= os.path.getmtime(s):
                    continue
                os.makedirs(os.path.dirname(d), exist_ok=True)
                with warnings.catch_warnings():
                    warnings.simplefilter("ignore", SyntaxWarning)   # invalid escapes in the reference's docstrings
                    py_compile.compile(s, cfile=d, dfile=os.path.join(rel, f), doraise=True)
    with open(os.path.join(DST, "SOURCE"), "w") as fh:
        fh.write(src + "\n")
    return DST


if __name__ == "__main__":
    print(stage(force="--force" in sys.argv))
