#!/usr/bin/env python
"""Install the UNMODIFIED upstream Flashy (facebookresearch/flashy) into oracle/_ref.

    FLASHY_REFERENCE=<upstream checkout> python oracle/install_ref.py

The upstream source is ``$FLASHY_REFERENCE`` when it is set; otherwise the first readable checkout of
``REFERENCE_DIRS``: one named ``reference`` beside this repository, then ``/root/reference``.
``oracle/_ref`` is git-ignored (never committed); once built it is all the solver drop-in tests need,
so a machine without the upstream source can run them from a copy of the tree.
Upstream's dependencies ``dora_search`` and ``colorlog`` are not needed offline: the package is
installed with ``--no-deps`` and the solver tests provide minimal stand-ins for the two
(tests/shims/, test-only).  pip builds in the source directory, so the build runs from a temporary
copy.  Prints one line with the outcome.
"""
import os
import shutil
import subprocess
import sys
import tempfile
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
REFERENCE_DIRS = (ROOT.parent / "reference", Path("/root/reference"))
DEST = ROOT / "oracle" / "_ref"


def install() -> str:
    if (DEST / "flashy" / "solver.py").exists():
        return f"already installed: {DEST}"
    env = os.environ.get("FLASHY_REFERENCE")
    ref, why = None, []
    for cand in [Path(env)] if env else REFERENCE_DIRS:
        try:
            if (cand / "flashy" / "solver.py").is_file():
                ref = cand
                break
            why.append(f"no upstream Flashy checkout at {cand}")
        except OSError as exc:                 # e.g. a directory this user may not enter
            why.append(str(exc))
    if ref is None:
        return "unavailable: " + "; ".join(why) + " (set FLASHY_REFERENCE)"
    with tempfile.TemporaryDirectory() as tmp:
        src = Path(tmp) / "reference"
        shutil.copytree(ref, src, ignore=shutil.ignore_patterns(".git"), copy_function=shutil.copyfile)
        for d in [src, *(p for p in src.rglob("*") if p.is_dir())]:
            d.chmod(0o755)                     # copytree keeps a read-only checkout's modes; pip writes build/ here
        cmd = [sys.executable, "-m", "pip", "install", "--no-index", "--no-build-isolation", "--no-deps",
               "--no-cache-dir", "--disable-pip-version-check", "--target", str(DEST), str(src)]
        res = subprocess.run(cmd, capture_output=True, text=True)
        if res.returncode != 0:
            shutil.rmtree(DEST, ignore_errors=True)
            return "failed: " + (res.stderr.strip().splitlines() or ["pip error"])[-1]
    # upstream also ships its own `tests` package: not needed here, and pytest would collect it
    shutil.rmtree(DEST / "tests", ignore_errors=True)
    return f"installed {DEST} (pip --no-deps; dora_search / colorlog are stand-ins under tests/shims)"


if __name__ == "__main__":
    print(install())
