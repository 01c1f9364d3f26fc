"""Place the unmodified original project (ReChorus) under oracle/_ref/src, git-ignored, as a build product.

The overlay (rechorus_b200.overlay), tools/run_reference.py, the reference arm of bench.py and the overlay tests run
the original ``main.py`` and model classes from there.  ReChorus is a plain Python source tree: there is nothing to
compile, and its packages discover their modules by globbing ``*.py``, so the files are copied as they are.

    python -m oracle.build_ref [SRC]

SRC is the original project's checkout (its ``src/`` is copied); it defaults to the RECHORUS_REF environment
variable, else /root/reference.  Without a checkout nothing is placed, and whatever needs the original skips."""
from __future__ import annotations

import os
import shutil
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
DST = os.path.join(HERE, "_ref", "src")


def build(checkout: str = "") -> str:
    src = os.path.join(checkout or os.environ.get("RECHORUS_REF") or "/root/reference", "src")
    if not os.path.isfile(os.path.join(src, "main.py")):
        return ""
    if os.path.isdir(DST):
        shutil.rmtree(DST)
    for base, dirs, files in os.walk(src):
        dirs[:] = sorted(d for d in dirs if d != "__pycache__")
        out = os.path.join(DST, os.path.relpath(base, src))
        os.makedirs(out, exist_ok=True)
        for f in files:
            if f.endswith(".py"):
                shutil.copyfile(os.path.join(base, f), os.path.join(out, f))     # contents only: the copy stays writable
    return DST


if __name__ == "__main__":
    print(build(sys.argv[1] if len(sys.argv) > 1 else "") or "no ReChorus checkout found")
