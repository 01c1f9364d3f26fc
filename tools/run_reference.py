#!/usr/bin/env python
"""Run the UNMODIFIED reference main.py (``--ref``, the RECHORUS_SRC environment variable, else the copy build() places
in oracle/_ref/src) on today's NumPy.

    python tools/run_reference.py [--ref DIR] <main.py arguments>

The only thing done before `runpy` is restoring the three NumPy aliases the reference still spells (np.object, np.int,
np.float; removed in NumPy 1.24 -- models/BaseModel.py:141, models/sequential/SASRec.py:69, utils/utils.py:65).  Used by
the overlay tests and by bench.py's reference arm as the CPU side of an A/B run; none of this package is imported."""
import os
import runpy
import sys

import numpy as np

HERE = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def main():
    argv = sys.argv[1:]
    ref = os.environ.get("RECHORUS_SRC") or os.path.join(HERE, "oracle", "_ref", "src")
    if "--ref" in argv:
        i = argv.index("--ref")
        ref = argv[i + 1]
        del argv[i:i + 2]
    for alias, typ in (("object", object), ("int", int), ("float", float)):
        if not hasattr(np, alias):
            setattr(np, alias, typ)
    sys.path.insert(0, ref)
    sys.argv = [os.path.join(ref, "main.py")] + argv
    runpy.run_path(os.path.join(ref, "main.py"), run_name="__main__")


if __name__ == "__main__":
    main()
