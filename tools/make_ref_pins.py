#!/usr/bin/env python
"""Stored outputs of the reference's own code -> tests/golden/ref_pins.npz (format: tests/ref_pins.py).

Needs oracle/_ref/libfuel_ref.so, which oracle/Makefile builds only where the reference sources are present: the
reference's sdf_map.cpp, raycast.cpp, bspline_optimizer.cpp, frontier_finder.cpp and perception_utils.cpp compiled
unmodified against the stand-ins of oracle/ref_standin.  Runs the reference side of every case the test modules below
list in their REF_PINS tables, on the same seeded inputs the tests build, and writes what it returns."""
import importlib
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import oracle as O  # noqa: E402
from tests import ref_pins as RP  # noqa: E402

MODULES = ("test_oracle_refpin", "test_host_frontier_bookkeeping", "test_gpu_fusion")


def main():
    O.build()
    assert O.ref_raycast() is not None, "oracle/_ref/libfuel_ref.so was not built (needs the reference sources)"
    out = {}
    for name in MODULES:
        mod = importlib.import_module("tests." + name)
        for case, (fn, arglist) in mod.REF_PINS.items():
            for args in arglist:
                out.update(RP.pack(RP.case_prefix(name, case, mod.REF_PINS, args), fn(*args)))
    RP.save(out)
    print("wrote %s: %d entries, %.0f KB" % (RP.PATH, len(out), os.path.getsize(RP.PATH) / 1024))


if __name__ == "__main__":
    main()
