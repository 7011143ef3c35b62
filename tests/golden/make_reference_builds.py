#!/usr/bin/env python
"""Generates tests/golden/reference_builds.npz: the answers of the reference's own zone_malloc.c, data.c,
two_dim_rectangle_cyclic.c and device.c (built into oracle/_ref by oracle/Makefile.ref) to the inputs of the tests in
tests/test_oracle.py, which check the oracle and the product against them.  Run after __graft_entry__.build() has
built oracle/_ref."""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]

import test_oracle as T  # noqa: E402

if __name__ == "__main__":
    answers = {"twodbc": T.twodbc_reference_answers, "select": T.select_reference_answers,
               "zone": T.zone_reference_answers, "coherency": T.coherency_reference_answers}
    np.savez_compressed(T.GOLDEN_REF, **{name: f() for name, f in answers.items()})
    print("wrote", T.GOLDEN_REF, os.path.getsize(T.GOLDEN_REF), "bytes")
