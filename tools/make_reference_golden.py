#!/usr/bin/env python3
"""Digests of the reference's outputs for tests/test_reference_pinned.py (tests/golden/reference_pinned.json).

The pinned tests compare the oracle with the reference's own C++ compiled unmodified (oracle/_ref/libbmm_ref.so), which
needs the reference sources.  Where they are absent the tests compare with these digests instead.  They are taken from
oracle/oracle.cpp, which the live comparison found bit-identical to the reference on every one of these calls, and only
for outputs that do not depend on the assignment solver (see SOLVER_FREE in the test module).  The my_lpsolve entries
are the optima of random cost matrices, recorded only when the optimum is unique, so any exact solver returns them.
    python tools/make_reference_golden.py
"""
import json
import os
import sys

import numpy as np
from scipy.optimize import linear_sum_assignment

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]


def unique_optimum_gap(c):
    """Cost of the best assignment that differs from the optimum, minus the optimum's cost."""
    r, col = linear_sum_assignment(c)
    best = c[r, col].sum()
    second = np.inf
    for i in range(len(r)):
        cc = c.copy()
        cc[r[i], col[i]] = 1e12
        rr, ccol = linear_sum_assignment(cc)
        second = min(second, cc[rr, ccol].sum())
    return second - best


def main():
    import test_reference_pinned as T
    from conftest import load_golden_matrix
    from oracle import pyoracle as O
    O.lib()
    datasets = {n: load_golden_matrix(n) for n in T.FIXTURES}
    out = {}

    def check(what, ref_call, oracle_result, relabel):
        key = "%s relabel=%s" % (what, relabel)
        assert key not in out, key
        out[key] = T.golden_entry(oracle_result.tail(), relabel)

    def check_array(what, ref_call, value):
        assert what not in out, what
        out[what] = T.digest(value)

    T.HAVE_REF, T.check, T.check_array = False, check, check_array
    orig_assign = O.assign

    def assign(c, use_ref=None):
        assert unique_optimum_gap(np.asarray(c)) > 1e-6, "tied optimum: not solver-independent"
        return orig_assign(c, use_ref)
    O.assign = assign
    for fn in (T.test_gibbs_full_equals_reference, T.test_gibbs_stickbreaking_equals_reference,
               T.test_gibbs_collapsed_equals_reference, T.test_gibbs_dp_equals_reference):
        for name in T.FIXTURES:
            for relabel in (False, True):
                fn(O, datasets, name, relabel)
    T.test_gibbs_stickbreaking_burnrelabel_above_burnin_equals_reference(O, datasets)
    T.test_gibbs_collapsed_empty_cluster_equals_reference(O, datasets)
    T.test_gibbs_dp_truncation_equals_reference(O, datasets)
    T.test_my_lpsolve_equals_reference(O)
    T.test_rdirichlet_and_update_alpha_equal_reference(O)
    with open(T.GOLDEN_PATH, "w") as f:
        json.dump(out, f, indent=0, sort_keys=True)
        f.write("\n")
    print("wrote", T.GOLDEN_PATH, len(out), "entries,", os.path.getsize(T.GOLDEN_PATH), "bytes")


if __name__ == "__main__":
    main()
