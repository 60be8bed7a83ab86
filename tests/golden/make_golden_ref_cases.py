#!/usr/bin/env python
"""Generate tests/golden/golden_ref_cases.json: what the REFERENCE'S OWN Naive<> (include/Utility.h:18-42) computes
for the cases of tests/test_oracle.py that compare the restatement with it (REF_CASES on the recipe inputs, and the
floating-point ones on mixed-sign / NaN / signed-zero / infinity inputs).  Needs oracle/_ref, i.e. a checkout of the
reference for oracle/build.py to compile it from:
    python oracle/build.py && python tests/golden/make_golden_ref_cases.py
"""
import hashlib
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, HERE)
sys.path.insert(0, os.path.dirname(HERE))
import oracle as O  # noqa: E402
import special_inputs as S  # noqa: E402
import test_oracle as T  # noqa: E402


def main():
    out = []
    for inputs, cases in (("recipe", T.REF_CASES), ("special", T.SPECIAL_REF_CASES)):
        for dt, mp, rd, ta, (n, k, m) in cases:
            dtype, m_, r_ = getattr(O, dt), getattr(O, mp), getattr(O, rd)
            assert O.ref_available(dtype, m_, r_, ta), O.ref_config_name(dtype, m_, r_, ta)
            a, b = T.ref_case_inputs(O, dt, inputs, n, k, m)
            c = O.ref_naive(dtype, m_, r_, a, b, n, k, m, transposed_a=ta)
            out.append({
                "case": T.ref_case_id(dt, mp, rd, ta, (n, k, m), inputs),
                "a_sha256": hashlib.sha256(a.tobytes()).hexdigest(), "b_sha256": hashlib.sha256(b.tobytes()).hexdigest(),
                "c_sha256": hashlib.sha256(c.tobytes()).hexdigest(), "c_sha256_nan_canonical": S.canonical_sha256(c),
                "c_nan_count": int(np.isnan(c.astype(np.float64)).sum()) if np.issubdtype(c.dtype, np.floating) else 0,
                "source": "reference Naive<> (include/Utility.h:18-42) via oracle/_ref, g++ -O2 -std=c++14",
            })
            print(out[-1]["case"], "NaNs in C:", out[-1]["c_nan_count"])
    with open(os.path.join(HERE, "golden_ref_cases.json"), "w") as f:
        json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
