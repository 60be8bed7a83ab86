"""CPU tests: the oracle restatement (oracle/naive.cpp) against
  (1) the reference's own Naive<> (include/Utility.h:18-42): what it computed for the cases below, recorded in
      tests/golden/golden_ref_cases.json by tests/golden/make_golden_ref_cases.py,
  (2) the committed golden vectors generated from it (tests/golden/golden.json),
  (3) the known-answer values recorded in SURVEY.md section 8(c).
"""
import hashlib
import json
import os

import numpy as np
import pytest

import sys

HERE = os.path.dirname(os.path.abspath(__file__))
GOLDEN = json.load(open(os.path.join(HERE, "golden", "golden.json")))
GOLDEN_SPECIAL = json.load(open(os.path.join(HERE, "golden", "golden_special.json")))
sys.path.insert(0, os.path.join(HERE, "golden"))
import special_inputs  # noqa: E402


def _id(rec):
    return "%s-%dx%dx%d" % (rec["config"], rec["n"], rec["k"], rec["m"])


@pytest.mark.parametrize("rec", [r for r in GOLDEN if r["n"] * r["k"] * r["m"] <= 513 * 528 * 528], ids=_id)
def test_oracle_matches_golden(oracle, rec):
    """Bit-exact agreement with vectors produced by the reference's Naive<>."""
    a, b = oracle.fill(rec["dtype"], rec["n"], rec["k"], rec["m"], rec["seed"])
    assert hashlib.sha256(a.tobytes()).hexdigest() == rec["a_sha256"]
    assert hashlib.sha256(b.tobytes()).hexdigest() == rec["b_sha256"]
    assert repr(float(a[0])) == rec["a0"] and repr(float(a[1])) == rec["a1"]
    c = oracle.naive(rec["dtype"], rec["map"], rec["reduce"], a, b, rec["n"], rec["k"], rec["m"],
                     transposed_a=rec["transposed_a"], threads=4)
    assert hashlib.sha256(c.tobytes()).hexdigest() == rec["c_sha256"]
    assert repr(float(c.astype(np.float64).flat[0])) == rec["c_first"]
    assert repr(float(c.astype(np.float64).sum())) == rec["c_sum"]


@pytest.mark.parametrize("rec", GOLDEN_SPECIAL, ids=lambda r: "%s-%s-%dx%dx%d" % (r["config"], r["inputs"], r["n"], r["k"], r["m"]))
def test_oracle_matches_golden_on_non_recipe_inputs(oracle, rec):
    """The restatement reproduces the reference-generated records on full-range bytes, mixed signs and NaN / signed-zero /
    infinity inputs (tests/golden/golden_special.json) — here and on the GPU box, where /root/reference does not exist."""
    dtype, n, k, m = rec["dtype"], rec["n"], rec["k"], rec["m"]
    a, b = special_inputs.make(rec["inputs"], oracle.NP_DTYPE[dtype], n, k, m, rec["seed"])
    assert hashlib.sha256(a.tobytes()).hexdigest() == rec["a_sha256"]      # the generator is the one the records were made with
    assert hashlib.sha256(b.tobytes()).hexdigest() == rec["b_sha256"]
    c = oracle.naive(dtype, rec["map"], rec["reduce"], a, b, n, k, m, threads=4)
    assert special_inputs.canonical_sha256(c) == rec["c_sha256_nan_canonical"]
    if np.issubdtype(c.dtype, np.floating):
        assert int(np.isnan(c.astype(np.float64)).sum()) == rec["c_nan_count"]


def test_oracle_matches_golden_1024_sampled_rows(oracle):
    """The 1024^3 float record, checked on sampled rows (first/last) to keep the CPU suite short."""
    rec = [r for r in GOLDEN if r["n"] == 1024][0]
    a, b = oracle.fill(rec["dtype"], 1024, 1024, 1024)
    top = oracle.naive(rec["dtype"], rec["map"], rec["reduce"], a, b, 1024, 1024, 1024, rows=(0, 1))
    bot = oracle.naive(rec["dtype"], rec["map"], rec["reduce"], a, b, 1024, 1024, 1024, rows=(1023, 1024))
    assert repr(float(top[0, 0])) == rec["c_first"]
    assert repr(float(bot[-1, -1])) == rec["c_last"]


SURVEY_KATS = [
    # (dtype, map, reduce, c[0], c[last]) at 256^3 — SURVEY.md section 8(c)
    ("FLOAT", "MULTIPLY", "ADD", 7229.57764, 7799.42236),
    ("DOUBLE", "MULTIPLY", "ADD", 7229.5778, 7799.42325),
    ("FLOAT", "ADD", "MIN", 2.85629749, 2.81436872),
    ("INT32", "MULTIPLY", "ADD", 7149, 8571),
]


@pytest.mark.parametrize("dt,mp,rd,c0,cl", SURVEY_KATS)
def test_survey_known_answers(oracle, dt, mp, rd, c0, cl):
    dtype, m_, r_ = getattr(oracle, dt), getattr(oracle, mp), getattr(oracle, rd)
    a, b = oracle.fill(dtype, 256, 256, 256)
    c = oracle.naive(dtype, m_, r_, a, b, 256, 256, 256)
    assert float(c.flat[0]) == pytest.approx(c0, rel=1e-7)
    assert float(c.flat[-1]) == pytest.approx(cl, rel=1e-7)


REF_CASES = [
    ("FLOAT", "MULTIPLY", "ADD", False, (97, 64, 80)),
    ("DOUBLE", "MULTIPLY", "ADD", False, (65, 24, 40)),
    ("INT32", "MULTIPLY", "ADD", False, (33, 48, 64)),
    ("UINT32", "MULTIPLY", "ADD", False, (33, 48, 64)),
    ("UINT8", "MULTIPLY", "ADD", False, (17, 128, 64)),
    ("FLOAT", "ADD", "MIN", False, (97, 64, 80)),
    ("FLOAT", "ADD", "MAX", False, (31, 32, 48)),
    ("FLOAT", "MIN", "MAX", False, (31, 32, 48)),
    ("DOUBLE", "ADD", "MIN", False, (31, 32, 48)),
    ("INT32", "ADD", "MIN", False, (31, 32, 48)),
    ("INT32", "AND", "ADD", False, (31, 32, 48)),
    ("HALF", "MULTIPLY", "ADD", False, (31, 64, 64)),
    ("FLOAT", "MULTIPLY", "ADD", True, (50, 32, 48)),
]
SPECIAL_REF_CASES = [c for c in REF_CASES if c[0] in ("FLOAT", "DOUBLE", "HALF")]


def ref_case_id(dt, mp, rd, ta, shape, inputs):
    return "%s_%s_%s%s_%dx%dx%d_%s" % (dt, mp, rd, "_TA" if ta else "", shape[0], shape[1], shape[2], inputs)


def ref_case_inputs(oracle, dt, inputs, n, k, m):
    """A and B of a reference comparison: the recipe (seed 7), or mixed signs with NaN / signed zeros / infinities."""
    if inputs == "recipe":
        return oracle.fill(getattr(oracle, dt), n, k, m, seed=7)
    return _special_inputs({"FLOAT": np.float32, "DOUBLE": np.float64, "HALF": np.float16}[dt], n, k, m, seed=11)


_golden_ref = {}


def _reference_record(oracle, dt, mp, rd, ta, shape, inputs):
    """The reference's Naive<> on this case's inputs, as recorded in tests/golden/golden_ref_cases.json; the inputs
    this test draws are checked to be the ones the record was made from."""
    if not _golden_ref:
        for r in json.load(open(os.path.join(HERE, "golden", "golden_ref_cases.json"))):
            _golden_ref[r["case"]] = r
    rec = _golden_ref[ref_case_id(dt, mp, rd, ta, shape, inputs)]
    a, b = ref_case_inputs(oracle, dt, inputs, *shape)
    assert hashlib.sha256(a.tobytes()).hexdigest() == rec["a_sha256"]
    assert hashlib.sha256(b.tobytes()).hexdigest() == rec["b_sha256"]
    return a, b, rec


@pytest.mark.parametrize("dt,mp,rd,ta,shape", REF_CASES)
def test_restatement_equals_reference_naive(oracle, dt, mp, rd, ta, shape):
    """Bit-exact comparison with what the reference's compiled Naive<> computed on the same inputs."""
    dtype, m_, r_ = getattr(oracle, dt), getattr(oracle, mp), getattr(oracle, rd)
    n, k, m = shape
    a, b, ref = _reference_record(oracle, dt, mp, rd, ta, shape, "recipe")
    mine = oracle.naive(dtype, m_, r_, a, b, n, k, m, transposed_a=ta)
    assert hashlib.sha256(mine.tobytes()).hexdigest() == ref["c_sha256"]


def _special_inputs(np_dtype, n, k, m, seed):
    """Mixed-sign values with -0, +0, NaN and infinities sprinkled in: what tests/test_variants_gpu.py feeds the GPU."""
    rng = np.random.default_rng(seed)
    vals = np.array([-3.5, -1.25, -0.5, 0.75, 1.0, 2.5, 6.0])
    pool = np.array([-0.0, 0.0, np.nan, np.inf, -np.inf, -0.0, 0.0])
    out = []
    for size in (n * k, k * m):
        x = rng.choice(vals, size=size)
        idx = rng.choice(size, size=max(4, size // 16), replace=False)
        x[idx] = rng.choice(pool, size=idx.size)
        out.append(x.astype(np_dtype))
    return out


@pytest.mark.parametrize("dt,mp,rd,ta,shape", SPECIAL_REF_CASES)
def test_restatement_equals_reference_naive_on_special_values(oracle, dt, mp, rd, ta, shape):
    """The GPU suite checks NaN / signed-zero / infinity behaviour against the restatement; here the restatement itself
    is pinned to the reference's compiled Naive<> on such inputs (`(a < b) ? a : b`, `a && b`, one rounding per
    operation — hlslib/xilinx/Operators.h:20-100).  NaN payloads are not compared (C++ leaves them open): the hash is
    taken with every NaN made canonical, so it pins the NaN positions and every other bit, signs of zeros included."""
    dtype, m_, r_ = getattr(oracle, dt), getattr(oracle, mp), getattr(oracle, rd)
    n, k, m = shape
    a, b, ref = _reference_record(oracle, dt, mp, rd, ta, shape, "special")
    mine = oracle.naive(dtype, m_, r_, a, b, n, k, m, transposed_a=ta)
    nan_mine = np.isnan(mine.astype(np.float64))
    assert int(nan_mine.sum()) == ref["c_nan_count"]
    assert special_inputs.canonical_sha256(mine) == ref["c_sha256_nan_canonical"]
    assert nan_mine.any() or dt == "HALF" or (mp, rd) != ("MULTIPLY", "ADD")      # the inputs do exercise NaN


def test_row_range_and_threads_are_consistent(oracle):
    a, b = oracle.fill(oracle.FLOAT, 40, 32, 48)
    full = oracle.naive(oracle.FLOAT, oracle.ADD, oracle.MIN, a, b, 40, 32, 48)
    thr = oracle.naive(oracle.FLOAT, oracle.ADD, oracle.MIN, a, b, 40, 32, 48, threads=3)
    part = oracle.naive(oracle.FLOAT, oracle.ADD, oracle.MIN, a, b, 40, 32, 48, rows=(10, 20))
    assert full.tobytes() == thr.tobytes()
    assert np.array_equal(part[10:20], full[10:20]) and not part[:10].any() and not part[20:].any()


def test_identities_follow_the_reference(oracle):
    """K = 0-like behaviour is not reachable, so probe identities through a 1-term reduction:
    Max's identity is numeric_limits<T>::min() (smallest positive), Operators.h:96 — trap 2."""
    a = np.array([-3.0] * 16, dtype=np.float32)      # 1 x 16
    b = np.zeros((16, 16), dtype=np.float32)
    c = oracle.naive(oracle.FLOAT, oracle.ADD, oracle.MAX, a, b, 1, 16, 16)
    # max(FLT_MIN, -3 + 0) = FLT_MIN, not -3
    assert float(c[0, 0]) == float(np.finfo(np.float32).tiny)
    c = oracle.naive(oracle.FLOAT, oracle.ADD, oracle.MIN, a, b, 1, 16, 16)
    assert float(c[0, 0]) == -3.0


def test_verify_criterion(oracle):
    ref = np.array([1000.0, 2000.0, 3000.0], dtype=np.float32)
    ok = ref * np.float32(1.0009)
    bad = ref.copy()
    bad[1] *= np.float32(1.002)
    assert oracle.verify(oracle.FLOAT, ok, ref) == -1
    assert oracle.verify(oracle.FLOAT, bad, ref) == 1
    # NaN quotient is not a mismatch in the reference (SURVEY.md trap 5)
    nanny = ref.copy()
    nanny[2] = np.nan
    assert oracle.verify(oracle.FLOAT, nanny, ref) == -1
    iref = np.array([1, 2, 3], dtype=np.int32)
    assert oracle.verify(oracle.INT32, iref, iref) == -1
    assert oracle.verify(oracle.INT32, iref + np.array([0, 0, 1], dtype=np.int32), iref) == 2
