"""GPU parity of everything the library can be PUT INTO (run with `-m gpu` on a B200):

  1. every tuning knob of include/mm_b200.h (mm_context_set_tuning) on the tensor-core kernels —
     the build-manager sweep of the reference changes tiles, never results (scripts/build_manager.py:224-306);
  2. the CUDA-core semiring kernel with the DEFAULT flags (what a caller gets without MM_FLAG_EXACT),
     on signed data, and with NaN / signed zeros / infinities under both flag settings
     (hlslib/include/hlslib/xilinx/Operators.h:76-100 is `(a < b) ? a : b`);
  3. the multi-chunk pipeline of the host-pointer entry (test/TestSimulation.cpp:66 at sizes where
     A does not fit one chunk);
  4. the row-block split over several GPUs (mm_multi_*, SURVEY.md 8e) — on ONE device here by
     listing it several times: slices of B, the gather kernel, panel counters and host barriers are
     the same code that runs over NVLink;
  5. argument checks that need a device (alignment, tuning ranges, scratch growth under capture).
"""
import json
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden"))
import special_inputs  # noqa: E402

pytestmark = pytest.mark.gpu
GOLDEN_SPECIAL = json.load(open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "golden_special.json")))

TOL = {"tcgen05_tf32": 5e-4, "dmma_f64": 1e-12, "tcgen05_f16": 1e-3}


def max_rel(c, ref):
    c64, r64 = c.astype(np.float64), ref.astype(np.float64)
    return float(np.max(np.abs(c64 - r64) / np.abs(r64)))


def half_inputs(oracle, n, k, m, seed=5):
    a, b = oracle.fill(oracle.HALF, n, k, m, seed)
    a = (a.astype(np.float32) * np.float32(min(1.0, 500.0 / k))).astype(np.float16)
    return a, b


# ---------------------------------------------------------------------------------------------
# 1. tuning knobs
# ---------------------------------------------------------------------------------------------
TCGEN05_VARIANTS = [
    dict(),                                   # defaults: CTA pairs, 256 columns, deepest ring, TMA stores, B overlapped
    dict(cta_group=1),
    dict(block_n=128),
    dict(cta_group=1, block_n=128),
    dict(stages=2), dict(stages=3), dict(stages=4), dict(stages=5), dict(stages=6),
    dict(block_n=128, stages=8),
    dict(raster_rows=256), dict(raster_rows=8192),
    dict(tile_sync=0),
    dict(b_mn=0),                             # K-major B from a transposed copy (the round-1 layout)
    dict(b_mn=0, cta_group=1, block_n=128),
    dict(b_overlap=0),
    dict(tma_store=0),                        # direct per-lane epilogue stores
    dict(tma_store=0, cta_group=1),
    dict(l2_policy=1), dict(l2_policy=2),
]


def _vid(v):
    return ",".join("%s=%s" % kv for kv in sorted(v.items())) or "default"


@pytest.mark.parametrize("variant", TCGEN05_VARIANTS, ids=_vid)
def test_tcgen05_tuning_variants_float(mm, oracle, variant):
    """float (Multiply, Add): the reference's CTest shape (ragged N, K % 32 != 0) and a multi-tile shape."""
    with mm.Context(0) as ctx:
        ctx.set_tuning(**variant)
        for name, value in variant.items():
            assert ctx.get_tuning(name) == value
        for n, k, m in ((513, 528, 528), (129, 48, 272), (1024, 1024, 1024)):
            a, b = oracle.fill(oracle.FLOAT, n, k, m)
            c, _, _ = ctx.gemm_host(mm.FLOAT, mm.MULTIPLY, mm.ADD, a, b, n, k, m)
            ref = oracle.naive(oracle.FLOAT, oracle.MULTIPLY, oracle.ADD, a, b, n, k, m, threads=8)
            assert oracle.verify(oracle.FLOAT, c, ref) == -1, (variant, n, k, m)
            assert max_rel(c, ref) <= TOL["tcgen05_tf32"], (variant, n, k, m)


@pytest.mark.parametrize("variant", TCGEN05_VARIANTS, ids=_vid)
def test_tcgen05_tuning_variants_half(mm, oracle, variant):
    with mm.Context(0) as ctx:
        ctx.set_tuning(**variant)
        for n, k, m in ((513, 544, 544), (130, 96, 160), (1024, 1024, 1024)):
            a, b = half_inputs(oracle, n, k, m)
            c, _, _ = ctx.gemm_host(mm.HALF, mm.MULTIPLY, mm.ADD, a, b, n, k, m)
            exact = a.reshape(n, k).astype(np.float64) @ b.reshape(k, m).astype(np.float64)
            assert np.all(np.isfinite(c.astype(np.float32)))
            assert max_rel(c, exact) <= TOL["tcgen05_f16"], (variant, n, k, m)


def test_tuning_variants_agree_bit_for_bit(mm, oracle):
    """Tiles, ring depth, rasterisation and the epilogue route change WHERE a product is computed, never
    the order of the k-loop: every variant must give the default's bits (float 513 x 528 x 528)."""
    n, k, m = 513, 528, 528
    a, b = oracle.fill(oracle.FLOAT, n, k, m)
    outs = []
    for variant in TCGEN05_VARIANTS:
        with mm.Context(0) as ctx:
            ctx.set_tuning(**variant)
            outs.append(ctx.gemm_host(mm.FLOAT, mm.MULTIPLY, mm.ADD, a, b, n, k, m)[0].tobytes())
    assert all(o == outs[0] for o in outs)


@pytest.mark.parametrize("tile_rows", [0, 64, 128])
def test_dmma_tile_rows(mm, oracle, tile_rows):
    with mm.Context(0) as ctx:
        ctx.set_tuning(dmma_tile_rows=tile_rows)
        for n, k, m in ((130, 24, 136), (513, 528, 528), (1024, 1024, 1024)):
            a, b = oracle.fill(oracle.DOUBLE, n, k, m)
            c, _, _ = ctx.gemm_host(mm.DOUBLE, mm.MULTIPLY, mm.ADD, a, b, n, k, m)
            ref = oracle.naive(oracle.DOUBLE, oracle.MULTIPLY, oracle.ADD, a, b, n, k, m, threads=8)
            assert oracle.verify(oracle.DOUBLE, c, ref) == -1
            assert max_rel(c, ref) <= TOL["dmma_f64"]


@pytest.mark.parametrize("ring", [0, 1])
@pytest.mark.parametrize("dt,mp,rd", [("FLOAT", "ADD", "MIN"), ("FLOAT", "MULTIPLY", "ADD"), ("FLOAT", "MAX", "MIN"),
                                      ("INT32", "MULTIPLY", "ADD"), ("UINT32", "ADD", "MAX")])
def test_semiring_ring_and_staged_kernels_agree(mm, oracle, ring, dt, mp, rd):
    """4-byte types have two CUDA-core kernels (TMA ring | register-staged, knob semiring_ring): both bit-exact, on
    ragged shapes (rows past N and columns past M are zero-filled by TMA in the ring kernel, never stored)."""
    dtype, m_, r_ = getattr(mm, dt), getattr(mm, mp), getattr(mm, rd)
    flags = mm.FLAG_EXACT if (mp, rd) == ("MULTIPLY", "ADD") else 0
    with mm.Context(0) as ctx:
        ctx.set_tuning(semiring_ring=ring)
        for n, k, m in ((513, 528, 528), (1, 16, 16), (127, 64, 192), (300, 1024, 320)):
            a, b = oracle.fill(dtype, n, k, m, 31)
            c, _, _ = ctx.gemm_host(dtype, m_, r_, a, b, n, k, m, flags=flags)
            ref = oracle.naive(dtype, m_, r_, a, b, n, k, m, threads=8)
            assert c.tobytes() == ref.tobytes(), (ring, n, k, m)


# uint8_t on tcgen05 kind::i8 (SURVEY.md 8 f3): exact integer accumulation, bit-exact modulo 256
def _u8_inputs(n, k, m, seed):
    return special_inputs.full_range_bytes(n, k, m, seed)


@pytest.mark.parametrize("variant", [dict(), dict(cta_group=1), dict(block_n=128), dict(cta_group=1, block_n=128),
                                     dict(b_mn=0), dict(b_mn=0, block_n=128), dict(tma_store=0), dict(stages=3)], ids=_vid)
def test_uint8_tensor_path_bit_exact(mm, oracle, variant):
    assert mm.kernel_path(mm.UINT8) == "tcgen05_i8"
    with mm.Context(0) as ctx:
        ctx.set_tuning(**variant)
        for n, k, m in ((513, 576, 576), (1, 64, 64), (129, 128, 192), (1024, 1024, 1024)):
            a, b = _u8_inputs(n, k, m, 41)
            c, _, _ = ctx.gemm_host(mm.UINT8, mm.MULTIPLY, mm.ADD, a, b, n, k, m)
            ref = oracle.naive(oracle.UINT8, oracle.MULTIPLY, oracle.ADD, a, b, n, k, m, threads=8)
            assert c.tobytes() == ref.tobytes(), (variant, n, k, m)
            ct, _, _ = ctx.gemm_host(mm.UINT8, mm.MULTIPLY, mm.ADD, np.ascontiguousarray(a.reshape(n, k).T), b, n, k, m,
                                     flags=mm.FLAG_TRANSPOSED_A)
            assert ct.tobytes() == ref.tobytes(), ("transposed A", variant, n, k, m)


def test_uint8_accumulator_headroom_and_fallback(mm, oracle):
    """255^2 * K fits the 32-bit accumulator up to K = 33024 (all-255 inputs: the largest possible sum); longer K takes
    the CUDA-core kernel.  Both sides of the switch give the reference's bits."""
    for k in (33024, 33088):
        n, m = 3, 64
        a = np.full(n * k, 255, dtype=np.uint8)
        b = np.full(k * m, 255, dtype=np.uint8)
        c = mm.matrix_multiplication_kernel(a, b, n, k, m, dtype=mm.UINT8)
        ref = oracle.naive(oracle.UINT8, oracle.MULTIPLY, oracle.ADD, a, b, n, k, m, threads=8)
        assert c.tobytes() == ref.tobytes(), k
        a2, b2 = _u8_inputs(n, k, m, 43)
        c = mm.matrix_multiplication_kernel(a2, b2, n, k, m, dtype=mm.UINT8)
        assert c.tobytes() == oracle.naive(oracle.UINT8, oracle.MULTIPLY, oracle.ADD, a2, b2, n, k, m, threads=8).tobytes(), k


def test_tuning_rejects_out_of_range_values(mm):
    with mm.Context(0) as ctx:
        for bad in (dict(cta_group=3), dict(block_n=192), dict(stages=9), dict(stages=1), dict(dmma_tile_rows=32),
                    dict(l2_policy=7), dict(tma_store=2)):
            with pytest.raises(mm.MMError) as e:
                ctx.set_tuning(**bad)
            assert e.value.code == 1
        assert ctx.get_tuning("cta_group") == 2 and ctx.get_tuning("block_n") == 256


def test_tuning_defaults_come_from_the_environment_at_context_creation(mm, oracle, monkeypatch):
    monkeypatch.setenv("MM_TCGEN05_CTA_GROUP", "1")
    monkeypatch.setenv("MM_TCGEN05_STAGES", "3")
    monkeypatch.setenv("MM_TCGEN05_BLOCK_N", "999")     # out of range: ignored
    with mm.Context(0) as ctx:
        assert ctx.get_tuning("cta_group") == 1 and ctx.get_tuning("stages") == 3 and ctx.get_tuning("block_n") == 256
    monkeypatch.delenv("MM_TCGEN05_CTA_GROUP")
    with mm.Context(0) as ctx:
        assert ctx.get_tuning("cta_group") == 2


# ---------------------------------------------------------------------------------------------
# 2. semiring kernel under the DEFAULT flags; special values
# ---------------------------------------------------------------------------------------------
FLOATING = ("FLOAT", "DOUBLE", "HALF")


def signed_inputs(mm, dtype, n, k, m, seed, special=False):
    """Mixed-sign data without zeros; `special` sprinkles -0, +0, NaN and infinities (tests/golden/special_inputs.py)."""
    return special_inputs.signed(mm.NP_DTYPE[dtype], n, k, m, seed, special)


def _all_semirings():
    import gemm_hls_b200 as G
    cases = []
    for name, w in (("FLOAT", 16), ("DOUBLE", 8), ("HALF", 32), ("INT32", 16), ("UINT32", 16), ("UINT8", 64)):
        for mp in range(5):
            for rd in range(5):
                if (mp, rd) == (G.MULTIPLY, G.ADD) and name in FLOATING:
                    continue   # default flags send these to the tensor cores: covered by the tolerance tests
                cases.append((name, mp, rd, 65, 2 * w, 3 * w))
    return cases


@pytest.mark.parametrize("dt,mp,rd,n,k,m", _all_semirings())
def test_semiring_default_flags_bit_exact_on_signed_data(mm, oracle, dt, mp, rd, n, k, m):
    """flags = 0 — what a caller gets: every non-(Multiply,Add) semiring and every integer type, on mixed-sign
    finite data without zeros, bit for bit against Naive<> (float Min / Max run on the hardware FMNMX)."""
    dtype = getattr(mm, dt)
    a, b = signed_inputs(mm, dtype, n, k, m, seed=100 + 7 * mp + rd)
    c = mm.matrix_multiplication_kernel(a, b, n, k, m, dtype=dtype, map_op=mp, reduce_op=rd, flags=0)
    ref = oracle.naive(dtype, mp, rd, a, b, n, k, m, threads=8)
    assert c.tobytes() == ref.tobytes()


@pytest.mark.parametrize("n,k,m", [(256, 256, 256), (513, 528, 528), (1, 64, 64), (127, 64, 192), (300, 1024, 320)])
@pytest.mark.parametrize("dt,mp,rd", [("FLOAT", "ADD", "MIN"), ("FLOAT", "MULTIPLY", "MIN"), ("FLOAT", "MAX", "ADD"),
                                      ("FLOAT", "MIN", "MIN"), ("FLOAT", "ADD", "MAX"), ("DOUBLE", "ADD", "MAX"),
                                      ("HALF", "ADD", "MIN"), ("INT32", "MULTIPLY", "ADD"), ("UINT8", "MULTIPLY", "ADD")])
def test_semiring_default_flags_shapes(mm, oracle, dt, mp, rd, n, k, m):
    dtype, m_, r_ = getattr(mm, dt), getattr(mm, mp), getattr(mm, rd)
    w = mm.memory_width(dtype)
    k, m = (k + w - 1) // w * w, (m + w - 1) // w * w
    a, b = oracle.fill(dtype, n, k, m, 13)
    c = mm.matrix_multiplication_kernel(a, b, n, k, m, dtype=dtype, map_op=m_, reduce_op=r_, flags=0)
    ref = oracle.naive(dtype, m_, r_, a, b, n, k, m, threads=8)
    assert c.tobytes() == ref.tobytes()


@pytest.mark.parametrize("rec", GOLDEN_SPECIAL, ids=lambda r: "%s-%s-%dx%dx%d" % (r["config"], r["inputs"], r["n"], r["k"], r["m"]))
def test_golden_records_on_non_recipe_inputs(mm, rec):
    """Records produced by the reference's OWN Naive<> (tests/golden/make_golden_special.py) on inputs its recipe never
    draws: full-range bytes (uint8_t on tcgen05 kind::i8), mixed signs (default flags, FMNMX), NaN / signed zeros /
    infinities (MM_FLAG_EXACT).  Compared by SHA-256 with NaNs canonicalised — no oracle in between."""
    import hashlib
    dtype, n, k, m = rec["dtype"], rec["n"], rec["k"], rec["m"]
    a, b = special_inputs.make(rec["inputs"], mm.NP_DTYPE[dtype], n, k, m, rec["seed"])
    assert hashlib.sha256(a.tobytes()).hexdigest() == rec["a_sha256"] and hashlib.sha256(b.tobytes()).hexdigest() == rec["b_sha256"]
    flags = mm.FLAG_EXACT if rec["inputs"] == "special" else 0
    c = mm.matrix_multiplication_kernel(a, b, n, k, m, dtype=dtype, map_op=rec["map"], reduce_op=rec["reduce"], flags=flags)
    assert special_inputs.canonical_sha256(c) == rec["c_sha256_nan_canonical"]
    if rec["inputs"] != "special":   # the exact datapath reproduces the non-special records too
        ce = mm.matrix_multiplication_kernel(a, b, n, k, m, dtype=dtype, map_op=rec["map"], reduce_op=rec["reduce"],
                                             flags=mm.FLAG_EXACT)
        assert special_inputs.canonical_sha256(ce) == rec["c_sha256_nan_canonical"]


def _bits_equal_nan_aware(c, ref):
    """Bit equality, except that any NaN equals any NaN (payload / sign of a NaN produced by inf - inf or
    0 * inf is not specified by the reference's C++ either)."""
    cn, rn = np.isnan(c.astype(np.float64)), np.isnan(ref.astype(np.float64))
    if not np.array_equal(cn, rn):
        return False
    ui = {2: np.uint16, 4: np.uint32, 8: np.uint64}[c.dtype.itemsize]
    return np.array_equal(c.view(ui)[~cn], ref.view(ui)[~rn])


@pytest.mark.parametrize("dt", FLOATING)
@pytest.mark.parametrize("mp", range(5))
@pytest.mark.parametrize("rd", range(5))
def test_semiring_exact_flag_reproduces_special_values(mm, oracle, dt, mp, rd):
    """MM_FLAG_EXACT is the reference's datapath for EVERY input: NaN, -0 / +0 and infinities included."""
    dtype = getattr(mm, dt)
    w = mm.memory_width(dtype)
    n, k, m = 65, 2 * w, 3 * w
    a, b = signed_inputs(mm, dtype, n, k, m, seed=200 + 7 * mp + rd, special=True)
    c = mm.matrix_multiplication_kernel(a, b, n, k, m, dtype=dtype, map_op=mp, reduce_op=rd, flags=mm.FLAG_EXACT)
    ref = oracle.naive(dtype, mp, rd, a, b, n, k, m, threads=8)
    assert _bits_equal_nan_aware(c, ref)


@pytest.mark.parametrize("dt", ("DOUBLE", "HALF"))
@pytest.mark.parametrize("mp,rd", [(1, 2), (1, 3), (2, 3), (0, 2), (3, 1), (2, 2)])
def test_semiring_default_flags_special_values_non_float(mm, oracle, dt, mp, rd):
    """Only FLOAT has a hardware min/max substitution: double and half are the literal datapath with flags = 0 too."""
    dtype = getattr(mm, dt)
    w = mm.memory_width(dtype)
    n, k, m = 65, 2 * w, 3 * w
    a, b = signed_inputs(mm, dtype, n, k, m, seed=300 + 7 * mp + rd, special=True)
    c = mm.matrix_multiplication_kernel(a, b, n, k, m, dtype=dtype, map_op=mp, reduce_op=rd, flags=0)
    ref = oracle.naive(dtype, mp, rd, a, b, n, k, m, threads=8)
    assert _bits_equal_nan_aware(c, ref)


def test_float_default_minmax_documented_exception(mm, oracle):
    """include/mm_b200.h (MM_FLAG_EXACT): float Min / Max use FMNMX by default — it returns -0 for min(-0, +0)
    whichever comes first and drops NaN operands, where `(a < b) ? a : b` returns the second operand of a tie
    and lets a NaN in the second operand through.  This test pins that documented behaviour: with NaN-free data
    the two agree up to the SIGN of zero results; with NaNs the default never returns NaN from Min."""
    n, k, m = 65, 32, 48
    a, b = signed_inputs(mm, mm.FLOAT, n, k, m, seed=77, special=True)
    a[np.isnan(a) | np.isinf(a)] = 1.0
    b[np.isnan(b) | np.isinf(b)] = 2.0
    c = mm.matrix_multiplication_kernel(a, b, n, k, m, dtype=mm.FLOAT, map_op=mm.ADD, reduce_op=mm.MIN, flags=0)
    ref = oracle.naive(oracle.FLOAT, oracle.ADD, oracle.MIN, a, b, n, k, m, threads=8)
    assert np.array_equal(c, ref)                      # numerically equal (-0 == +0) everywhere
    a[3] = np.nan
    c = mm.matrix_multiplication_kernel(a, b, n, k, m, dtype=mm.FLOAT, map_op=mm.ADD, reduce_op=mm.MIN, flags=0)
    assert not np.any(np.isnan(c))                     # FMNMX dropped the NaN terms


# ---------------------------------------------------------------------------------------------
# 3. the multi-chunk host pipeline
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dt,mp,rd,n,k,m", [
    ("FLOAT", "MULTIPLY", "ADD", 1000, 512, 272),     # tcgen05: B prepared once (overlapped), 8 chunks of A
    ("HALF", "MULTIPLY", "ADD", 700, 256, 160),
    ("DOUBLE", "MULTIPLY", "ADD", 520, 264, 136),     # DMMA
    ("FLOAT", "ADD", "MIN", 777, 64, 144),            # semiring
    ("UINT8", "MULTIPLY", "ADD", 300, 128, 128),
])
def test_host_pipeline_with_several_chunks(mm, oracle, monkeypatch, dt, mp, rd, n, k, m):
    """mm_gemm_host cuts A / C into row chunks above 32 MiB (the bench's e2e figure runs that path);
    MM_HOST_CHUNK_ROWS forces the same code at test sizes.  Same bits as the single-chunk call."""
    dtype, m_, r_ = getattr(mm, dt), getattr(mm, mp), getattr(mm, rd)
    a, b = half_inputs(oracle, n, k, m) if dt == "HALF" else oracle.fill(dtype, n, k, m, 3)
    whole = mm.matrix_multiplication_kernel(a, b, n, k, m, dtype=dtype, map_op=m_, reduce_op=r_)
    monkeypatch.setenv("MM_HOST_CHUNK_ROWS", "128")
    chunked = mm.matrix_multiplication_kernel(a, b, n, k, m, dtype=dtype, map_op=m_, reduce_op=r_)
    assert chunked.tobytes() == whole.tobytes()
    if dt == "HALF":
        exact = a.reshape(n, k).astype(np.float64) @ b.reshape(k, m).astype(np.float64)
        assert max_rel(chunked, exact) <= TOL["tcgen05_f16"]
    else:
        ref = oracle.naive(dtype, m_, r_, a, b, n, k, m, threads=8)
        assert oracle.verify(dtype, chunked, ref) == -1
        if mm.kernel_path(dtype, m_, r_) == "semiring_simt":
            assert chunked.tobytes() == ref.tobytes()


# ---------------------------------------------------------------------------------------------
# 4. the row-block split (mm_multi_*) — same code as over NVLink, on one device listed several times
# ---------------------------------------------------------------------------------------------
MULTI_CASES = [
    ("FLOAT", "MULTIPLY", "ADD", 513, 528, 528),
    ("FLOAT", "MULTIPLY", "ADD", 1024, 1024, 1024),
    ("HALF", "MULTIPLY", "ADD", 513, 544, 544),
    ("DOUBLE", "MULTIPLY", "ADD", 300, 264, 136),
    ("FLOAT", "ADD", "MIN", 257, 192, 144),
    ("INT32", "MULTIPLY", "ADD", 130, 64, 96),
    ("UINT8", "MULTIPLY", "ADD", 513, 576, 576),
]


@pytest.mark.parametrize("gpus", [2, 3])
@pytest.mark.parametrize("dt,mp,rd,n,k,m", MULTI_CASES)
def test_multi_gemm_host_equals_single_context(mm, oracle, gpus, dt, mp, rd, n, k, m):
    """concat of the per-GPU C row-blocks == the single-GPU C bit for bit (SURVEY.md 8e "Check"), with B
    uploaded in slices and gathered by the library's kernels."""
    dtype, m_, r_ = getattr(mm, dt), getattr(mm, mp), getattr(mm, rd)
    a, b = half_inputs(oracle, n, k, m) if dt == "HALF" else oracle.fill(dtype, n, k, m, 17)
    single = mm.matrix_multiplication_kernel(a, b, n, k, m, dtype=dtype, map_op=m_, reduce_op=r_)
    with mm.Multi(gpus, devices=[0] * gpus) as multi:
        assert multi.peer_access
        for rep in range(2):   # the second call reuses buffers, slice tables and counters
            c, sec_dev, sec_wall = multi.gemm_host(dtype, m_, r_, a, b, n, k, m)
            assert c.tobytes() == single.tobytes(), (gpus, rep)
            assert 0 < sec_dev <= sec_wall


def _real_devices():
    try:
        import torch
        return torch.cuda.device_count()
    except Exception:
        return 0


@pytest.mark.skipif(_real_devices() < 2, reason="needs two GPUs (logs of 2- and 8-GPU runs in profiles/)")
@pytest.mark.parametrize("dt,mp,rd,n,k,m", MULTI_CASES + [("FLOAT", "MULTIPLY", "ADD", 4096, 2048, 4096),
                                                          ("HALF", "MULTIPLY", "ADD", 2048, 4096, 2048)])
def test_multi_gemm_host_over_nvlink(mm, oracle, dt, mp, rd, n, k, m):
    """The same check on DISTINCT devices: B's slices cross NVLink (peer loads in the gather kernel)."""
    dtype, m_, r_ = getattr(mm, dt), getattr(mm, mp), getattr(mm, rd)
    gpus = min(_real_devices(), 8)
    a, b = half_inputs(oracle, n, k, m) if dt == "HALF" else oracle.fill(dtype, n, k, m, 19)
    single = mm.matrix_multiplication_kernel(a, b, n, k, m, dtype=dtype, map_op=m_, reduce_op=r_)
    with mm.Multi(gpus) as multi:
        assert multi.peer_access
        for rep in range(2):
            c, _, _ = multi.gemm_host(dtype, m_, r_, a, b, n, k, m)
            assert c.tobytes() == single.tobytes(), (gpus, rep)
        multi.upload(dtype, a, b, n, k, m)
        multi.execute(dtype, m_, r_, n, k, m)
        assert multi.download(dtype, n, m).tobytes() == single.tobytes()


def test_multi_more_gpus_than_rows_or_slices(mm, oracle):
    n, k, m = 3, 64, 64          # 4 "GPUs": one has no rows; K has a single 64-row slice
    a, b = oracle.fill(oracle.FLOAT, n, k, m, 23)
    single = mm.matrix_multiplication_kernel(a, b, n, k, m)
    with mm.Multi(4, devices=[0, 0, 0, 0]) as multi:
        c, _, _ = multi.gemm_host(mm.FLOAT, mm.MULTIPLY, mm.ADD, a, b, n, k, m)
    assert c.tobytes() == single.tobytes()


def test_multi_device_resident_lifecycle(mm, oracle):
    """upload / execute / execute / download: RunHardware's sequence over G devices."""
    n, k, m = 640, 512, 384
    a, b = oracle.fill(oracle.FLOAT, n, k, m, 29)
    ref = oracle.naive(oracle.FLOAT, oracle.MULTIPLY, oracle.ADD, a, b, n, k, m, threads=8)
    single = mm.matrix_multiplication_kernel(a, b, n, k, m)
    with mm.Multi(2, devices=[0, 0]) as multi:
        multi.upload(mm.FLOAT, a, b, n, k, m)
        multi.execute(mm.FLOAT, mm.MULTIPLY, mm.ADD, n, k, m)
        sec_dev, sec_wall = multi.execute(mm.FLOAT, mm.MULTIPLY, mm.ADD, n, k, m)
        assert 0 < sec_dev <= sec_wall
        c = multi.download(mm.FLOAT, n, m)
        with pytest.raises(mm.MMError):
            multi.execute(mm.FLOAT, mm.MULTIPLY, mm.ADD, n + 1, k, m)   # no matching upload
    assert c.tobytes() == single.tobytes()
    assert oracle.verify(oracle.FLOAT, c, ref) == -1


def test_multi_rejects_transposed_a(mm, oracle):
    a, b = oracle.fill(oracle.FLOAT, 64, 64, 64)
    with mm.Multi(2, devices=[0, 0]) as multi:
        with pytest.raises(mm.MMError) as e:
            multi.gemm_host(mm.FLOAT, mm.MULTIPLY, mm.ADD, a, b, 64, 64, 64, flags=mm.FLAG_TRANSPOSED_A)
    assert e.value.code == 5


def test_default_entry_splits_over_mm_num_gpus(mm, oracle, tmp_path):
    """MatrixMultiplicationKernel's default context honours MM_NUM_GPUS (one process = one default, so this
    runs in a subprocess; with a single visible device the request fails loudly instead of shrinking)."""
    import subprocess
    import sys
    code = ("import numpy as np, gemm_hls_b200 as G, oracle as O\n"
            "a, b = O.fill(O.FLOAT, 300, 64, 64)\n"
            "try:\n"
            "    c = G.matrix_multiplication_kernel(a, b, 300, 64, 64)\n"
            "    ref = O.naive(O.FLOAT, O.MULTIPLY, O.ADD, a, b, 300, 64, 64)\n"
            "    print('OK' if O.verify(O.FLOAT, c, ref) == -1 else 'MISMATCH')\n"
            "except G.MMError as e:\n"
            "    print('ERR', e.code, e)\n")
    import torch
    env = dict(os.environ, MM_NUM_GPUS="2", PYTHONPATH=os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, env=env, timeout=300)
    out = r.stdout.strip().splitlines()[-1] if r.stdout.strip() else r.stderr[-300:]
    if torch.cuda.device_count() >= 2:
        assert out == "OK", r.stdout + r.stderr
    else:
        assert out.startswith("ERR 1") and "2 devices requested" in out, r.stdout + r.stderr


# ---------------------------------------------------------------------------------------------
# 5. checks that need a device
# ---------------------------------------------------------------------------------------------
def test_misaligned_device_pointers_are_rejected(mm):
    with mm.Context(0) as ctx:
        d = ctx.alloc(1 << 20)
        try:
            with pytest.raises(mm.MMError) as e:
                ctx.execute(mm.FLOAT, mm.MULTIPLY, mm.ADD, d + 4, d, d, 16, 16, 16)
            assert e.value.code == 1 and "16-byte aligned" in str(e.value)
            with pytest.raises(mm.MMError):
                ctx.enqueue(mm.FLOAT, mm.ADD, mm.MIN, d, d + 8, d, 16, 16, 16)
        finally:
            ctx.free(d)


def test_reserve_then_capture_without_warm_up(mm, oracle):
    """mm_context_reserve sizes the scratch, so the FIRST enqueue of a size may already be under stream capture;
    growth after a capture keeps the superseded scratch alive, so the captured graph stays replayable."""
    torch = pytest.importorskip("torch")
    n, k, m = 256, 256, 256
    a, b = oracle.fill(oracle.FLOAT, n, k, m)
    ref = oracle.naive(oracle.FLOAT, oracle.MULTIPLY, oracle.ADD, a, b, n, k, m, threads=8)
    dev = torch.device("cuda", 0)
    ta = torch.from_numpy(a.reshape(n, k)).to(dev)
    tb = torch.from_numpy(b.reshape(k, m)).to(dev)
    tc = torch.zeros((n, m), device=dev, dtype=torch.float32)
    with mm.Context(0) as ctx:
        ctx.execute(mm.FLOAT, mm.MULTIPLY, mm.ADD, ta.data_ptr(), tb.data_ptr(), tc.data_ptr(), 64, 64, 64)  # loads kernels
        ctx.reserve(mm.FLOAT, n, k, m)
        s = torch.cuda.Stream(device=dev)
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=s):
            ctx.enqueue(mm.FLOAT, mm.MULTIPLY, mm.ADD, ta.data_ptr(), tb.data_ptr(), tc.data_ptr(), n, k, m,
                        stream=torch.cuda.current_stream().cuda_stream)
        tc.zero_()
        g.replay()
        torch.cuda.synchronize()
        assert oracle.verify(oracle.FLOAT, tc.cpu().numpy(), ref) == -1
        # a larger problem after a capture: the old scratch stays alive, the graph still replays correctly
        big = torch.ones((512, 512), device=dev, dtype=torch.float32)
        out = torch.empty((512, 512), device=dev, dtype=torch.float32)
        ctx.execute(mm.FLOAT, mm.MULTIPLY, mm.ADD, big.data_ptr(), big.data_ptr(), out.data_ptr(), 512, 512, 512)
        tc.zero_()
        g.replay()
        torch.cuda.synchronize()
        assert oracle.verify(oracle.FLOAT, tc.cpu().numpy(), ref) == -1
