"""Pins tests/fusion_ref.py, the stage references of the fused decode layers (no GPU)."""
import numpy as np
import pytest

import fusion_ref as FR
import reflib as R
from util import rand_quant_rows


@pytest.mark.parametrize("t", R.QUANT_TYPES)
def test_float64_product_matches_oracle_mul_mat(t):
    rng = np.random.default_rng(40 + t)
    N, K = 48, 2048
    W = rand_quant_rows(t, N, K, rng)
    x = (rng.standard_normal((3, K)) * np.array([[1.0], [1e-3], [30.0]])).astype(np.float32)
    want = R.orc_mul_mat(t, W, x, N, K)
    got = FR.mm_f64(t, W, x, K)
    assert np.abs(got - want).max() <= FR.REL * np.abs(want).max()
    rows = np.array([0, 5, 47])
    assert np.abs(FR.mm_f64(t, W, x, K, rows=rows) - got[:, rows]).max() <= 1e-12 * np.abs(want).max()


def test_flip_bound_flags_a_hand_placed_tie():
    rng = np.random.default_rng(3)
    K = 512
    h = rng.uniform(-1, 1, (1, K)).astype(np.float32)
    h[0, 0] = 1.0                                     # block maximum: iscale = 127 in block 0
    h[0, 7] = np.float32(40.5 / 127)                  # |h * iscale| = 40.5 (to f32 rounding): a tie
    W = rng.uniform(-1, 1, (4, K))
    mask, step = FR.ambiguous(h, R.Q4_K, 3e-6)
    assert mask[0, 7]
    tol = FR.flip_bound(h, R.Q4_K, W, 3e-6, scale=1.0)
    extra = tol - FR.REL
    assert np.all(extra >= step[0, 7] * np.abs(W[:, 7]) * (1 - 1e-12))


@pytest.mark.parametrize("t", [R.Q4_K, R.Q8_0])
def test_flip_bound_is_tight_without_near_ties(t):
    rng = np.random.default_rng(4)
    K = 1024
    be = 256 if R.act_type(t) == R.Q8_K else 32
    # every element an integer + 0.25 steps of its block: far from any rounding boundary
    q = rng.integers(-120, 120, (2, K)).astype(np.float64) + 0.25
    q[:, ::be] = 127.0
    h = (q / 127.0 * 0.7).astype(np.float32)
    W = rng.uniform(-1, 1, (6, K))
    tol = FR.flip_bound(h, t, W, 3e-6, scale=2.0)
    assert np.array_equal(tol, np.full((2, 6), FR.REL * 2.0))


@pytest.mark.parametrize("kvt", [R.F16, R.Q8_0, R.Q4_0])
def test_kv_bytes_rule(kvt):
    rng = np.random.default_rng(5 + kvt)
    x = rng.standard_normal((8, 128)).astype(np.float32)
    x[6] = 0                                          # an all-zero row: d = 0, every quant zero (q4_0: the offset 8)
    if kvt == R.F16:
        b = x.astype(np.float16).view(np.uint8)
    else:
        b = R.orc_quantize_act(kvt, x)
    assert FR.kv_bytes_ok(b, x, kvt, 0.0).all()
    assert FR.kv_bytes_ok(b, x, kvt, 1e-6 * np.abs(x).max(1)).all()
    assert FR.kv_bytes_ok(b[6:7], x[6:7], kvt, 0.0).all()
    if kvt != R.F16:
        nz = b[6:7].copy()
        nz[0, 2] ^= 1                                 # a nonzero quant in the zero block
        assert not FR.kv_bytes_ok(nz, x[6:7], kvt, 0.0).all()
    bad = b.copy()
    if kvt == R.F16:
        v = bad.view(np.uint16)
        v[2, 9] ^= 1                                  # one ulp off, not a tie
        flagged = (2, 9)
    else:
        bb = R.BLOCK[kvt][1]
        bad[3, bb + 5] ^= 1 if kvt == R.Q4_0 else 2   # second block, low nibble / int8 changed
        flagged = (3, 32 + 3) if kvt == R.Q8_0 else (3, 32 + 3)
    ok = FR.kv_bytes_ok(bad, x, kvt, 1e-7 * np.abs(x).max(1))
    assert not ok[flagged] and ok.sum() == ok.size - 1
