"""The test-side BF16 MUL_MAT_ID reference (tests/bf16_moe_ref.py, no GPU): every (token, slot) pair against a per-pair BF16 matmul of its
expert and its activation column, for both activation layouts (one column per token, or one per pair); and with_bf16_moe routing the oracle's
MUL_MAT_ID to it for BF16 only."""
import numpy as np
import pytest

import bf16_moe_ref as BM
import bf16_ref as B
import reflib as R


def rand_bf16_bytes(rng, n):
    return B.f32_to_bf16_bits(rng.standard_normal(n).astype(np.float32) * 0.05).view(np.uint8)


@pytest.mark.parametrize("b_ne1", [1, 2])
def test_mul_mat_id_bf16_matches_per_pair_matmul(b_ne1):
    rng = np.random.default_rng(7 + b_ne1)
    n_expert, n_used, n_tok, N, K = 5, 2, 9, 24, 72
    As = rand_bf16_bytes(rng, n_expert * N * K)
    b = rng.standard_normal((n_tok, b_ne1, K)).astype(np.float32)
    ids = np.stack([rng.choice(n_expert - 1, n_used, replace=False) for _ in range(n_tok)]).astype(np.int32)   # expert 4 idle
    got = BM.mul_mat_id_bf16(As, b, ids, N, K, n_expert)
    assert got.shape == (n_tok, n_used, N) and got.dtype == np.float32
    row = N * K * 2
    for t in range(n_tok):
        for s in range(n_used):
            e = ids[t, s]
            want = B.mul_mat_bf16(As[e * row:(e + 1) * row], b[t, s % b_ne1][None], N, K)[0]
            assert np.array_equal(got[t, s], want), (t, s)


def test_with_bf16_moe_routes_only_bf16_mul_mat_id(monkeypatch):
    seen = []
    monkeypatch.setattr(R, "orc_mul_mat_id", lambda *a: seen.append(a[0]) or "oracle")
    BM.with_bf16_moe(monkeypatch)
    rng = np.random.default_rng(3)
    As = rand_bf16_bytes(rng, 2 * 8 * 16)
    b = rng.standard_normal((3, 1, 16)).astype(np.float32)
    ids = np.array([[0, 1], [1, 0], [1, 1]], np.int32)
    assert isinstance(R.orc_mul_mat_id(B.BF16, As, b, ids, 8, 16, 2), np.ndarray)
    assert R.orc_mul_mat_id(R.F16, As, b, ids, 8, 16, 2) == "oracle"
    assert seen == [R.F16]
