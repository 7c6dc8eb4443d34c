"""The test-side BF16 reference (tests/bf16_ref.py, no GPU): its fp32 -> bf16 rounding against torch's, bit for bit, and the
16-bit weight matmuls (BF16 here, F16 in the C oracle) against a float64 matmul of operands rounded by torch."""
import numpy as np
import pytest

import bf16_ref as B
import reflib as R


def torch_bf16_bits(x):
    import torch
    return torch.from_numpy(np.asarray(x, np.float32)).to(torch.bfloat16).view(torch.int16).numpy().view(np.uint16)


def bits_to_f32(u32):
    return np.asarray(u32, np.uint32).view(np.float32)


def test_bf16_rounding_random_values():
    rng = np.random.default_rng(1)
    x = (rng.standard_normal(200000) * np.exp(rng.uniform(-40, 40, 200000))).astype(np.float32)
    assert np.array_equal(B.f32_to_bf16_bits(x), torch_bf16_bits(x))


def test_bf16_rounding_exact_ties_both_parities():
    # low half exactly 0x8000: halfway between two bf16 values; the even neighbour wins whichever parity the high half has
    hi = np.array([0x3F80, 0x3F81, 0x4049, 0x404A, 0xC2F6, 0xC2F7, 0x0001, 0x0002, 0x7F7E, 0x7F7F], np.uint32)
    x = bits_to_f32((hi << 16) | 0x8000)
    got = B.f32_to_bf16_bits(x)
    assert np.array_equal(got, torch_bf16_bits(x))
    assert np.array_equal(got, np.where(hi & 1, hi + 1, hi).astype(np.uint16)), "ties must round to even"
    near = bits_to_f32(np.concatenate([(hi << 16) | 0x7FFF, (hi << 16) | 0x8001]))      # just below / above the tie
    assert np.array_equal(B.f32_to_bf16_bits(near), torch_bf16_bits(near))


def test_bf16_rounding_subnormals_inf_nan():
    sub = bits_to_f32(np.array([0x00000001, 0x00007FFF, 0x00008000, 0x00018000, 0x007FFFFF, 0x80000001, 0x80408000, 0x00400000], np.uint32))
    special = np.array([np.inf, -np.inf, 0.0, -0.0, np.finfo(np.float32).max, -np.finfo(np.float32).max], np.float32)
    x = np.concatenate([sub, special])
    assert np.array_equal(B.f32_to_bf16_bits(x), torch_bf16_bits(x))
    # NaN: ggml forces a quiet NaN with the input's high half (0x7FC0 for the default NaN); torch's vectorised CPU conversion emits
    # 0xFFFF.  NaN payloads carry no value, so NaN is compared as a class: both results quiet NaNs
    nans = bits_to_f32(np.array([0x7FC00000, 0xFFC00000, 0x7F800001, 0x7FBFFFFF], np.uint32))
    got, ref = B.f32_to_bf16_bits(nans), torch_bf16_bits(nans)
    for g in (got, ref):
        assert np.all((g & 0x7F80) == 0x7F80) and np.all((g & 0x40) != 0), g
    assert got[0] == 0x7FC0 and got[1] == 0xFFC0


@pytest.mark.parametrize("t", [R.F16, B.BF16])
@pytest.mark.parametrize("N,K,M", [(7, 64, 1), (33, 1000, 3), (16, 4104, 5)])
def test_16bit_mul_mat_matches_float64_of_rounded_operands(t, N, K, M):
    import torch
    rng = np.random.default_rng(N * K + M + t)
    w = torch.from_numpy((rng.standard_normal((N, K)) * 0.05).astype(np.float32))
    x = (rng.standard_normal((M, K))).astype(np.float32)
    dt = torch.float16 if t == R.F16 else torch.bfloat16
    wq = w.to(dt)
    raw = wq.view(torch.int16).numpy().view(np.uint8).reshape(-1)
    got = R.orc_mul_mat(t, raw, x, N, K) if t == R.F16 else B.mul_mat_bf16(raw, x, N, K)
    want = torch.from_numpy(x).to(dt).double().numpy() @ wq.double().numpy().T
    assert np.abs(got - want).max() <= 1e-6 * np.abs(want).max()


def test_with_bf16_extends_reflib_for_one_test_only(monkeypatch):
    rng = np.random.default_rng(3)
    N, K = 5, 64
    x = rng.standard_normal((2, K)).astype(np.float32)
    wb = B.f32_to_bf16_bits(rng.standard_normal((N, K)).astype(np.float32) * 0.1).view(np.uint8).reshape(-1)
    wf = (rng.standard_normal((N, K)) * 0.1).astype(np.float16).view(np.uint8).reshape(-1)
    f16_before = R.orc_mul_mat(R.F16, wf, x, N, K)
    with monkeypatch.context() as m:
        B.with_bf16(m)
        assert R.row_size(B.BF16, K) == 2 * K
        assert np.array_equal(R.orc_mul_mat(B.BF16, wb, x, N, K), B.mul_mat_bf16(wb, x, N, K))
        assert np.array_equal(R.orc_mul_mat(R.F16, wf, x, N, K), f16_before)       # other types still go to the C oracle
    assert B.BF16 not in R.BLOCK
