"""BF16 weights for the test-side reference (no GPU): the CPU backend's arithmetic for a BF16 weight MUL_MAT.

ggml converts src1 to the weight's vec_dot_type BF16 with ggml_compute_fp32_to_bf16 (round-to-nearest-even; NaN -> quiet NaN
keeping the high half), multiplies exact bf16 x bf16 products and accumulates them.  The reference here sums in float64, like the
C oracle's F16 branch, so a device result differs from it only by the f32 rounding of the device's own additions.

`with_bf16(monkeypatch)` teaches reflib the type for one test: BF16 joins reflib.BLOCK and reflib.orc_mul_mat (through which
oracle/llama_forward.py multiplies) handles BF16 here and defers every other type to the C oracle."""
import numpy as np

import reflib as R

BF16 = 30                      # ggml type id (ggml.h GGML_TYPE_BF16)


def f32_to_bf16_bits(x):
    """ggml_compute_fp32_to_bf16 over an array: uint16 bits"""
    u = np.asarray(x, np.float32).reshape(-1).view(np.uint32).astype(np.uint64)
    nan = (u & 0x7FFFFFFF) > 0x7F800000
    r = (u + 0x7FFF + ((u >> 16) & 1)) >> 16
    return np.where(nan, (u >> 16) | 64, r).astype(np.uint16).reshape(np.shape(x))


def bf16_bits_to_f32(b):
    return (np.asarray(b, np.uint16).astype(np.uint32) << 16).view(np.float32)


def round_bf16(x):
    return bf16_bits_to_f32(f32_to_bf16_bits(x))


def mul_mat_bf16(W, x, N, K):
    """W raw bytes of N BF16 rows of K, x f32 [M, K] -> f32 [M, N]: x rounded to bf16, products summed in float64"""
    w = bf16_bits_to_f32(np.ascontiguousarray(W, np.uint8)[:N * K * 2].view(np.uint16)).reshape(N, K).astype(np.float64)
    xr = round_bf16(np.ascontiguousarray(x, np.float32)).astype(np.float64)
    return (xr @ w.T).astype(np.float32)


def with_bf16(monkeypatch):
    monkeypatch.setitem(R.BLOCK, BF16, (1, 2))
    orc = R.orc_mul_mat

    def orc_mul_mat(t, W, x, N, K):
        return mul_mat_bf16(W, x, N, K) if t == BF16 else orc(t, W, x, N, K)
    monkeypatch.setattr(R, "orc_mul_mat", orc_mul_mat)
