"""BF16 MoE experts for the test-side reference (no GPU): the CPU backend's arithmetic for a BF16 MUL_MAT_ID, built on bf16_ref.

`with_bf16_moe(monkeypatch)` extends bf16_ref.with_bf16 for one test: reflib.orc_mul_mat_id (through which oracle/llama_forward.py's
moe_ffn multiplies the experts) also handles BF16 here and defers every other type to the C oracle."""
import numpy as np

import bf16_ref as B
import reflib as R


def mul_mat_id_bf16(As, b, ids, N, K, n_expert):
    """reflib.orc_mul_mat_id for BF16 experts: As bytes of [n_expert, N, K]; b f32 [n_tok, b_ne1, K]; ids i32 [n_tok, n_used] ->
    f32 [n_tok, n_used, N], dst[t, s] = As[ids[t, s]] . b[t, s % b_ne1]"""
    b = np.ascontiguousarray(b, np.float32)
    ids = np.asarray(ids, np.int32)
    n_tok, n_used = ids.shape
    A = np.ascontiguousarray(As, np.uint8)[:n_expert * N * K * 2]
    dst = np.zeros((n_tok, n_used, N), np.float32)
    for e in range(n_expert):
        t, s = np.nonzero(ids == e)
        if t.size:
            dst[t, s] = B.mul_mat_bf16(A[e * N * K * 2:(e + 1) * N * K * 2], b[t, s % b.shape[1]], N, K)
    return dst


def with_bf16_moe(monkeypatch):
    B.with_bf16(monkeypatch)
    orc_id = R.orc_mul_mat_id

    def orc_mul_mat_id(t, As, b, ids, N, K, n_expert):
        return mul_mat_id_bf16(As, b, ids, N, K, n_expert) if t == B.BF16 else orc_id(t, As, b, ids, N, K, n_expert)
    monkeypatch.setattr(R, "orc_mul_mat_id", orc_mul_mat_id)
