"""GPU parity of the prompt-batch GEMMs against the oracle's mul_mat (ggml_compute_forward_mul_mat with q8_K / q8_0 activations):
the tcgen05 kind::f16 GEMM (gemm_tc.cu: K-quants, the default for more than 32 token columns; its 32- and 64-token tiles and split-K
are exercised in a subprocess with GGML_B200_TC_MIN_M=5), the mma.sync tile GEMM (gemm_mma.cu: all five formats; the default for
Q4_0 / Q8_0, for K-quants selected with GGML_B200_NO_GEMM_TC=1).  The integer stage is the CPU's exactly, so the results agree
to f32 summation order: 3e-6 relative."""
import os
import subprocess
import sys
import numpy as np
import pytest

import reflib as R
from util import dev_bytes, rand_quant_rows, to_dev

pytestmark = pytest.mark.gpu


def gpu_mul_mat(b200, ctx, t, W, x, N, K):
    M = x.shape[0]
    Wd = dev_bytes(W.size + 256, 0)
    Wd[:W.size] = to_dev(W)
    xd = to_dev(x)
    out = dev_bytes(M * N * 4, 0xFF)
    op = b200.make_op(b200.OP_MUL_MAT, b200.tensor(out.data_ptr(), b200.F32, [N, M]),
                      [b200.tensor(Wd.data_ptr(), t, [K, N], flags=1), b200.tensor(xd.data_ptr(), b200.F32, [K, M])])
    assert b200.supports(op)
    ctx.compute_op(op)
    ctx.sync()
    return out.cpu().numpy().view(np.float32).reshape(M, N)


@pytest.mark.parametrize("N,K,M", [(128, 256, 16), (128, 512, 128), (256, 1024, 130), (128, 4096, 9), (384, 2048, 300), (1024, 4096, 512),
                                   (256, 5632, 32), (1024, 14336, 32)])      # the last two: split-K with uneven / 8 slices, a quarter-full token tile
@pytest.mark.parametrize("t", R.QUANT_TYPES)
def test_gemm_vs_oracle(b200, ctx, t, N, K, M):
    rng = np.random.default_rng(N + K + M + t)
    W = rand_quant_rows(t, N, K, rng)
    x = (rng.standard_normal((M, K)) * rng.uniform(0.1, 4.0, (M, 1))).astype(np.float32)
    got = gpu_mul_mat(b200, ctx, t, W, x, N, K)
    assert np.isfinite(got).all()
    rows = np.unique(np.concatenate([np.arange(min(N, 8)), rng.integers(0, N, 8), [N - 1, N - 128, 127 if N > 127 else 0]]))
    cols = np.unique(np.concatenate([np.arange(min(M, 4)), rng.integers(0, M, 6), [M - 1]]))
    rb = R.row_size(t, K)
    want = R.orc_mul_mat(t, W.reshape(N, rb)[rows].reshape(-1), x[cols], len(rows), K)
    sub = got[np.ix_(cols, rows)]
    scale = max(np.abs(want).max(), 1e-6)
    assert np.abs(sub - want).max() <= 3e-6 * scale, np.abs(sub - want).max() / scale



@pytest.mark.parametrize("t", R.QUANT_TYPES)
def test_gemm_mma_whole_matrix_and_determinism(b200, ctx, t):
    """every element of a multi-tile product (2 row tiles x 3 token tiles, the last one ragged) and run-to-run bit reproducibility"""
    rng = np.random.default_rng(90 + t)
    N, K, M = 256, 1280, 300
    W = rand_quant_rows(t, N, K, rng)
    x = rng.standard_normal((M, K)).astype(np.float32)
    l0 = ctx.launches()
    got = gpu_mul_mat(b200, ctx, t, W, x, N, K)
    assert ctx.launches() - l0 == 2, "pack + gemm_mma"
    want = R.orc_mul_mat(t, W, x, N, K)
    assert np.abs(got - want).max() <= 3e-6 * np.abs(want).max()
    assert np.array_equal(got, gpu_mul_mat(b200, ctx, t, W, x, N, K))


def _run_gemm_cases(env_extra, cases, tag):
    """runs K-quant matmuls in a fresh process (the dispatch switches are read once per process) and compares every element with the oracle"""
    env = dict(os.environ, **env_extra)
    code = ("import sys; sys.path.insert(0, %r); sys.path.insert(0, %r)\n"
            "import numpy as np, reflib as R\n"
            "from conftest import load_package\n"
            "from util import dev_bytes, rand_quant_rows, to_dev\n"
            "b200 = load_package(); ctx = b200.Context(0)\n"
            "for t in (R.Q4_K, R.Q5_K, R.Q6_K):\n"
            "    for (N, K, M) in %r:\n"
            "        rng = np.random.default_rng(t + N + K + M)\n"
            "        W = rand_quant_rows(t, N, K, rng); x = (rng.standard_normal((M, K)) * rng.uniform(0.1, 4.0, (M, 1))).astype(np.float32)\n"
            "        Wd = dev_bytes(W.size + 256, 0); Wd[:W.size] = to_dev(W); xd = to_dev(x); out = dev_bytes(M * N * 4, 0xFF)\n"
            "        op = b200.make_op(b200.OP_MUL_MAT, b200.tensor(out.data_ptr(), b200.F32, [N, M]), [b200.tensor(Wd.data_ptr(), t, [K, N], flags=1), b200.tensor(xd.data_ptr(), b200.F32, [K, M])])\n"
            "        ctx.compute_op(op); ctx.sync()\n"
            "        got = out.cpu().numpy().view(np.float32).reshape(M, N); want = R.orc_mul_mat(t, W, x, N, K)\n"
            "        err = np.abs(got - want).max() / np.abs(want).max()\n"
            "        assert np.isfinite(got).all() and err <= 3e-6, (t, N, K, M, err)\n"
            "        ctx.compute_op(op); ctx.sync()\n"
            "        assert np.array_equal(got, out.cpu().numpy().view(np.float32).reshape(M, N)), 'run-to-run reproducibility'\n"
            "print(%r)\n") % (os.path.dirname(os.path.abspath(__file__)), os.path.dirname(os.path.dirname(os.path.abspath(__file__))), cases, tag)
    p = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, timeout=900)
    assert p.returncode == 0 and tag in p.stdout, p.stdout[-500:] + p.stderr[-1500:]


def test_gemm_tc_small_token_tiles_and_split_k():
    """gemm_tc.cu from 5 token columns up: 32- and 64-token tiles, ragged tiles, split-K with uneven slices (K = 5632: 22 super-blocks),
    a single super-block, multi-row-tile grids -- every element against the oracle, bit-reproducible run to run"""
    _run_gemm_cases({"GGML_B200_TC_MIN_M": "5"}, [(128, 256, 5), (256, 1024, 17), (128, 4096, 32), (256, 5632, 32), (384, 2048, 48), (128, 1536, 64),
                                                  (256, 768, 100), (128, 512, 129)], "GEMM_TC SMALL OK")


def test_gemm_mma_still_green_for_k_quants():
    """GGML_B200_NO_GEMM_TC=1 sends K-quant prompt batches back to the mma.sync tile GEMM"""
    _run_gemm_cases({"GGML_B200_NO_GEMM_TC": "1"}, [(256, 1024, 130), (128, 2048, 300)], "GEMM_MMA KQ OK")
