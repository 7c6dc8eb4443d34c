"""b200_supports_op on row-split weights (B200_TENSOR_FLAG_SPLIT, the op the plugin's split buffer type emits for --split-mode row):
F16 / BF16 weights are accepted with a shard table and with the NULL table llama.cpp probes before shards exist, in every layout
the per-shard dispatch can run; F32 weights, batched weights and any op other than MUL_MAT over a split tensor are refused; the
quantised decisions are the ones they were.  supports_op reads no device memory, so no GPU is needed."""
import ctypes as C

import pytest

SPLIT = 2


class Split(C.Structure):
    _fields_ = [("n_dev", C.c_int32), ("device", C.c_int32 * 16), ("shard", C.c_void_p * 16), ("row_low", C.c_int64 * 17)]


@pytest.fixture(scope="module")
def table():
    sp = Split()
    sp.n_dev = 2
    sp.device[0], sp.device[1] = 0, 1
    sp.shard[0], sp.shard[1] = 0x100000, 0x200000          # never dereferenced by supports_op
    sp.row_low[0], sp.row_low[1], sp.row_low[2] = 0, 768, 1536
    return sp


def split_w(b200, sp, t, K, N, ne2=1):
    data = C.addressof(sp) if sp is not None else 0
    return b200.tensor(data, t, [K, N, ne2], flags=b200.TENSOR_FLAG_WEIGHT | SPLIT)


def mm(b200, w, K, N, M, x_nb1=None, d_nb1=None, xt=None):
    x_nb1, d_nb1 = x_nb1 or K * 4, d_nb1 or N * 4
    x = b200.tensor(0x300000, xt if xt is not None else b200.F32, [K, M], nb=[4, x_nb1, x_nb1 * M, x_nb1 * M])
    d = b200.tensor(0x400000, b200.F32, [N, M], nb=[4, d_nb1, d_nb1 * M, d_nb1 * M])
    return b200.make_op(b200.OP_MUL_MAT, d, [w, x])


@pytest.mark.parametrize("with_table", [True, False])
@pytest.mark.parametrize("M", [1, 32, 33, 512])
@pytest.mark.parametrize("tname", ["F16", "BF16"])
def test_split_16bit_mul_mat_accepted(b200, table, tname, M, with_table):
    t = getattr(b200, tname)
    sp = table if with_table else None
    assert b200.supports(mm(b200, split_w(b200, sp, t, 4096, 1536), 4096, 1536, M))
    # layouts the tensor-core kernels refuse: every shard runs the float kernel
    assert b200.supports(mm(b200, split_w(b200, sp, t, 1004, 1536), 1004, 1536, M))                      # K % 8 != 0
    assert b200.supports(mm(b200, split_w(b200, sp, t, 4096, 1536), 4096, 1536, M, x_nb1=4097 * 4))     # x columns unaligned
    assert b200.supports(mm(b200, split_w(b200, sp, t, 4096, 1536), 4096, 1536, M, d_nb1=1600 * 4))     # strided dst


@pytest.mark.parametrize("with_table", [True, False])
def test_split_refusals(b200, table, with_table):
    sp = table if with_table else None
    K, N = 4096, 1536
    assert not b200.supports(mm(b200, split_w(b200, sp, b200.F32, K, N), K, N, 1))                      # F32 split weights
    for t in (b200.F16, b200.BF16, b200.Q4_K):
        w3 = split_w(b200, sp, t, K, N, ne2=2)
        x3 = b200.tensor(0x300000, b200.F32, [K, 1, 2])
        d3 = b200.tensor(0x400000, b200.F32, [N, 1, 2])
        assert not b200.supports(b200.make_op(b200.OP_MUL_MAT, d3, [w3, x3]))                             # ne[2] > 1
        w = split_w(b200, sp, t, K, N)
        x = b200.tensor(0x300000, b200.F32, [K, 1])
        assert not b200.supports(b200.make_op(b200.OP_MUL_MAT, b200.tensor(0x400000, b200.F32, [K, N]), [x, w]))   # split src1
        # MUL_MAT_ID over a split expert stack, GET_ROWS out of a split matrix, an element-wise op reading one
        ids = b200.tensor(0x500000, b200.I32, [1, 1])
        xe = b200.tensor(0x300000, b200.F32, [K, 1, 1])
        de = b200.tensor(0x400000, b200.F32, [N, 1, 1])
        assert not b200.supports(b200.make_op(b200.OP_MUL_MAT_ID, de, [split_w(b200, sp, t, K, N, ne2=1), xe, ids]))
        rows = b200.tensor(0x500000, b200.I32, [3])
        assert not b200.supports(b200.make_op(b200.OP_GET_ROWS, b200.tensor(0x400000, b200.F32, [K, 3]), [w, rows]))
    wf = split_w(b200, sp, b200.F16, K, N)
    assert not b200.supports(b200.make_op(b200.OP_CPY, b200.tensor(0x400000, b200.F32, [K, N]), [wf]))
    # 16-bit split weights take f32 activations only
    assert not b200.supports(mm(b200, split_w(b200, sp, b200.F16, K, N), K, N, 1, xt=b200.F16))


def test_split_table_device_count_checked(b200):
    sp = Split()
    for n_dev in (0, 17):
        sp.n_dev = n_dev
        assert not b200.supports(mm(b200, split_w(b200, sp, b200.BF16, 4096, 1536), 4096, 1536, 1))


@pytest.mark.parametrize("with_table", [True, False])
def test_split_quantised_decisions_unchanged(b200, table, with_table):
    sp = table if with_table else None
    K, N = 4096, 1536
    assert b200.supports(mm(b200, split_w(b200, sp, b200.Q4_K, K, N), K, N, 1))
    assert b200.supports(mm(b200, split_w(b200, sp, b200.Q4_K, K, N), K, N, 64))
    assert not b200.supports(mm(b200, split_w(b200, sp, b200.Q4_K, K, N), K, N, 1, x_nb1=4097 * 4))      # the quantiser's float4 loads
    assert not b200.supports(mm(b200, split_w(b200, sp, b200.Q4_K, 4000, N), 4000, N, 1))                 # K not whole super-blocks
