"""The reference's OWN op-parity harness against the product: llama.cpp's unmodified tests/test-backend-ops.cpp (built into
oracle/_ref by oracle/Makefile) loads libggml-b200.so through GGML_BACKEND_PATH, runs every case of the hot-path ops on
the B200 backend and on the reference CPU backend, and compares them with its own NMSE limits (1e-7 default, 5e-4 for
MUL_MAT / MUL_MAT_ID / FLASH_ATTN_EXT; SURVEY.md 4).  test-backend-ops counts "not supported" as a pass, so the test
also requires a minimum number of cases that really RAN on the device for every op of the path (SURVEY.md 8b)."""
import os
import re
import subprocess

import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = os.path.join(ROOT, "oracle", "_ref")
EXE = os.path.join(REF, "test-backend-ops")
PLUGIN = os.path.join(ROOT, "cortex.llamacpp_b200", "libggml-b200.so")

# op -> minimum number of cases that must have executed on the B200 backend (round-1 run: profiles/r1_test_backend_ops.txt)
MIN_RAN = {"MUL_MAT": 240, "MUL_MAT_ID": 100, "FLASH_ATTN_EXT": 620, "RMS_NORM": 8, "ROPE": 144, "CPY": 48, "SOFT_MAX": 78,
           "GET_ROWS": 30, "ADD": 24, "MUL": 24, "DIV": 24, "SILU": 2, "ARGSORT": 6, "SUM_ROWS": 1, "SCALE": 1, "CONT": 6, "ARGMAX": 6}
ANSI = re.compile(r"\x1b\[[0-9;]*m")


@pytest.mark.parametrize("op", sorted(MIN_RAN))
def test_reference_test_backend_ops(op):
    if not (os.path.exists(EXE) and os.path.exists(PLUGIN)):
        pytest.skip("needs a llama.cpp checkout: make -C oracle ref REF=<llama.cpp> && make -C cortex.llamacpp_b200 backend REF=<llama.cpp>")
    env = dict(os.environ)
    env["GGML_BACKEND_PATH"] = PLUGIN
    env["LD_LIBRARY_PATH"] = os.path.join(ROOT, "cortex.llamacpp_b200") + ":" + REF + ":" + env.get("LD_LIBRARY_PATH", "")
    p = subprocess.run([EXE, "test", "-b", "B2000", "-o", op], env=env, capture_output=True, text=True, timeout=1800)
    out = ANSI.sub("", p.stdout + p.stderr)
    lines = out.splitlines()
    ok = sum(1 for ln in lines if ln.rstrip().endswith("OK") and op in ln)
    fail = [ln for ln in lines if "FAIL" in ln]
    ns = sum(1 for ln in lines if "not supported" in ln)
    print("BACKEND_OPS %-16s ok=%d fail=%d not_supported=%d rc=%d" % (op, ok, len(fail), ns, p.returncode))
    assert "Backend B2000" in out or "B2000" in out, "the B200 backend was not enumerated:\n" + out[-600:]
    assert not fail, "\n".join(fail[:10])
    assert p.returncode == 0, out[-800:]
    assert ok >= MIN_RAN[op], "only %d %s cases ran on the device (%d not supported)" % (ok, op, ns)
