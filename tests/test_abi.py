"""The C-ABI library loads and exports every symbol include/go1mpc.h declares; without a
GPU every compute entry fails loudly (no CPU fallback)."""
import ctypes
import os
import re
import subprocess
import sys

import quadrupedal_loco_b200 as q

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_header_symbols_exported():
    hdr = open(os.path.join(ROOT, "include", "go1mpc.h")).read()
    declared = set(re.findall(r"\b(go1mpc_[a-z0-9_]+)\s*\(", hdr))
    assert declared, "no declarations found"
    assert declared == set(q.EXPORTED_SYMBOLS)
    lib = q.load_library()
    for s in declared:
        assert hasattr(lib, s), f"{s} not exported"


def test_version_and_strides():
    lib = q.load_library()
    assert b"sm_100a" in lib.go1mpc_version()
    for nh in (3, 4, 10, 20, 40):
        assert lib.go1mpc_body_in_stride(nh) == q.body_in_stride(nh)
        assert lib.go1mpc_body_out_stride(nh) == q.body_out_stride(nh)
        assert lib.go1mpc_body_diag_stride(nh) == q.body_diag_stride(nh)
        assert q.body_in_stride(nh) % 2 == 0 and q.body_out_stride(nh) % 2 == 0   # TMA: 16-byte records
        assert lib.go1mpc_body_tick_in_stride(nh) == q.body_tick_in_stride(nh)


def test_split_body_record_is_a_partition_of_the_full_record():
    """Resident entry: tx | tick record | warm start together hold every double of the full record."""
    import numpy as np
    nh, B = 10, 5
    rec = np.arange(B * q.body_in_stride(nh), dtype=np.float64).reshape(B, -1) + 1.0
    rec[:, 36 + 11 * nh:] = 0.0
    tx, xw, tick = q.split_body_record(nh, rec)
    assert tx.shape == (B, 28) and tick.shape == (B, q.body_tick_in_stride(nh)) and xw.shape == (B, 2 * nh)
    back = np.zeros_like(rec)
    back[:, :27] = tx[:, :27]; back[:, 27:36] = tick[:, :9]
    back[:, 36:36 + 2 * nh] = xw; back[:, 36 + 2 * nh:36 + 11 * nh] = tick[:, 9:9 + 9 * nh]
    np.testing.assert_array_equal(back, rec)
    assert (tx[:, 27] == 0).all() and (tick[:, 9 + 9 * nh:] == 0).all()


def test_no_device_is_an_error_not_a_fallback():
    """In a child process that sees no CUDA device (CUDA_VISIBLE_DEVICES empty), so the check also runs where a GPU is."""
    code = (f"import sys; sys.path.insert(0, {ROOT!r})\n"
            "import quadrupedal_loco_b200 as q\n"
            "try:\n    q.Go1Mpc()\nexcept q.Go1MpcError:\n    sys.exit(0)\n"
            "sys.exit('Go1Mpc() succeeded without a CUDA device')\n")
    r = subprocess.run([sys.executable, "-c", code], env=dict(os.environ, CUDA_VISIBLE_DEVICES=""), capture_output=True,
                       text=True, timeout=300)
    assert r.returncode == 0, r.stderr[-2000:]


def test_product_does_not_touch_oracle():
    """The product package must not import, link or reference anything under oracle/."""
    pkg = os.path.join(ROOT, "quadrupedal_loco_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h", ".hpp", ".cpp")):
                txt = open(os.path.join(dirpath, f), errors="ignore").read()
                assert "oracle_lib" not in txt and "liboracle" not in txt and "go1_oracle" not in txt, f
