"""oracle/nrc.cpp's hash-grid and one-blob encodings against the reference's own tiny-cuda-nn kernels (kernel_grid<__half,3,2>,
kernel_one_blob_soa<__half>) compiled from the reference's vendored tiny-cuda-nn into oracle/_ref/libtcnn_ref.so with
-fmad=false, i.e. under the oracle's arithmetic model (the reference's own build contracts a*b+c into FMAs, which no CPU
restatement can follow bit for bit; what is compared here is the algorithm): every half bit-identical.  The kernels' outputs are
stored in tests/golden/golden_tcnn_ref.npz (written by `python tests/tcnn_ref_check.py --write-golden`), so the check needs
neither the reference tree nor a GPU; it runs in a child process like the live check does."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden", "golden_tcnn_ref.npz")


def test_oracle_encoding_equals_tcnn_kernels():
    proc = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "tcnn_ref_check.py"), "--golden", GOLDEN],
                          capture_output=True, text=True, timeout=240)
    line = proc.stdout.strip().splitlines()[-1] if proc.stdout.strip() else ""
    assert proc.returncode == 0, f"rc={proc.returncode} {line} {proc.stderr[-400:]}"
    result = json.loads(line)
    assert result["grid"]["mismatches"] == 0 and result["oneblob"]["mismatches"] == 0, line
    assert result["grid"]["all_rows_equal"] and result["oneblob"]["all_rows_equal"], line
