"""The NRC network against the reference's own code on the GPU: tiny-cuda-nn's NetworkWithInputEncoding + Trainer built from
neural_radiance_caching/network_interface.cu's config (oracle/ref_tcnn/tcnn_nrc.cu -> oracle/_ref/libtcnn_nrc.so, compiled from
the reference's vendored tiny-cuda-nn).  Its outputs on the check's seeded inputs are stored in tests/golden/golden_tcnn_nrc.npz
(written by `python tests/tcnn_nrc_check.py --write-golden`; a fixed sample of the rows and parameters, the initial parameters as
digests), so the test needs no reference build.  tests/tcnn_nrc_check.py does the work in a child process and prints one JSON
line; the relative L2 bars against tiny-cuda-nn hold over the stored sample:

  * gfx_nrc_create's initial parameters == tcnn::Trainer{seed 1337}'s, every fp32 master weight bit for bit;
  * inferred radiance within 1e-3 relative L2 of tiny-cuda-nn's (BASELINE.json north_star), before and after four training steps;
  * the oracle in its half-accumulate mode (tiny-cuda-nn's arithmetic model, oracle/nrc.cpp header) within 1e-4 of tiny-cuda-nn on
    the forward pass - which pins the restatement - and within 1e-3 on the hash-grid gradient;
  * one training step's gradients: this repo accumulates in fp32 where tiny-cuda-nn accumulates in half (wmma fragments and
    CUTLASS half accumulators of the split-k weight-gradient GEMMs), so it sits at the reference's own rounding noise from the
    exact gradient: <= 2.5e-3 on every weight matrix, <= 2e-2 on the hash grid (whose entries are sums of a few tiny terms),
    and - the statement that matters - never further from tiny-cuda-nn than the half-accumulating oracle is from the
    fp32-accumulating one plus 1e-3;
  * the loss of each of four steps within 1e-4 relative of tiny-cuda-nn's."""
import json
import os
import subprocess
import sys

import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden", "golden_tcnn_nrc.npz")


def test_nrc_network_matches_tiny_cuda_nn():
    proc = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "tcnn_nrc_check.py"), "--golden", GOLDEN], capture_output=True,
                          text=True, timeout=400)
    line = proc.stdout.strip().splitlines()[-1] if proc.stdout.strip() else ""
    assert proc.returncode == 0, f"rc={proc.returncode} {line[:400]} {proc.stderr[-600:]}"
    r = json.loads(line)
    init = r["init"]
    assert init["master_equal"] and init["training_half_equal"] and init["inference_all_zero"], init
    fwd = r["forward"]
    assert fwd["ours_vs_tcnn"] <= 1e-3, fwd
    assert fwd["oracle_halfacc_vs_tcnn"] <= 1e-4, fwd
    assert fwd["ours_vs_oracle_fp32acc"] <= 1e-4, fwd
    g = r["gradients"]
    for name in ("W0", "W1", "W2"):
        assert g[name]["ours_vs_tcnn"] <= 2.5e-3, (name, g[name])
        assert g[name]["ours_vs_oracle_fp32acc"] <= 1e-4, (name, g[name])
    assert g["grid"]["oracle_halfacc_vs_tcnn"] <= 1e-3, g["grid"]
    assert g["grid"]["ours_vs_tcnn"] <= 2e-2, g["grid"]
    assert g["grid"]["ours_vs_oracle_fp32acc"] <= 1e-3, g["grid"]
    losses = r["weights"]["losses"]
    for a, b in zip(losses["ours"], losses["tcnn"]):
        assert abs(a - b) <= 1e-4 * abs(b), losses
    w = r["weights"]
    assert w["inference_after_training_ours_vs_tcnn"] <= 1e-3, w["inference_after_training_ours_vs_tcnn"]
    for name in ("W0", "W1", "W2", "grid"):
        assert w[name]["inference_ours_vs_tcnn"] <= 1e-2, (name, w[name])
