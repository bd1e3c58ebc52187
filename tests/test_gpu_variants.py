"""The retained A/B code paths (environment switches read once per process) stay correct: a slice of the GPU suite
re-run in a subprocess with the non-default kernels selected -- the one-thread-per-element fold kernels with and without
the endomorphisms (RIPP_B200_FOLD=endo / plain), three-warp teams (RIPP_B200_FOLD=w3), one thread per element for the
scalings, the six-lane shape everywhere (RIPP_B200_L18_WARPS=0), and the fused folds of a round without / always with
one team per endomorphism part (RIPP_B200_XP_MAX=0 / 100000)."""
import os
import subprocess
import sys

import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.parametrize("env", [
    {"RIPP_B200_FOLD": "endo"},
    {"RIPP_B200_FOLD": "plain"},
    {"RIPP_B200_FOLD": "w3"},
    {"RIPP_B200_SCALE_PARTS_MAX": "0"},
    {"RIPP_B200_SCALE_PARTS_MAX": "0", "RIPP_B200_SCALE_XT_MAX": "100000"},
    {"RIPP_B200_L18_WARPS": "0"},
    {"RIPP_B200_XP_MAX": "0"},
    {"RIPP_B200_XP_MAX": "100000"},
], ids=lambda e: ",".join("%s=%s" % kv for kv in e.items()))
def test_variant_paths(env):
    sel = ["tests/test_gpu_msm.py::test_folds", "tests/test_gpu_msm.py::test_scalings_match_oracle",
           "tests/test_gpu_msm.py::test_msm_g1_matches_oracle", "tests/test_gpu_pairing.py::test_pairing_ip_matches_oracle",
           "tests/test_gpu_protocols.py::test_aggregate_proofs_bytes_match_oracle"]
    if any(k.startswith("RIPP_B200_L18") for k in env):  # the pairing engine's shape thresholds: the sizes that cross them
        sel.append("tests/test_gpu_fullsize.py::test_pairing_product_engine_shapes_match_cpu_oracle")
    r = subprocess.run([sys.executable, "-m", "pytest", "-q", "-x", "-m", "gpu"] + sel, cwd=ROOT, env=dict(os.environ, **env),
                       capture_output=True, text=True, timeout=1500)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-2000:]
