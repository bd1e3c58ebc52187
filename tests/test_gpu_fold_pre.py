"""The fold over precomputed bases (k_fold_pre on a side stream during the round's products, then k_fold4_xp<true>)
gives the proof bytes of the plain fused folds: the GIPA kinds, TIPA, the aggregation and the fold entry points re-run in
a subprocess with it off (RIPP_B200_FOLD_PRE_MAX=0), at its default range, and for every lane-team round (100000),
plus the 2^12 aggregation against the CPU oracle."""
import os
import subprocess
import sys

import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.parametrize("pre_max", ["0", None, "100000"], ids=lambda v: "default" if v is None else v)
def test_fold_pre_switch(pre_max):
    sel = ["tests/test_gpu_protocols.py::test_gipa_proof_bytes_match_oracle",
           "tests/test_gpu_protocols.py::test_tipa_proof_bytes_match_oracle",
           "tests/test_gpu_protocols.py::test_tipa_ssm_proof_bytes_match_oracle",
           "tests/test_gpu_protocols.py::test_aggregate_proofs_bytes_match_oracle",
           "tests/test_gpu_msm.py::test_folds",
           "tests/test_gpu_fullsize.py::test_tipp_2p12_proof_bytes_match_cpu_oracle_and_oracle_verifier_accepts"]
    env = dict(os.environ)
    env.pop("RIPP_B200_FOLD_PRE_MAX", None)
    if pre_max is not None:
        env["RIPP_B200_FOLD_PRE_MAX"] = pre_max
    r = subprocess.run([sys.executable, "-m", "pytest", "-q", "-x", "-m", "gpu"] + sel, cwd=ROOT, env=env,
                       capture_output=True, text=True, timeout=1500)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-2000:]
