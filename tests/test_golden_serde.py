"""Decoder rules against arkworks itself, when somebody has produced tests/golden/ark_golden.json (tools/ark_golden; see
tests/test_golden.py).  tests/golden/serde_cases.txt lists the encodings whose verdicts the dumper records: each flag
rule, x = p, an x off the curve, a point off the subgroup and valid points (oracle/serde_cases.py named_cases)."""
import json
import os

import pytest

from oracle import serde as S
from oracle import serde_cases as SC
from oracle import synth as OS
from oracle import bls12_381 as E

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
CASES = os.path.join(GOLDEN_DIR, "serde_cases.txt")


def _case_lines():
    lines = []
    for group in (1, 2):
        for compressed in (True, False):
            for name, b in SC.named_cases(group, compressed, seed=0):
                lines.append("serde_case_%d_%s_%s %s" % (group, "c" if compressed else "u", name, b.hex()))
    return "\n".join(lines) + "\n"


def test_case_file_is_current():
    """The committed input list of the dumper is what oracle/serde_cases.py generates."""
    assert open(CASES).read() == _case_lines(), "regenerate tests/golden/serde_cases.txt from oracle/serde_cases.py"


@pytest.fixture(scope="module")
def golden():
    path = os.path.join(GOLDEN_DIR, "ark_golden.json")
    if not os.path.exists(path):
        pytest.skip("tests/golden/ark_golden.json absent: run tools/ark_golden with a Rust toolchain (parity unpinned)")
    return {k: bytes.fromhex(v) for k, v in json.load(open(path)).items()}


def test_compressed_encodings(golden):
    assert S.ser_g1_compressed(OS.g1_points("gipa-a", 1)[0]) == golden["g1c_gipa-a_0"]
    assert S.ser_g2_compressed(OS.g2_points("gipa-b", 1)[0]) == golden["g2c_gipa-b_0"]
    assert S.ser_g1_compressed(E.G1_GEN) == golden["g1c_generator"]
    assert S.ser_g2_compressed(E.G2_GEN) == golden["g2c_generator"]


def test_decoder_verdicts(golden):
    for line in open(CASES).read().split("\n"):
        if not line:
            continue
        key, hx = line.split()
        group, mode = int(key.split("_")[2]), key.split("_")[3]
        compressed = mode == "c"
        pt, st = (S.de_g1 if group == 1 else S.de_g2)(bytes.fromhex(hx), compressed)
        got = golden[key.replace("serde_case_", "serde_verdict_")]
        if st == S.OK:
            assert got == b"ok" + (S.ser_g1(pt) if group == 1 else S.ser_g2(pt)), key
        elif st == S.FLAGS and "infinity_nonzero" not in key:
            assert got == b"flags", key
        else:  # an infinity flag with coordinate bits set is InvalidData in read_g*_*, not UnexpectedFlags
            assert got == b"invalid", key
