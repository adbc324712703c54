"""CPU tests of jf_aligner --details: the restatement of the reference's print_details (tests/details_lib.py) over the
oracle port's taps against the reference's own golden files, and which option combinations the tool accepts."""
import os
import subprocess

import pytest

from details_lib import port_details

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
JFA = os.path.join(ROOT, "pacbio_b200", "bin", "jf_aligner")
GOLD = os.path.join(ROOT, "tests", "golden", "aligner_output")


@pytest.fixture(scope="module")
def jfa():
    if not os.path.exists(JFA):
        subprocess.check_call(["make", "-C", os.path.join(ROOT, "pacbio_b200", "csrc"), "all"], stdout=subprocess.DEVNULL)
    return JFA


def _has_gpu():
    try:
        import torch
        return torch.cuda.is_available()
    except Exception:
        return False


@pytest.mark.parametrize("forward", [False, True])
def test_port_details_match_reference_goldens(port, tmp_path, forward):
    """tests/aligner_output (k = 17, --stretch-cap 200): the lines of details_*_expected, in any order (the reference's
    line order follows its map of super-read name pointers)."""
    sr = os.path.join(GOLD, "test_super_reads.fa")
    h = port.index_create(sr, 13, 17)
    a = port.aligner_create(h, stretch_cap=200.0, forward=forward)
    try:
        got = port_details(port, a, sr, os.path.join(GOLD, "test_pacbio.fa"))
    finally:
        port.aligner_destroy(a)
        port.index_destroy(h)
    golden = os.path.join(GOLD, "details_forward_expected" if forward else "details_normal_expected")
    assert sorted(got) == sorted(open(golden).read().splitlines())


def _jf_aligner(jfa, tmp_path, extra):
    return subprocess.run([jfa, "-s", "10k", "-m", "17", "-r", os.path.join(GOLD, "test_super_reads.fa"),
                           "-p", os.path.join(GOLD, "test_pacbio.fa"), "--details", str(tmp_path / "d"),
                           "--coords", str(tmp_path / "c")] + extra, stdout=subprocess.PIPE, stderr=subprocess.PIPE)


def test_jf_aligner_rejects_details_with_fine_pass(jfa, tmp_path):
    """What the reference prints with --details after a fine pass is not pinned by anything here: refused, exit 1."""
    r = _jf_aligner(jfa, tmp_path, ["-F", "12"])
    assert r.returncode == 1
    assert b"[--details] is not available together with -F" in r.stderr


def test_jf_aligner_accepts_details_with_max_match(jfa, tmp_path):
    r = _jf_aligner(jfa, tmp_path, ["--max-match"])
    assert b"not available together" not in r.stderr
    if _has_gpu():
        assert r.returncode == 0, r.stderr.decode()[-2000:]
    else:
        assert r.returncode == 1 and b"no CUDA device" in r.stderr
