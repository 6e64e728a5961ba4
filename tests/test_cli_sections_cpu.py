"""CPU checks of the CLI's --sections option: argument errors need no GPU, and without one the option
fails loudly like every other analysis (no CPU fallback)."""
import os
import subprocess

import pytest

import oracle_lib as O
from phaserotate.lv2_b200 import build


def _has_gpu():
    try:
        import torch
        return torch.cuda.is_available()
    except Exception:
        return False


def _cli(*argv):
    build.build_host()
    return subprocess.run([os.path.join(build.BIN_DIR, "phase-rotate")] + list(argv), capture_output=True, text=True)


@pytest.fixture()
def wav(tmp_path):
    p = str(tmp_path / "x.wav")
    O.write_wav_f32(p, O.two_sine(48000, 0.1, 2), 48000)
    return p


def test_sections_argument_errors(wav, tmp_path):
    out = str(tmp_path / "y.wav")
    combo = "Error: --sections cannot be combined with -a, --true-peak or --gpus.\n"
    value = "Error: --sections takes a section length in seconds > 0.\n"
    cases = [(["--sections", "10", "-a", "10", wav, out], combo),
             (["--sections", "10", "--true-peak", wav], combo),
             (["--true-peak=2", "--sections", "10", wav], combo),
             (["--sections", "10", "--gpus", "2", wav], combo),
             (["--gpus", "0", "--sections", "10", wav], combo),
             (["--sections", "0", wav], value),
             (["--sections", "-5", wav], value),
             (["--sections", "abc", wav], value),
             (["--sections", "nan", wav], value),
             (["--sections", "inf", wav], value)]
    for argv, msg in cases:
        r = _cli(*argv)
        assert r.returncode == 1, argv
        assert r.stderr == msg, (argv, r.stderr)
        assert r.stdout == ""


@pytest.mark.skipif(_has_gpu(), reason="only meaningful on a machine without a GPU")
def test_sections_fail_loudly_without_gpu(wav):
    r = _cli("--sections", "0.5", wav)
    assert r.returncode == 1 and "CUDA backend" in r.stderr and r.stdout == ""
