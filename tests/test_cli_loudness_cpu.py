"""CPU checks of the CLI's --loudness option: its argument errors need no GPU, the --sections errors are
checked first and keep their text, and without a GPU the option fails loudly (no CPU fallback)."""
import os
import subprocess

import pytest

import oracle_lib as O
from phaserotate.lv2_b200 import build

COMBO = "Error: --loudness cannot be combined with -a, --sections or --gpus.\n"
SECTIONS_COMBO = "Error: --sections cannot be combined with -a, --true-peak or --gpus.\n"


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


def test_loudness_argument_errors(wav, tmp_path):
    out = str(tmp_path / "y.wav")
    cases = [(["--loudness", "-a", "10", wav, out], COMBO),
             (["-a", "10", "--loudness", wav, out], COMBO),
             (["--loudness", "--sections", "10", wav], COMBO),
             (["--sections", "10", "--loudness", wav], COMBO),
             (["--loudness", "--gpus", "2", wav], COMBO),
             (["--gpus", "0", "--loudness", wav], COMBO),
             # the --sections errors come first and keep their text
             (["--loudness", "--sections", "10", "-a", "10", wav, out], SECTIONS_COMBO),
             (["--sections", "10", "--true-peak", "--loudness", wav], SECTIONS_COMBO),
             (["--loudness", "--gpus", "2", "--sections", "10", wav], SECTIONS_COMBO),
             (["--loudness", "--sections", "0", wav], "Error: --sections takes a section length in seconds > 0.\n")]
    for argv, msg in cases:
        r = _cli(*argv)
        assert r.returncode == 1, argv
        assert r.stderr == msg, (argv, r.stderr)
        assert r.stdout == ""


@pytest.mark.skipif(_has_gpu(), reason="only meaningful on a machine without a GPU")
def test_loudness_fails_loudly_without_gpu(wav):
    r = _cli("--loudness", wav)
    assert r.returncode == 1 and "CUDA backend" in r.stderr and r.stdout == ""
