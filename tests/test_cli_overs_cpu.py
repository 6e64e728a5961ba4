"""CPU checks of the CLI's --overs option: its argument errors need no GPU, the --sections and --loudness errors are
checked first and keep their text, and without a GPU the option fails loudly (no CPU fallback)."""
import os
import subprocess

import pytest

import oracle_lib as O
from phaserotate.lv2_b200 import build

RANGE = "Error: --overs takes a ceiling in dBFS from -60 to 20.\n"
COMBO = "Error: --overs cannot be combined with --sections or --gpus.\n"
SECTIONS_COMBO = "Error: --sections cannot be combined with -a, --true-peak or --gpus.\n"
LOUDNESS_COMBO = "Error: --loudness cannot be combined with -a, --sections or --gpus.\n"


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


def test_overs_argument_errors(wav, tmp_path):
    out = str(tmp_path / "y.wav")
    cases = [(["--overs", "-60.01", wav], RANGE),
             (["--overs", "20.5", wav], RANGE),
             (["--overs", "nan", wav], RANGE),
             (["--overs", "inf", wav], RANGE),
             (["--overs", "-1dB", wav], RANGE),
             (["--overs", "", wav], RANGE),
             (["--overs", "-1", "--sections", "10", wav], COMBO),
             (["--sections", "10", "--overs", "-1", wav], COMBO),
             (["--overs", "-1", "--gpus", "2", wav], COMBO),
             (["--gpus", "0", "--overs", "0", wav], COMBO),
             # the --sections and --loudness errors come first and keep their text
             (["--overs", "-1", "--sections", "10", "-a", "10", wav, out], SECTIONS_COMBO),
             (["--overs", "-1", "--sections", "10", "--true-peak", wav], SECTIONS_COMBO),
             (["--overs", "-1", "--gpus", "2", "--sections", "10", wav], SECTIONS_COMBO),
             (["--overs", "-1", "--loudness", "--sections", "10", wav], LOUDNESS_COMBO),
             (["--overs", "-1", "--loudness", "--gpus", "2", wav], LOUDNESS_COMBO),
             (["--overs", "-1", "--loudness", "-a", "10", wav, out], LOUDNESS_COMBO)]
    for argv, msg in cases:
        r = _cli(*argv)
        assert r.returncode == 1, argv
        assert r.stderr == msg, (argv, r.stderr)
        assert r.stdout == ""


@pytest.mark.skipif(_has_gpu(), reason="only meaningful on a machine without a GPU")
@pytest.mark.parametrize("extra", [[], ["--true-peak"], ["--loudness"], ["-l", "--subsample", "10"]])
def test_overs_fails_loudly_without_gpu(wav, extra):
    r = _cli("--overs", "-1", *extra, wav)
    assert r.returncode == 1 and "CUDA backend" in r.stderr and r.stdout == ""


@pytest.mark.skipif(_has_gpu(), reason="only meaningful on a machine without a GPU")
def test_overs_with_angle_fails_loudly_without_gpu(wav, tmp_path):
    r = _cli("--overs", "-3", "-a", "30", wav, str(tmp_path / "y.wav"))
    assert r.returncode == 1 and "CUDA backend" in r.stderr and r.stdout == ""
