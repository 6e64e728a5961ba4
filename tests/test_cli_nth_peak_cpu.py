"""CPU checks of the CLI's --nth-peak option: its argument and combination errors need no GPU, the existing
--sections / --loudness / --overs errors are checked first and keep their text, and without a GPU the option
fails loudly (no CPU fallback)."""
import os
import subprocess

import pytest

import oracle_lib as O
from phaserotate.lv2_b200 import build

RANGE = "Error: --nth-peak takes a rank of 1 .. 256.\n"
COMBO = "Error: --nth-peak cannot be combined with -a, --sections, --gpus or --loudness.\n"
SECTIONS_COMBO = "Error: --sections cannot be combined with -a, --true-peak or --gpus.\n"
LOUDNESS_COMBO = "Error: --loudness cannot be combined with -a, --sections or --gpus.\n"
OVERS_COMBO = "Error: --overs cannot be combined with --sections or --gpus.\n"


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


def test_nth_peak_argument_errors(wav):
    for arg in ["0", "257", "-1", "", "1.5", "11x", "x", "1e2", "99999999999999999999"]:
        r = _cli("--nth-peak", arg, wav)
        assert r.returncode == 1, arg
        assert r.stderr == RANGE, (arg, r.stderr)
        assert r.stdout == ""


def test_nth_peak_combination_errors(wav, tmp_path):
    out = str(tmp_path / "y.wav")
    cases = [(["--nth-peak", "11", "-a", "10", wav, out], COMBO),
             (["-a", "10", "--nth-peak", "1", wav, out], COMBO),
             (["--nth-peak", "11", "--gpus", "2", wav], COMBO),
             (["--gpus", "0", "--nth-peak", "2", wav], COMBO),
             (["--nth-peak", "11", "--loudness", wav], COMBO),
             (["--loudness", "--nth-peak", "256", wav, out], COMBO),
             (["--nth-peak", "3", "--sections", "10", wav], COMBO),
             # the --sections, --loudness and --overs errors come first and keep their text
             (["--nth-peak", "11", "--sections", "10", "-a", "10", wav, out], SECTIONS_COMBO),
             (["--nth-peak", "11", "--sections", "10", "--true-peak", wav], SECTIONS_COMBO),
             (["--nth-peak", "11", "--sections", "10", "--gpus", "2", wav], SECTIONS_COMBO),
             (["--nth-peak", "11", "--loudness", "--sections", "10", wav], LOUDNESS_COMBO),
             (["--nth-peak", "11", "--loudness", "--gpus", "2", wav], LOUDNESS_COMBO),
             (["--nth-peak", "11", "--loudness", "-a", "10", wav, out], LOUDNESS_COMBO),
             (["--nth-peak", "11", "--overs", "-1", "--sections", "10", wav], OVERS_COMBO),
             (["--nth-peak", "11", "--overs", "-1", "--gpus", "2", wav], OVERS_COMBO)]
    for argv, msg in cases:
        r = _cli(*argv)
        assert r.returncode == 1, argv
        assert r.stderr == msg, (argv, r.stderr)
        assert r.stdout == ""


def test_messages_without_nth_peak_unchanged(wav, tmp_path):
    # the combinations the new option joins keep their own messages when it is absent
    out = str(tmp_path / "y.wav")
    cases = [(["--sections", "10", "-a", "10", wav, out], SECTIONS_COMBO),
             (["--loudness", "--gpus", "2", wav], LOUDNESS_COMBO),
             (["--loudness", "-a", "10", wav, out], LOUDNESS_COMBO),
             (["--overs", "-1", "--gpus", "2", wav], OVERS_COMBO),
             (["--overs", "-1", "--sections", "10", wav], OVERS_COMBO)]
    for argv, msg in cases:
        r = _cli(*argv)
        assert r.returncode == 1 and r.stderr == msg and r.stdout == "", (argv, r.stderr)


@pytest.mark.skipif(_has_gpu(), reason="only meaningful on a machine without a GPU")
@pytest.mark.parametrize("extra", [[], ["--true-peak"], ["--overs", "-1"], ["-l", "--subsample", "10", "-s", "1"]])
def test_nth_peak_fails_loudly_without_gpu(wav, extra):
    r = _cli("--nth-peak", "11", *extra, wav)
    assert r.returncode == 1 and "CUDA backend" in r.stderr and r.stdout == ""
