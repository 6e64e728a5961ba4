"""CPU checks of the BS.1770-4 restatement (tests/loudness_ref.py) that the GPU loudness tests compare
against: the derived K-weighting reproduces the standard's 48 kHz table, and the integrated loudness of
EBU Tech 3341 cases 1-5 is -23 / -33 LUFS within the +-0.1 LU the test document allows."""
import numpy as np
import pytest

import loudness_ref as R


def test_kweight_coefficients_match_bs1770_table_at_48k():
    for (b, a), (bt, at) in zip(R.kweight_coefs(48000.0), R.TABLE_48K):
        assert np.max(np.abs(np.subtract(b, bt))) <= 1e-12
        assert np.max(np.abs(np.subtract(a, at))) <= 1e-12


def test_kweight_gain_is_standard():
    # +4 dB high shelf, high pass at 38 Hz: the 1 kHz gain that the -0.691 constant offsets (BS.1770-4 Annex 1)
    from scipy.signal import freqz
    g = 1.0
    for b, a in R.kweight_coefs(48000.0):
        g *= abs(freqz(b, a, [1000.0], fs=48000.0)[1][0])
    assert abs(20 * np.log10(g) - 0.691) < 0.01


@pytest.mark.parametrize("case", sorted(R.TECH3341))
def test_tech3341_cases(case):
    x = R.sine_segments(48000, R.TECH3341[case])
    got = R.integrated(x, 48000)
    assert abs(got - R.TECH3341_EXPECTED[case]) <= 0.1, got


def test_short_and_silent_streams_are_minus_inf():
    assert R.integrated(np.ones((19199, 2), np.float32) * 0.1, 48000) == -np.inf   # one sample short of 400 ms
    assert R.integrated(np.zeros((48000, 2), np.float32), 48000) == -np.inf
    assert np.isfinite(R.integrated(np.ones((19200, 2), np.float32) * 0.1, 48000))  # exactly one block
