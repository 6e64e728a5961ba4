"""tests/stream_ref.py against the C restatement on short streams, and its hull peak table against brute force.

stream_ref is the float64 reference the long-stream GPU tests (test_gpu_segment_runs.py) compare the library
with; these checks pin it first, on lengths the oracle handles in milliseconds."""
import numpy as np
import pytest

import oracle_lib as O
import stream_ref as R


def oracle_lut(S):
    s = np.zeros(180 * S, np.float32)
    c = np.zeros(180 * S, np.float32)
    O.oracle().pro_sincos_lut(S, s, c)
    return s, c


def relmax(a, b):
    return float(np.max(np.abs(a - b) / np.maximum(np.abs(b), 1e-30)))


SHORT = {
    "programme_2ch_L2048": (lambda: O.programme(48000, 0.7, 2), 2048),
    "harmonic_3ch_L8192": (lambda: O.harmonic(48000, 0.9, 3)[:40001], 8192),
    "pink_mono_L1024": (lambda: O.pink_noise(23457, 4)[:, None], 1024),
    "harmonic_2ch_L32768": (lambda: O.harmonic(192000, 0.4, 2), 32768),
}


@pytest.mark.parametrize("name", sorted(SHORT))
def test_peak_table_matches_oracle(oracle_built, name):
    gen, L = SHORT[name]
    x = gen()
    lut = oracle_lut(2)
    want = O.oracle_analyze(x, L)
    got = R.peak_table(x, L, lut=lut)
    assert relmax(got, want) <= 1e-6
    assert np.array_equal(got[:, 0], want[:, 0].astype(np.float64))   # raw input peak: no arithmetic


@pytest.mark.parametrize("name", sorted(SHORT))
@pytest.mark.parametrize("os_", [2, 4])
def test_true_peak_table_matches_oracle(oracle_built, name, os_):
    gen, L = SHORT[name]
    x = gen()
    want = O.oracle_analyze_tp(x, L, oversample=os_)
    got = R.peak_table(x, L, os_=os_, lut=oracle_lut(2))
    assert relmax(got, want) <= 1e-6


@pytest.mark.parametrize("name", sorted(SHORT))
@pytest.mark.parametrize("flush", [0, 1, 2])
def test_render_matches_oracle(oracle_built, name, flush):
    gen, L = SHORT[name]
    x = gen()
    C = x.shape[1]
    ang = [541, -91, 90][:C] if C > 1 else [719]          # indices outside [0, MS) wrap like the CLI
    want = O.oracle_apply(x, L, ang, flush)
    got = R.render_ref(x, L, ang, flush, lut=oracle_lut(2))
    assert got.shape == want.shape
    assert np.max(np.abs(got - want)) <= 1e-6 * float(np.abs(want).max())


def test_pair_window_equals_whole_stream():
    x = O.programme(48000, 0.5, 1)[:, 0].astype(np.float64)
    L = 4096
    xd, H = R.analytic_pair(x, L, first_block=False)[0]
    for t0, t1 in [(0, 100), (3000, 9000), (len(x) - 50, len(xd))]:
        wd, wh = R.pair_window(x, L, t0, t1)
        assert np.allclose(wd, xd[t0:t1], rtol=0, atol=0)
        assert np.max(np.abs(wh - H[t0:t1])) <= 1e-12


MATERIAL = {
    "programme": lambda n: O.programme(48000, n / 48000, 2)[:n],
    "sine": lambda n: (0.8 * np.sin(2 * np.pi * 997.0 / 48000 * np.arange(n))).astype(np.float32)[:, None] * np.ones((1, 2), np.float32),
    "two_sine": lambda n: O.two_sine(48000, n / 48000, 2)[:n],
    "zero_channel": lambda n: np.stack([O.pink_noise(n, 3), np.zeros(n, np.float32)], 1),
    "dc": lambda n: np.full((n, 2), 0.25, np.float32),
    "one_frame": lambda n: np.array([[0.5, -0.25]], np.float32),
}


@pytest.mark.parametrize("mat", sorted(MATERIAL))
@pytest.mark.parametrize("os_", [0, 4])
def test_hull_table_equals_brute_force(mat, os_):
    """The hull only chooses which points are evaluated: the table is the brute-force maximum bit for bit."""
    x = MATERIAL[mat](30011)
    L = 2048
    pairs = R.analytic_pair(x, L)
    for S in (2, 10):
        lut = R.closed_form_lut(S)
        hull = R.peak_table(x, L, S, os_, lut, pairs)
        brute = R.peak_table(x, L, S, os_, lut, pairs, hull=False)
        assert np.array_equal(hull, brute), S
    if mat == "zero_channel":
        assert np.all(hull[1] == 0) and np.all(hull[0, 1:] > 0)


def test_hull_candidates_are_few_on_programme():
    x = O.programme(48000, 2.0, 1)[:, 0]
    xd, H = R.analytic_pair(x, 8192)[0]
    cand = R.hull_candidates(xd, H)
    assert 3 <= len(cand) < 1e-3 * len(xd)


def test_overs_counts_match_restatement():
    """The radius-filtered count of stream_ref equals a direct count over every sample."""
    x = O.programme(48000, 0.6, 2)
    L = 2048
    pairs = R.analytic_pair(x, L)
    lut = R.closed_form_lut(2)
    pk = R.peak_table(x, L, lut=lut, pairs=pairs)
    T = 0.5 * float(pk.min() + pk.max())
    lo, hi = R.overs_counts(x, L, T, lut=lut, pairs=pairs)
    s, c = (np.asarray(v, np.float64) for v in lut)
    for ch, (xd, H) in enumerate(pairs):
        for a in (1, 45, 180, 359):
            v = np.abs(c[a] * xd[L // 2:] + s[a] * H[L // 2:])
            assert lo[ch, a] == np.count_nonzero(v > T * (1 + 2e-6)) and hi[ch, a] == np.count_nonzero(v > T * (1 - 2e-6))
    assert lo.max() > 0 and lo.min() < lo.max()


def test_geometry():
    assert [R.seg_samples(L) for L in (1024, 4096, 8192, 16384, 32768)] == [31744, 28672, 24576, 16384, 16384]
    assert R.chunk_frames(2) == 4 << 20 and R.chunk_frames(8) == 1 << 20 and R.chunk_frames(3) % 4 == 0
    assert R.n_segments(0, 8192) == 1 and R.n_segments(8192, 8192) == 1 and R.n_segments(3 * 8192, 8192) == 2
    runs = R.cta_runs(450, 3, 148)
    assert len(runs) == 50 + 45 + 45 and sum(runs) == 3 * 450 and min(runs) == 9   # 50 CTAs of 9 segments, 2 x 45 of 10
    assert R.cta_runs(5, 2, 148) == [1] * 10
    assert R.segs_first(2, 148) == 592 and R.segs_first(8, 148) == 148
