"""Rank table (phaserot_nth_peaks*, phase-rotate --nth-peak) on the GPU.

References: an independent float64 rank table (closed-form Hilbert taps and the interpolator of
test_truepeak_independent, through stream_ref), and three identities that hold bit for bit: rank 1 is the sweep's
peak table, min (overs count, N) is the number of entries above the ceiling, and the pruned table is the table of
a PHASEROT_FLAG_NO_PRUNE handle, which lists every examined sample."""
import functools
import os
import re
import subprocess

import numpy as np
import pytest

import oracle_lib as O
import stream_ref as R
from phaserotate.lv2_b200 import capi

pytestmark = pytest.mark.gpu

RANKS = (1, 2, 11, 256)

CASES = {
    "programme_2ch_L8192": (lambda: O.programme(48000, 1.0, 2), 8192),
    "pink_mono_L4096": (lambda: O.pink_noise(48000, seed=7)[:, None], 4096),
    "odd_3ch_L1024": (lambda: O.programme(48000, 0.6, 3, seed=11)[:24007], 1024),
    "one_frame_L2048": (lambda: np.array([[0.7, -0.3]], np.float32), 2048),
    "programme_8ch_L8192": (lambda: O.programme(48000, 0.4, 8, seed=5), 8192),
}


def _x(case):
    return np.ascontiguousarray(CASES[case][0](), np.float32)


def _top(v, N):
    out = np.zeros(N)
    k = min(N, len(v))
    if k:
        out[:k] = np.sort(np.partition(v, len(v) - k)[len(v) - k:])[::-1]
    return out


@functools.lru_cache(maxsize=None)
def rank_ref(case, os_, N=256, S=2):
    """out[c][a][k] in float64: the (k+1)-th largest detector value at grid index a (index 0: the raw input over
    the frames of the raw-peak rule; a >= 1: the samples t >= L/2 of the pass, first-block rule applied)."""
    x = _x(case)
    L = CASES[case][1]
    F, C = x.shape
    MS = 180 * S
    s, c = (np.asarray(v, np.float64) for v in R.closed_form_lut(S))
    B = -(-F // L)
    out = np.zeros((C, MS, N))
    for ch, (xd, H) in enumerate(R.analytic_pair(x, L)):
        rx = R.detector_rows(xd, os_)[:, L // 2:]
        ry = R.detector_rows(H, os_)[:, L // 2:]
        rad = np.hypot(rx, ry).max(0)
        # the N-th values over the samples of largest radius bound every angle's N-th value from below; a sample
        # whose radius is below the smallest of them cannot rank at any angle
        top = np.argsort(rad)[::-1][:4096]
        lb = min(_top(np.abs(c[a] * rx[:, top] + s[a] * ry[:, top]).max(0), N)[-1] for a in range(1, MS))
        keep = np.nonzero(rad >= lb * (1 - 1e-9))[0]
        kx, ky = rx[:, keep], ry[:, keep]
        for a in range(1, MS):
            out[ch, a] = _top(np.abs(c[a] * kx + s[a] * ky).max(0), N)
        raw = np.zeros((B + 1) * L)
        raw[:F] = x[:, ch]
        f_end = min(F + (11 if os_ > 1 else 0), (B + 1) * L - L // 2)
        out[ch, 0] = _top(np.abs(R.detector_rows(raw, os_)).max(0)[:f_end], N)
    return out


def _check_table(t, N):
    assert t.shape[2] == N
    assert (np.diff(t, axis=2) <= 0).all()                              # every row non-increasing
    assert (t >= 0).all()


def _ceilings(t, N):
    """ceilings equal to table entries (ties) and between them, all > 0"""
    vals = [t[0, 5, N - 1], t[-1, 100, 0], t[0, 0, min(N, 3) - 1], t[-1, -1, N // 2], 0.5 * (t[0, 7, 0] + t[0, 7, N - 1]), 0.3 * t.max()]
    return sorted({float(np.float32(v)) for v in vals if v > 0})


def _identity2(h, x, t, N):
    for T in _ceilings(t, N):
        cnt, _ = h.overs(x, T)
        assert np.array_equal(np.minimum(cnt, N), (t > np.float32(T)).sum(2)), T


@pytest.mark.parametrize("os_", [0, 2, 4])
@pytest.mark.parametrize("case", sorted(CASES))
def test_independent_float64(case, os_):
    x = _x(case)
    ref = rank_ref(case, os_)
    with capi.Phaserot(n_channels=x.shape[1], blksiz=CASES[case][1], oversample=os_) as h:
        for N in RANKS:
            t = h.nth_peaks(x, N)
            _check_table(t, N)
            np.testing.assert_allclose(t, ref[:, :, :N], rtol=1e-5, atol=1e-5 * max(float(ref.max()), 1e-30), err_msg=f"rank {N}")


@pytest.mark.parametrize("os_", [0, 2, 4])
@pytest.mark.parametrize("case", sorted(CASES))
def test_identities(case, os_):
    x = _x(case)
    L = CASES[case][1]
    nc = x.shape[1]
    with capi.Phaserot(n_channels=nc, blksiz=L, oversample=os_) as h, \
            capi.Phaserot(n_channels=nc, blksiz=L, oversample=os_, flags=capi.FLAG_NO_PRUNE) as hb:
        h.sweep(x)
        pk = h.peaks()
        for N in RANKS:
            t = h.nth_peaks(x, N)
            assert np.array_equal(t[:, :, 0], pk), N                          # 1: rank 1 is the peak table
            assert np.array_equal(t, hb.nth_peaks(x, N)), N                   # 3: pruning changes nothing
            _identity2(h, x, t, N)                                            # 2: the overs counts


@pytest.mark.parametrize("os_", [0, 4])
def test_long_stream_fine_grid(os_):
    # 10 minutes of stereo at 0.1 degree: several contiguous FFT launches, rows merged across them
    x = O.programme(48000, 600.0, 2, seed=21)
    F = x.shape[0]
    assert R.n_segments(F, 8192) > R.segs_first(2, 148)                   # premise: more than one contiguous launch
    with capi.Phaserot(n_channels=2, blksiz=8192, subsample=10, oversample=os_) as h, \
            capi.Phaserot(n_channels=2, blksiz=8192, subsample=10, oversample=os_, flags=capi.FLAG_NO_PRUNE) as hb:
        h.sweep(x)
        pk = h.peaks()
        for N in (1, 11, 256):
            t = h.nth_peaks(x, N)
            _check_table(t, N)
            assert np.array_equal(t[:, :, 0], pk), N
            assert np.array_equal(t, hb.nth_peaks(x, N)), N
        _identity2(h, x, t, 256)


def _sine(sr, seconds, channels, f=997.0, amp=0.8):
    t = np.arange(int(sr * seconds))
    return np.stack([amp * np.sin(2 * np.pi * f / sr * t + 0.4 * c) for c in range(channels)], 1).astype(np.float32)


@pytest.mark.parametrize("os_", [0, 4])
@pytest.mark.parametrize("mat", ["sine", "two_sine"])
def test_dense_material_exactly_once(mat, os_):
    # every sample of a pure tone stays near the N-th value: lists overflow and are re-run in pieces; a record
    # merged twice or dropped would break identity 1 or 3
    x = _sine(48000, 240.0, 2) if mat == "sine" else O.two_sine(48000, 240.0, 2)
    with capi.Phaserot(n_channels=2, blksiz=8192, oversample=os_) as h, \
            capi.Phaserot(n_channels=2, blksiz=8192, oversample=os_, flags=capi.FLAG_NO_PRUNE) as hb:
        h.sweep(x)
        pk = h.peaks()
        for N in (1, 11):
            h.reset_stats()
            t = h.nth_peaks(x, N)
            if mat == "sine":
                assert h.stats()["dense_repeats"] > 0
            assert np.array_equal(t[:, :, 0], pk), N
            assert np.array_equal(t, hb.nth_peaks(x, N)), N


def _schedule(MS, start, end, stride):
    idx, a = set(), start
    while a <= end:
        idx.add(a % MS)
        a += stride
        if a >= end:
            break
    return sorted(idx)


@pytest.mark.parametrize("os_", [0, 2])
def test_forms_ranges_repeats(os_):
    import torch
    q = (O.programme(48000, 1.7, 2) * 32767).astype(np.int16)
    x16 = (q.astype(np.float32) / 32768).astype(np.float32)
    v24 = (O.programme(48000, 1.7, 2, seed=9) * 8388607).astype(np.int32)
    b = v24.astype("<i4").view(np.uint8).reshape(-1, 4)[:, :3].reshape(-1)
    x24 = (v24.astype(np.float64) / 2 ** 23).astype(np.float32)
    v32 = v24 << 8
    N = 11
    with capi.Phaserot(n_channels=2, blksiz=4096, oversample=os_) as h:
        MS = h.maxsample
        for pcms, xf in (((q,), x16), ((b, v32), x24)):
            xd = torch.from_numpy(np.ascontiguousarray(xf)).cuda()
            ref = h.nth_peaks_device(xd.data_ptr(), xf.shape[0], N)
            for got in [h.nth_peaks(p, N) for p in pcms] + [h.nth_peaks(xf, N), h.nth_peaks_device(xd.data_ptr(), xf.shape[0], N)]:
                assert np.array_equal(got, ref)
            # (0, 720, 360): index 0 as angle 0 and wrapped; (10, 800, 10): wrapped only
            for start, end, stride, chn in [(10, 200, 7, -1), (0, 360, 5, 1), (0, 1, 1, -1), (200, 500, 3, 0), (37, 37, 1, -1), (0, 720, 360, -1),
                                            (10, 800, 10, -1)]:
                t = h.nth_peaks(xf, N, start, end, stride, chn)
                mask = np.zeros((2, MS), bool)
                mask[np.ix_([0, 1] if chn < 0 else [chn], _schedule(MS, start, end, stride))] = True
                sel = mask.copy()
                sel[:, 0] = False                         # index 0: checked against the sweep of the same schedule below
                assert np.array_equal(t[sel], ref[sel]), (start, end, stride, chn)
                assert not t[~mask].any()
                with capi.Phaserot(n_channels=2, blksiz=4096, oversample=os_) as hs:
                    hs.sweep(xf, start, end, stride, chn)
                    assert np.array_equal(t[:, :, 0], hs.peaks()), (start, end, stride, chn)


def test_no_side_effects():
    import torch
    x = O.programme(48000, 2.2, 2)
    with capi.Phaserot(n_channels=2, blksiz=8192) as h:
        y0 = h.render(x, [37, 181], 1)               # before any rank-table call
        t = h.nth_peaks(x, 11)
        assert not h.peaks().any()
        assert np.array_equal(h.render(x, [37, 181], 1), y0)
        h.sweep_sections(x, 2 * R.seg_samples(8192))
        sp = h.section_peaks()
        h.nth_peaks(x, 11)
        assert np.array_equal(h.section_peaks(), sp)
        xd = torch.from_numpy(x).cuda()
        h.sweep_device(xd.data_ptr(), x.shape[0])   # pending
        assert np.array_equal(h.nth_peaks(x, 11), t)
        pk = h.peaks()
        assert np.array_equal(h.render(x, [37, 181], 1), y0)
    with capi.Phaserot(n_channels=2, blksiz=8192) as r:
        r.sweep_device(xd.data_ptr(), x.shape[0])
        assert np.array_equal(pk, r.peaks())


def test_errors():
    lib = capi.load()
    x = O.programme(48000, 0.3, 2)
    out = np.zeros((2, 360, 256), np.float32)
    with capi.Phaserot(mode=capi.MODE_PLUGIN, n_channels=2, sample_rate=48000.0) as p:
        with pytest.raises(capi.PhaserotError) as e:
            p.nth_peaks(x, 11)
        assert e.value.code == capi.E_STATE
    with capi.Phaserot(n_channels=2, blksiz=8192) as h:
        for n in (0, -1, 257):
            with pytest.raises(capi.PhaserotError) as e:
                h.nth_peaks(x, n)
            assert e.value.code == capi.E_INVAL and "n_rank" in str(e.value)
        F = x.shape[0]
        assert lib.phaserot_nth_peaks(h._h, capi._ptr(x), capi.PCM_F32, 0, 11, 0, 360, 1, -1, capi._ptr(out)) == capi.E_INVAL
        assert lib.phaserot_nth_peaks(h._h, capi._ptr(x), capi.PCM_F32, F, 11, 0, 360, 1, -1, None) == capi.E_INVAL
        assert lib.phaserot_nth_peaks(h._h, None, capi.PCM_F32, F, 11, 0, 360, 1, -1, capi._ptr(out)) == capi.E_INVAL
        assert lib.phaserot_nth_peaks(h._h, capi._ptr(x), capi.PCM_F32, F, 11, 0, 360, 0, -1, capi._ptr(out)) == capi.E_INVAL
        assert lib.phaserot_nth_peaks(h._h, capi._ptr(x), capi.PCM_F32, F, 11, 0, 360, 1, 2, capi._ptr(out)) == capi.E_INVAL
        assert lib.phaserot_nth_peaks(h._h, capi._ptr(x), capi.PCM_F32, F, 256, 0, 360, 1, -1, capi._ptr(out)) == capi.OK
        assert lib.phaserot_nth_peaks_device(h._h, None, F, 11, 0, 360, 1, -1, capi._ptr(out)) == capi.E_INVAL


def _db(v):
    v = np.float32(v)
    return float(np.float32(20.0) * np.log10(v)) if v >= 1e-15 else -np.inf


def _replay(tab, MS, S=2):
    """the CLI's search with -s 1 (cli:815-929) on a [C][MS] table: the result lines"""
    C = tab.shape[0]
    ang, p_min = [0] * C, [np.inf] * C
    for c in range(C):
        row = tab[c]
        if row.max() - row.min() == 0:
            continue
        p_min[c] = row.min()
        ang[c] = max(a for a in range(MS) if row[a] <= row.min())         # ties: the largest angle
    valid = [c for c in range(C) if p_min[c] != np.inf]
    avg = np.float32(sum(ang[c] for c in valid)) / np.float32(len(valid))
    dist = np.float32(MS) / np.float32(len(valid))
    out = list(ang)
    for c in valid:
        if ang[c] > 90 * S and abs(np.float32(ang[c]) - avg) > dist:
            out[c] -= MS
        elif avg > 90 * S:
            out[c] -= MS
    lines = []
    for c in range(C):
        if p_min[c] == np.inf:
            lines.append((c, 0, None))
        else:
            lines.append((c, out[c], (_db(tab[c, 0]) - _db(tab[c, ang[c]]), _db(tab[c, 0]), _db(tab[c, ang[c]]))))
    return lines


@pytest.mark.parametrize("tp", [False, True])
def test_cli_end_to_end(tmp_path, tp):
    from phaserotate.lv2_b200 import build
    x = O.programme(48000, 6.0, 2)
    wav = str(tmp_path / "in.wav")
    O.write_wav_f32(wav, x, 48000)
    exe = os.path.join(build.BIN_DIR, "phase-rotate")
    extra = ["--true-peak"] if tp else []

    def run(*argv):
        r = subprocess.run([exe] + extra + list(argv), capture_output=True, text=True)
        assert r.returncode == 0, r.stderr
        return r

    # rank 1: byte for byte the run without the option, stdout, stderr and the written file
    for argv in (["-s", "1"], [], ["-vv", "-l"], ["--overs", "-3"]):
        a, b = run(*argv, wav), run("--nth-peak", "1", *argv, wav)
        assert (a.stdout, a.stderr) == (b.stdout, b.stderr), argv
    o1, o2 = str(tmp_path / "o1.wav"), str(tmp_path / "o2.wav")
    a, b = run("-v", wav, o1), run("-v", "--nth-peak", "1", wav, o2)
    assert (a.stdout, a.stderr) == (b.stdout, b.stderr)
    assert np.array_equal(O.read_wav_f32(o1)[0], O.read_wav_f32(o2)[0])

    # rank 11: the search on out[..., 10], and the file rendered at the printed angles
    with capi.Phaserot(n_channels=2, blksiz=8192, oversample=4 if tp else 0) as h:
        t = h.nth_peaks(x, 11)
        MS = h.maxsample
        want = _replay(t[:, :, 10], MS)
        out = str(tmp_path / "o11.wav")
        r = run("-v", "-s", "1", "--fixed-write", "--nth-peak", "11", wav, out)
        lines = r.stdout.splitlines()
        k = lines.index("# Result -- Minimize digital peak, rank 11")
        got = lines[k + 1:k + 3]
        angles = []
        for line, (c, a, db) in zip(got, want):
            m = re.match(r"Channel: +(\d+) Phase: +(-?[\d.]+) deg(?:, gain: +(-?[\d.]+) dB \(att\. (-?[\d.]+) to (-?[\d.]+) dBFS\))?$", line)
            assert m and int(m[1]) == c + 1, line
            assert float(m[2]) == a / 2, (line, a)
            if a != 0:
                assert np.allclose([float(v) for v in m.group(3, 4, 5)], db, atol=0.0051), (line, db)
            angles.append(a)
        y = h.render(x, angles, 1)
        assert np.array_equal(O.read_wav_f32(out)[0], y[4096:4096 + x.shape[0]])
    r = run("-s", "1", "--nth-peak", "11", wav)
    assert r.stdout.splitlines()[0] == "# Result -- Minimize digital peak, rank 11"
