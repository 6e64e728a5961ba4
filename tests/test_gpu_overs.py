"""Overs table (phaserot_overs*, phase-rotate --overs) on the GPU.

References: the unpruned brute force of the library itself (PHASEROT_FLAG_NO_PRUNE lists every point: equal
bit for bit), the peak table of phaserot_sweep (counts[c][a] > 0 exactly when peak[c][a] > T), and an
independent float64 restatement of the sample set (closed-form Hilbert taps, fftconvolve, upfirdn)."""
import os
import re
import subprocess

import numpy as np
import pytest
import scipy.signal as sg

import oracle_lib as O
from phaserotate.lv2_b200 import capi
from test_truepeak_independent import hilbert_taps, interpolated

pytestmark = pytest.mark.gpu


def _sine(sr, seconds, channels, f=997.0, amp=0.8):
    t = np.arange(int(sr * seconds))
    return np.stack([amp * np.sin(2 * np.pi * f / sr * t + 0.4 * c) for c in range(channels)], 1).astype(np.float32)


MATERIAL = {
    "programme": lambda sec, nc: O.programme(48000, sec, nc),
    "two_sine": lambda sec, nc: O.two_sine(48000, sec, nc),
    "sine": lambda sec, nc: _sine(48000, sec, nc),
}


def _peaks(x, nc, L, os_):
    with capi.Phaserot(n_channels=nc, blksiz=L, oversample=os_) as h:
        h.sweep(x)
        return h.peaks()


def _ceilings(pk):
    return {"above": float(pk.max()) * 1.01, "between": 0.5 * float(pk.min() + pk.max()), "minus12": float(pk.max()) * 10 ** (-12 / 20)}


CASES = [(nc, L, os_, mat) for os_ in (0, 2, 4) for mat in sorted(MATERIAL) for nc, L in [(1, 1024), (2, 8192), (8, 32768)]]


@pytest.mark.parametrize("nc,L,os_,mat", CASES)
def test_pruned_equals_brute_force_and_sweep(nc, L, os_, mat):
    x = MATERIAL[mat](1.3 if nc < 8 else 0.6, nc)
    pk = _peaks(x, nc, L, os_)
    with capi.Phaserot(n_channels=nc, blksiz=L, oversample=os_) as hp, \
            capi.Phaserot(n_channels=nc, blksiz=L, oversample=os_, flags=capi.FLAG_NO_PRUNE) as hb:
        for name, T in _ceilings(pk).items():
            T = float(np.float32(T))
            hp.reset_stats()
            hb.reset_stats()
            cp, ep = hp.overs(x, T)
            cb, eb = hb.overs(x, T)
            assert np.array_equal(cp, cb), name
            assert np.array_equal(ep, eb), name
            assert np.array_equal(cp > 0, pk > np.float32(T)), name      # identity with the sweep, index 0 included
            # the brute force evaluates every examined point; the pruned pass only those at or above the radius
            sp, sb = hp.stats(), hb.stats()
            assert sb["points_evaluated"] == sb["points_total"] == sp["points_total"] > 0, name
            assert sp["points_evaluated"] <= sp["points_total"]
            if name == "above":
                assert not cp.any() and not ep.any()
                assert sp["points_evaluated"] < sp["points_total"]


def _restated(x, L, S, os_, T):
    """(lo, hi, excess, vsum) per [c][a] in float64: counts of v > T (1 + 2e-6) and v > T (1 - 2e-6), the excess
    sum (v - T) over v > T and the sum of v over the same samples."""
    F, nc = x.shape
    D = L // 2
    B = -(-F // L)
    Tn = (B + 1) * L
    MS = 180 * S
    taps = hilbert_taps(L)
    ang = -np.arange(MS) * np.pi / MS
    out = np.zeros((4, nc, MS))
    rows = (lambda s: s[None, :]) if os_ <= 1 else (lambda s: interpolated(s, os_))

    def tally(v, c, a):
        out[0, c, a] = np.count_nonzero(v > T * (1 + 2e-6))
        out[1, c, a] = np.count_nonzero(v > T * (1 - 2e-6))
        o = v > T
        out[2, c, a] = np.sum(v[o] - T)
        out[3, c, a] = np.sum(v[o])

    for c in range(nc):
        xc = np.zeros(Tn)
        xc[:F] = x[:, c].astype(np.float64)
        H = sg.fftconvolve(xc, taps)[:Tn]
        xd = np.concatenate([np.zeros(D), xc])[:Tn]
        xd[:L] = 0.0                                       # first-block rule
        xi, hi = rows(xd)[:, D:], rows(H)[:, D:]          # examined samples t >= L/2
        for a in range(1, MS):
            tally(np.abs(np.cos(ang[a]) * xi + np.sin(ang[a]) * hi).max(0), c, a)
        tally(np.abs(rows(xc)).max(0), c, 0)              # raw input, same detector
    return out


@pytest.mark.parametrize("os_", [0, 2, 4])
@pytest.mark.parametrize("mat,L", [("programme", 2048), ("two_sine", 8192)])
def test_independent_float64(os_, mat, L):
    x = MATERIAL[mat](0.8, 2)
    pk = _peaks(x, 2, L, os_)
    with capi.Phaserot(n_channels=2, blksiz=L, oversample=os_) as h:
        for T in (0.5 * float(pk.min() + pk.max()), float(pk.max()) * 10 ** (-6 / 20)):
            T = float(np.float32(T))
            cnt, exc = h.overs(x, T)
            lo, hi, ex, vs = _restated(x, L, 2, os_, T)
            assert np.all(cnt >= lo) and np.all(cnt <= hi)
            # Each term v - T carries the fp32 error of v itself, which the peak tests bound at 1e-5 of v, not of
            # v - T: near the ceiling v - T is far smaller than v, so the bound is 1e-5 of the sum of v over the
            # overs (not of the excess), plus one 2^-32 truncation per term.
            assert np.all(np.abs(exc - ex) <= 1e-5 * vs + cnt * 2.0 ** -32)


@pytest.mark.parametrize("os_", [0, 4])
def test_overflow_repeats_equal_brute_force(os_):
    x = _sine(48000, 40.0, 8)
    with capi.Phaserot(n_channels=8, blksiz=8192, oversample=os_) as hp, \
            capi.Phaserot(n_channels=8, blksiz=8192, oversample=os_, flags=capi.FLAG_NO_PRUNE) as hb:
        T = float(np.float32(0.8 * 10 ** (-20 / 20)))
        cp, ep = hp.overs(x, T)
        assert hp.stats()["dense_repeats"] > 0
        cb, eb = hb.overs(x, T)
        assert np.array_equal(cp, cb) and np.array_equal(ep, eb)
        assert cp[:, 1:].min() > 0.9 * x.shape[0]


def _schedule(MS, start, end, stride):
    idx, raw, a = set(), False, start
    while a <= end:
        if a == 0:
            raw = True
        else:
            idx.add(a % MS)
        a += stride
        if a >= end:
            break
    if raw:
        idx.add(0)
    return sorted(idx)


@pytest.mark.parametrize("os_", [0, 2])
def test_forms_ranges_repeats(os_):
    import torch
    q = (O.programme(48000, 1.7, 2) * 32767).astype(np.int16)
    x16 = (q.astype(np.float32) / 32768).astype(np.float32)
    v24 = (O.programme(48000, 1.7, 2, seed=9) * 8388607).astype(np.int32)
    b = v24.astype("<i4").view(np.uint8).reshape(-1, 4)[:, :3].reshape(-1)
    x24 = (v24.astype(np.float64) / 2 ** 23).astype(np.float32)
    with capi.Phaserot(n_channels=2, blksiz=4096, oversample=os_) as h:
        MS = h.maxsample
        for pcm, xf in ((q, x16), (b, x24)):
            T = float(np.float32(0.6 * np.abs(xf).max()))
            ref = h.overs(xf, T)
            for got in (h.overs(pcm, T), h.overs(xf, T)):
                assert np.array_equal(got[0], ref[0]) and np.array_equal(got[1], ref[1])
            xd = torch.from_numpy(np.ascontiguousarray(xf)).cuda()
            got = h.overs_device(xd.data_ptr(), xf.shape[0], T)
            assert np.array_equal(got[0], ref[0]) and np.array_equal(got[1], ref[1])
            for start, end, stride, chn in [(10, 200, 7, -1), (0, 360, 5, 1), (0, 1, 1, -1), (200, 500, 3, 0), (37, 37, 1, -1)]:
                c, e = h.overs(xf, T, start, end, stride, chn)
                mask = np.zeros((2, MS), bool)
                mask[np.ix_([0, 1] if chn < 0 else [chn], _schedule(MS, start, end, stride))] = True
                assert np.array_equal(c[mask], ref[0][mask]) and np.array_equal(e[mask], ref[1][mask]), (start, end, stride, chn)
                assert not c[~mask].any() and not e[~mask].any()


def test_no_side_effects():
    import torch
    x = O.programme(48000, 2.2, 2)
    T = float(np.float32(0.3 * np.abs(x).max()))
    with capi.Phaserot(n_channels=2, blksiz=8192) as h:
        y0 = h.render(x, [37, 181], 1)               # before any overs call
        h.overs(x, T)
        assert not h.peaks().any()
        assert np.array_equal(h.render(x, [37, 181], 1), y0)
        xd = torch.from_numpy(x).cuda()
        h.sweep_device(xd.data_ptr(), x.shape[0])   # pending
        h.overs(x, T)
        pk = h.peaks()
        assert np.array_equal(h.render(x, [37, 181], 1), y0)
    with capi.Phaserot(n_channels=2, blksiz=8192) as r:
        r.sweep_device(xd.data_ptr(), x.shape[0])
        assert np.array_equal(pk, r.peaks())


def test_errors():
    lib = capi.load()
    x = O.programme(48000, 0.3, 2)
    cnt = np.zeros((2, 360), np.uint64)
    with capi.Phaserot(mode=capi.MODE_PLUGIN, n_channels=2, sample_rate=48000.0) as p:
        with pytest.raises(capi.PhaserotError) as e:
            p.overs(x, 0.5)
        assert e.value.code == capi.E_STATE
    with capi.Phaserot(n_channels=2, blksiz=8192) as h:
        for T in (0.0, -0.5, float("nan"), float("inf")):
            with pytest.raises(capi.PhaserotError) as e:
                h.overs(x, T)
            assert e.value.code == capi.E_INVAL and "ceiling" in str(e.value)
        assert lib.phaserot_overs(h._h, capi._ptr(x), capi.PCM_F32, 0, 0.5, 0, 360, 1, -1, capi._ptr(cnt), None) == capi.E_INVAL
        assert lib.phaserot_overs(h._h, capi._ptr(x), capi.PCM_F32, x.shape[0], 0.5, 0, 360, 1, -1, None, None) == capi.E_INVAL
        assert lib.phaserot_overs(h._h, capi._ptr(x), capi.PCM_F32, x.shape[0], 0.5, 0, 360, 0, -1, capi._ptr(cnt), None) == capi.E_INVAL
        assert lib.phaserot_overs(h._h, capi._ptr(x), capi.PCM_F32, x.shape[0], 0.5, 0, 360, 1, 2, capi._ptr(cnt), None) == capi.E_INVAL
        assert lib.phaserot_overs(h._h, capi._ptr(x), capi.PCM_F32, x.shape[0], 0.5, 0, 360, 1, -1, capi._ptr(cnt), None) == capi.OK


def _overs_block(lines, nc):
    rows = []
    for l in lines:
        m = re.fullmatch(r"Channel: +(\d+) Input: (\d+) Output: (\d+) Fewest: (\d+) at ([\d.]+) deg", l)
        assert m, l
        rows.append((int(m[2]), int(m[3]), int(m[4]), float(m[5])))
    assert len(rows) == nc
    return rows


def _check_rows(rows, cnt, out_idx, S=2):
    for c, (n_in, n_out, n_few, at) in enumerate(rows):
        best = cnt.shape[1] - 1 - int(np.argmin(cnt[c][::-1]))          # ties: the largest index
        assert (n_in, n_out, n_few) == (int(cnt[c, 0]), int(cnt[c, out_idx[c]]), int(cnt[c, best]))
        assert abs(at - best / S) < 1e-6


@pytest.mark.parametrize("tp", [False, True])
def test_cli_end_to_end(tmp_path, tp):
    from phaserotate.lv2_b200 import build
    x = O.programme(48000, 6.0, 2)
    wav = str(tmp_path / "in.wav")
    O.write_wav_f32(wav, x, 48000)
    exe = os.path.join(build.BIN_DIR, "phase-rotate")
    extra = ["--true-peak"] if tp else []
    T = float(np.float32(10 ** (-3 / 20)))
    with capi.Phaserot(n_channels=2, blksiz=8192, oversample=4 if tp else 0) as h:
        cnt, _ = h.overs(x, T)
        MS = h.maxsample
    plain = subprocess.run([exe, "-s", "1"] + extra + [wav], capture_output=True, text=True)
    r = subprocess.run([exe, "-s", "1", "--overs", "-3"] + extra + [wav], capture_output=True, text=True)
    assert plain.returncode == 0 and r.returncode == 0, r.stderr
    lines = r.stdout.splitlines()
    assert "\n".join(lines[:-3]) + "\n" == plain.stdout                 # without --overs: the output as before
    assert lines[-3] == "# Overs -- samples above -3.00 " + ("dBTP" if tp else "dBFS")
    ang = [int(round(float(re.search(r"Phase: +(-?[\d.]+) deg", l)[1]) * 2)) for l in lines[:-3] if l.startswith("Channel:")]
    _check_rows(_overs_block(lines[-2:], 2), cnt, [a % MS for a in ang])
    # with --loudness: the loudness block first
    r = subprocess.run([exe, "-s", "1", "--loudness", "--overs", "-3"] + extra + [wav], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    lines = r.stdout.splitlines()
    assert "\n".join(lines[:-6]) + "\n" == plain.stdout
    assert lines[-6].startswith("# Loudness") and lines[-3].startswith("# Overs")
    _check_rows(_overs_block(lines[-2:], 2), cnt, [a % MS for a in ang])
    # with -a: the applied angles, wrapped into [0, 180) degrees; the written file does not change
    out, out2 = str(tmp_path / "out.wav"), str(tmp_path / "out2.wav")
    r = subprocess.run([exe, "--overs", "-3", "-a", "30,-45"] + extra + [wav, out], capture_output=True, text=True)
    w = subprocess.run([exe, "-a", "30,-45"] + extra + [wav, out2], capture_output=True, text=True)
    assert r.returncode == 0 and w.returncode == 0 and w.stdout == "", r.stderr
    lines = r.stdout.splitlines()
    assert len(lines) == 3 and lines[0].startswith("# Overs")
    _check_rows(_overs_block(lines[1:], 2), cnt, [60, (-90) % MS])
    assert np.array_equal(O.read_wav_f32(out)[0], O.read_wav_f32(out2)[0])
