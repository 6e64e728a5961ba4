"""Integrated loudness of the rotated output (phaserot_loudness*, phase-rotate --loudness) on the GPU.

The oracle is the float64 restatement in tests/loudness_ref.py applied to what phaserot_render writes
after the latency trim at the same angles: the device result must agree within 1e-3 LU."""
import os
import re
import subprocess

import ctypes as C
import numpy as np
import pytest

import loudness_ref as R
import oracle_lib as O
from phaserotate.lv2_b200 import capi

pytestmark = pytest.mark.gpu

TOL = 1e-3


def _rendered(h, x, angles, fs, weights=None):
    """Restatement on the trimmed render (the --fixed-write output) at per-channel angles."""
    y = h.render(x, angles, 1)
    D = h.blksiz // 2
    return R.integrated(y[D:D + x.shape[0]], fs, weights)


def _device(h, x, sets, fs, weights=None):
    import torch
    xd = torch.from_numpy(np.ascontiguousarray(x, np.float32)).cuda()
    return h.loudness_device(xd.data_ptr(), x.shape[0], sets, fs, weights)


@pytest.mark.parametrize("case", sorted(R.TECH3341))
def test_tech3341_at_angle_zero(case):
    x = R.sine_segments(48000, R.TECH3341[case])
    with capi.Phaserot(n_channels=2, blksiz=8192) as h:
        got = _device(h, x, [[0, 0]], 48000)[0]
    assert abs(got - R.integrated(x, 48000)) <= TOL
    assert abs(got - R.TECH3341_EXPECTED[case]) <= 0.1


@pytest.mark.parametrize("nc,blksiz,fs", [(1, 1024, 44100), (2, 8192, 48000), (6, 32768, 96000), (2, 32768, 44100), (6, 1024, 48000)])
def test_angle_sets_match_render(nc, blksiz, fs):
    x = O.programme(fs, 4.3, nc)
    G = R.WEIGHTS_5_1 if nc == 6 else None
    with capi.Phaserot(n_channels=nc, blksiz=blksiz) as h:
        MS = h.maxsample
        rng = np.random.default_rng(nc * 7 + blksiz)
        sets = [[0] * nc, [37] * nc, [-90] * nc, [MS + 45] * nc, list(rng.integers(-2 * MS, 2 * MS, nc)), list(rng.integers(0, MS, nc))]
        got = _device(h, x, sets, fs, G)
        assert abs(got[0] - R.integrated(x, fs, G)) <= TOL      # angle 0 is the input itself
        for k, s in enumerate(sets):
            want = _rendered(h, x, s, fs, G)
            assert abs(got[k] - want) <= TOL, (k, s, got[k], want)


def test_full_grid_sweep_of_common_angles():
    x = O.programme(48000, 3.0, 2)
    with capi.Phaserot(n_channels=2, blksiz=8192) as h:
        grid = list(range(0, h.maxsample, 15))
        got = _device(h, x, [[a, a] for a in grid], 48000)
        for a, g in zip(grid, got):
            assert abs(g - _rendered(h, x, [a, a], 48000)) <= TOL, a
    # the Hilbert branch loses gain near DC: the loudness moves with the angle, a little
    assert 0 < np.ptp(got) < 1.0


def test_host_forms_and_repeats_are_identical():
    x = O.programme(48000, 2.5, 2)
    sets = [[0, 0], [91, -17], [400, 3]]
    q16 = np.clip(np.round(x * 32768.0), -32768, 32767).astype(np.int16)
    q32 = (np.clip(np.round(x * 8388608.0), -8388608, 8388607).astype(np.int32) << 8)
    b24 = np.ascontiguousarray((q32 >> 8).astype("<i4").view(np.uint8).reshape(-1, 4)[:, :3]).reshape(-1)
    with capi.Phaserot(n_channels=2, blksiz=8192) as h:
        f = h.loudness(x, sets, 48000)
        assert np.array_equal(f, _device(h, x, sets, 48000))
        assert np.array_equal(f, h.loudness(x, sets, 48000))
        for pcm, wide in [(q16, q16.astype(np.float32) / np.float32(32768.0)),
                          (q32, (q32.astype(np.float64) / 2147483648.0).astype(np.float32)),
                          (b24, ((q32 >> 8).astype(np.float64) / 8388608.0).astype(np.float32))]:
            assert np.array_equal(h.loudness(pcm, sets, 48000), _device(h, wide, sets, 48000)), pcm.dtype
    # a true-peak handle measures the same
    with capi.Phaserot(n_channels=2, blksiz=8192, oversample=4) as h:
        assert np.array_equal(h.loudness(x, sets, 48000), f)


def test_edge_cases():
    fs = 48000
    with capi.Phaserot(n_channels=2, blksiz=8192) as h:
        x = O.programme(fs, 1.2, 2)
        assert h.loudness(x[:19199], [[0, 0], [50, 50]], fs).tolist() == [-np.inf, -np.inf]   # shorter than 400 ms
        assert h.loudness(np.zeros((96000, 2), np.float32), [[0, 0], [50, 50]], fs).tolist() == [-np.inf, -np.inf]
        for n in (19200, 19200 + 1234, 48000 + 4799):                                         # one block; F % step != 0
            got = h.loudness(x[:n], [[0, 0], [123, 300]], fs)
            assert abs(got[0] - R.integrated(x[:n], fs)) <= TOL, n
            assert abs(got[1] - _rendered(h, x[:n], [123, 300], fs)) <= TOL, n


def test_handle_state_untouched():
    x = O.programme(48000, 2.0, 2)
    with capi.Phaserot(n_channels=2, blksiz=8192) as h:
        before = h.render(x, [33, 77], 1)
        h.loudness(x, [[0, 0], [33, 77]], 48000)
        assert np.array_equal(h.peaks(), np.zeros_like(h.peaks()))
        assert np.array_equal(h.render(x, [33, 77], 1), before)


def test_errors():
    x = O.programme(48000, 1.0, 2)
    with capi.Phaserot(mode=capi.MODE_PLUGIN, n_channels=2, sample_rate=48000.0) as p:
        with pytest.raises(capi.PhaserotError) as e:
            p.loudness(x, [[0, 0]], 48000)
        assert e.value.code == capi.E_STATE
    with capi.Phaserot(n_channels=2, blksiz=8192) as h:
        lib, hh = h._lib, h._h
        ang = np.zeros(2, np.int32)
        out = np.zeros(1, np.float64)
        xp = x.ctypes.data_as(C.c_void_p)

        def call(data=xp, fmt=capi.PCM_F32, n=x.shape[0], fs=48000.0, w=None, a=ang, ns=1, o=out):
            wp = None if w is None else np.asarray(w, np.float32).ctypes.data_as(C.c_void_p)
            return lib.phaserot_loudness(hh, data, fmt, n, fs, wp, None if a is None else a.ctypes.data_as(C.c_void_p), ns,
                                         None if o is None else o.ctypes.data_as(C.c_void_p))

        assert call() == capi.OK
        bad = [dict(ns=0), dict(ns=-1), dict(a=None), dict(o=None), dict(w=[1.0, -1.0]), dict(w=[np.nan, 1.0]), dict(w=[1.0, np.inf]),
               dict(n=0), dict(fs=7999.0), dict(fs=768001.0), dict(fs=float("nan")), dict(data=None), dict(fmt=7)]
        for kw in bad:
            assert call(**kw) == capi.E_INVAL, kw
            assert lib.phaserot_last_error().decode(), kw
        assert lib.phaserot_loudness_device(hh, None, 100, 48000.0, None, ang.ctypes.data_as(C.c_void_p), 1, out.ctypes.data_as(C.c_void_p)) == capi.E_INVAL


def _to_db(v):
    return 20.0 * np.log10(np.float32(v)) if v >= 1e-15 else -np.inf


def test_cli_loudness_end_to_end(tmp_path):
    from phaserotate.lv2_b200 import build
    x = O.programme(48000, 8.0, 2)
    wav, out, out2 = str(tmp_path / "in.wav"), str(tmp_path / "out.wav"), str(tmp_path / "out2.wav")
    O.write_wav_f32(wav, x, 48000)
    exe = os.path.join(build.BIN_DIR, "phase-rotate")
    plain = subprocess.run([exe, "-s", "1", wav], capture_output=True, text=True)
    r = subprocess.run([exe, "--loudness", "-s", "1", wav], capture_output=True, text=True)
    assert plain.returncode == 0 and r.returncode == 0, r.stderr
    lines = r.stdout.splitlines()
    assert "\n".join(lines[:-3]) + "\n" == plain.stdout                 # without --loudness: the output as before
    assert lines[-3] == "# Loudness -- ITU-R BS.1770-4 integrated"
    m_in = re.fullmatch(r"Input : (-?[\d.]+|-inf) LUFS, PLR (-?[\d.]+|inf) dB", lines[-2])
    m_out = re.fullmatch(r"Output: (-?[\d.]+|-inf) LUFS, PLR (-?[\d.]+|inf) dB", lines[-1])
    assert m_in and m_out, lines[-3:]
    l_in, plr_in, l_out, plr_out = float(m_in[1]), float(m_in[2]), float(m_out[1]), float(m_out[2])
    assert abs(l_in - R.integrated(x, 48000)) <= 0.01
    # the peaks of the result lines: raw peak and the peak at the applied angle of every channel
    ang = [int(round(float(re.search(r"Phase: +(-?[\d.]+) deg", l)[1]) * 2)) for l in lines if l.startswith("Channel:")]
    with capi.Phaserot(n_channels=2, blksiz=8192) as h:
        h.sweep(x)
        pk = h.peaks()
        MS = h.maxsample
    assert abs(plr_in - (_to_db(pk[:, 0].max()) - l_in)) <= 0.011
    assert abs(plr_out - (_to_db(max(pk[c, a % MS] for c, a in enumerate(ang))) - l_out)) <= 0.011
    # the Output line measures the --fixed-write render, and --loudness does not change what is written
    r = subprocess.run([exe, "--loudness", "--fixed-write", "-s", "1", wav, out], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    w = subprocess.run([exe, "--fixed-write", "-s", "1", wav, out2], capture_output=True, text=True)
    assert w.returncode == 0 and w.stdout == "", w.stderr
    lines = r.stdout.splitlines()
    assert lines[0] == "# Loudness -- ITU-R BS.1770-4 integrated" and len(lines) == 3
    y = O.read_wav_f32(out)[0]
    assert np.array_equal(y, O.read_wav_f32(out2)[0])
    assert abs(float(lines[2].split()[1]) - R.integrated(y, 48000)) <= 0.01
    assert abs(float(lines[2].split()[1]) - l_out) <= 0.01
