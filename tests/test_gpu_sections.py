"""Per-section analysis and render (phaserot_sweep_sections*, phaserot_render_sections*) on the GPU.

Every section table must equal the shard sweep of that section bit for bit (history = the blksiz frames
before it), and the max over the sections must equal the whole-stream sweep bit for bit."""
import os

import numpy as np
import pytest

import oracle_lib as O
from phaserotate.lv2_b200 import capi

pytestmark = pytest.mark.gpu


def _tones(seconds, parts, sr=48000):
    t = np.arange(int(sr * seconds)) / sr
    x = np.zeros((t.size, 2), np.float32)
    for c in range(2):
        x[:, c] = sum(a * np.sin(2 * np.pi * f * t + ph[c]) for a, f, ph in parts)
    return x


def _shard_tables(torch, x, xd, S, blksiz, subsample, ang, chn):
    """Reference: one phaserot_sweep_shard_device call per section on a fresh table."""
    n, nc = x.shape
    L = blksiz
    ns = (n + S - 1) // S
    out = []
    with capi.Phaserot(n_channels=nc, blksiz=blksiz, subsample=subsample) as h:
        for k in range(ns):
            f0, f1 = k * S, min(n, (k + 1) * S)
            h.reset()
            hist = xd[f0 - L:f0].data_ptr() if k else None
            h.sweep_shard_device(xd[f0:].data_ptr(), f1 - f0, hist, k == 0, k == ns - 1, *ang, chn=chn)
            out.append(h.peaks())
        h.reset()
        h.sweep_device(xd.data_ptr(), n, *ang, chn=chn)
        whole = h.peaks()
    return np.stack(out), whole


def _check(x, blksiz=8192, units=1, subsample=2, ang=(0, None, 1), chn=-1, form="device", expect_dense=False):
    import torch
    x = np.ascontiguousarray(x, np.float32)
    xd = torch.from_numpy(x).cuda()
    nc = x.shape[1]
    with capi.Phaserot(n_channels=nc, blksiz=blksiz, subsample=subsample) as h:
        S = units * h.shard_align()
        ang = (ang[0], h.maxsample if ang[1] is None else ang[1], ang[2])
        h.reset_stats()
        if form == "device":
            h.sweep_sections_device(xd.data_ptr(), x.shape[0], S, *ang, chn=chn)
        elif form == "float":
            h.sweep_sections(x, S, *ang, chn=chn)
        else:
            q = np.clip(np.round(x * 32768.0), -32768, 32767).astype(np.int16)
            h.sweep_sections(q, S, *ang, chn=chn)
            x = (q.astype(np.float32) / 32768.0).astype(np.float32)   # what sf_readf_float delivers
            xd = torch.from_numpy(x).cuda()
        got = h.section_peaks()
        st = h.stats()
        assert np.array_equal(h.peaks(), np.zeros_like(h.peaks()))    # the handle's own table is not touched
    ref, whole = _shard_tables(torch, x, xd, S, blksiz, subsample, ang, chn)
    assert got.shape == ref.shape == ((x.shape[0] + S - 1) // S, nc, 180 * subsample)
    for k in range(got.shape[0]):
        assert np.array_equal(got[k], ref[k]), f"section {k} differs from its shard sweep"
    assert np.array_equal(got.max(0), whole)
    if expect_dense:
        assert st["dense_repeats"] > 0
    return got, st


@pytest.mark.parametrize("nc,seconds,units", [
    (1, 12.0, 1),        # sections of one alignment unit
    (2, 30.0, 3),        # short last section
    (8, 6.0, 2),
])
def test_sections_equal_shards_programme(nc, seconds, units):
    _check(O.programme(48000, seconds, nc), units=units)


def test_sections_exactly_aligned_and_single_section():
    x = O.programme(48000, 30.0, 2)
    with capi.Phaserot(n_channels=2, blksiz=8192) as h:
        al = h.shard_align()
    n = 6 * al
    _check(x[:n], units=2)                                  # three full sections, no remainder
    got, _ = _check(x, units=(x.shape[0] + al - 1) // al)   # one section (length >= stream)
    assert got.shape[0] == 1


def test_sections_two_partitions():
    _check(O.programme(48000, 24.0, 2), blksiz=32768, units=2)


def test_sections_channel_stride_and_fine_grid():
    _check(O.programme(48000, 15.0, 2), units=2, subsample=10, ang=(30, 1250, 7), chn=1)


def test_sections_host_forms():
    x = O.programme(48000, 15.0, 2)
    _check(x, units=2, form="float")
    _check(x, units=2, form="int16")


def test_sections_two_tones_and_sine_overflow_fallback():
    _check(O.two_sine(48000, 20.0, 2), units=3)
    _check(_tones(10.0, [(0.5, 440.0, [0.0, 1.0])]), units=4, expect_dense=True)


def test_sections_match_oracle():
    x = O.programme(48000, 3.0, 2)
    with capi.Phaserot(n_channels=2, blksiz=8192) as h:
        S = h.shard_align()
        h.sweep_sections(x, S)
        got = h.section_peaks()
    ns = got.shape[0]
    for k in range(ns):
        f0, f1 = k * S, min(x.shape[0], (k + 1) * S)
        po = O.oracle_analyze_shard(x[f0:f1], 8192, x[f0 - 8192:f0] if k else None, k == 0, k == ns - 1)
        assert np.max(np.abs(got[k][:, 1:] - po[:, 1:]) / po[:, 1:]) <= 1e-5
        # grid index 0: the raw peak of the direct branch x[t - blksiz/2] over the section's output samples
        # (the oracle's block form takes the undelayed block; both give the whole file's value in the max)
        raw = np.abs(x[max(0, f0 - 4096):(x.shape[0] if k == ns - 1 else f1 - 4096)]).max(0)
        assert np.array_equal(got[k][:, 0], raw)


def test_sections_launches_do_not_grow_and_limits():
    import torch
    x = O.programme(48000, 120.0, 2)
    xd = torch.from_numpy(x).cuda()
    with capi.Phaserot(n_channels=2, blksiz=8192) as h:
        al = h.shard_align()
        launches = []
        for S in ((x.shape[0] + al - 1) // al * al, 20 * al):     # one section, then twelve of ~10 s
            h.reset_stats()
            h.sweep_sections_device(xd.data_ptr(), x.shape[0], S)
            st = h.stats()
            assert st["dense_repeats"] == 0
            launches.append(st["kernel_launches"])
        assert h.section_peaks().shape[0] == 12
        assert launches[0] == launches[1], launches
        with pytest.raises(capi.PhaserotError) as e:
            h.sweep_sections_device(xd.data_ptr(), x.shape[0], al + 8192)
        assert e.value.code == capi.E_INVAL
        with pytest.raises(capi.PhaserotError) as e:        # 65536 rows: over the documented limit
            h.sweep_sections_device(xd.data_ptr(), 32768 * al, al)
        assert e.value.code == capi.E_INVAL and "section rows" in str(e.value)
    with capi.Phaserot(n_channels=2, blksiz=8192, oversample=4) as h:
        with pytest.raises(capi.PhaserotError) as e:
            h.sweep_sections_device(xd.data_ptr(), x.shape[0], al)
        assert e.value.code == capi.E_UNSUPPORTED
    with capi.Phaserot(mode=capi.MODE_PLUGIN, n_channels=2, sample_rate=48000.0) as h:
        with pytest.raises(capi.PhaserotError) as e:
            h.sweep_sections_device(xd.data_ptr(), x.shape[0], 24576)
        assert e.value.code == capi.E_STATE


def test_render_sections():
    x = O.programme(48000, 5.0, 2)
    n, L = x.shape[0], 8192
    with capi.Phaserot(n_channels=2, blksiz=L) as h:
        MS = h.maxsample
        S = h.shard_align()
        # one section: phaserot_render bit for bit
        one = h.render_sections(x, (n + S - 1) // S * S, [[37, 181]])
        assert np.array_equal(one, h.render(x, [37, 181]))
        ns = (n + S - 1) // S
        rng = np.random.default_rng(7)
        ang = rng.integers(0, 2 * MS, size=(ns, 2)).astype(np.int32)
        ang[1] = [MS + 20, 5]              # a +180 degree representative
        y = h.render_sections(x, S, ang)
        T = y.shape[0]
        xd_ = h.render(x, [0, 0]).astype(np.float64)              # ca = 1, sa = 0: the delayed direct branch
        s_lut, c_lut = h.lut()
        y90 = h.render(x, [MS // 2, MS // 2]).astype(np.float64)
        H = (y90 - float(c_lut[MS // 2]) * xd_) / float(s_lut[MS // 2])
        mp = float(np.float32(2.0 * np.pi / 2 / -360.0))
        peak = float(np.abs(y).max())
        for k in range(ns):
            t0, t1 = k * S, (T if k == ns - 1 else (k + 1) * S)
            ref = h.render(x, ang[k] % MS)
            for c in range(2):
                sg = -1.0 if (ang[k, c] // MS) % 2 else 1.0
                s0 = t0 + (L if k else 0)
                assert np.array_equal(y[s0:t1, c], (sg * ref[s0:t1, c]).astype(np.float32)), (k, c)
                if k:
                    j = np.arange(L)
                    phi = ang[k - 1, c] + (ang[k, c] - ang[k - 1, c]) * (j + 1) / L
                    want = np.cos(phi * mp) * xd_[t0:t0 + L, c] + np.sin(phi * mp) * H[t0:t0 + L, c]
                    assert np.max(np.abs(y[t0:t0 + L, c] - want)) <= 1e-5 * peak, (k, c)
        # device form
        import torch
        xt = torch.from_numpy(np.ascontiguousarray(x)).cuda()
        yt = torch.zeros((T, 2), dtype=torch.float32, device="cuda")
        h.render_sections_device(xt.data_ptr(), n, S, ang, 1, yt.data_ptr())
        assert np.array_equal(yt.cpu().numpy(), y)


def _lround(v):
    import math
    return int(math.copysign(math.floor(abs(v) + 0.5), v))


def _replay_stride1(tab, S):
    """The CLI's search on one table with -s 1 (cli:815-929): the largest angle of the minimum, then the
    phase-distance rule.  Returns the applied angles (None for a channel without a minimum)."""
    C, MS = tab.shape
    ang, ok = [0] * C, [False] * C
    for c in range(C):
        pk = tab[c]
        if pk.max() - pk.min() == 0:
            continue
        ok[c] = True
        ang[c] = int(np.nonzero(pk <= pk.min())[0].max())
    n = sum(ok)
    avg = np.float32(sum(a for a, o in zip(ang, ok) if o)) / np.float32(n)
    dist = np.float32(MS) / np.float32(n)
    for c in range(C):
        if not ok[c]:
            continue
        if ang[c] > 90 * S and abs(np.float32(ang[c]) - avg) > dist:
            ang[c] -= MS
        elif avg > 90 * S:
            ang[c] -= MS
    return [a if o else None for a, o in zip(ang, ok)]


def test_cli_sections_end_to_end(tmp_path):
    from phaserotate.lv2_b200 import build
    import subprocess
    x = np.concatenate([O.programme(48000, 6.0, 2), O.two_sine(48000, 6.0, 2)])
    wav, out = str(tmp_path / "in.wav"), str(tmp_path / "out.wav")
    O.write_wav_f32(wav, x, 48000)
    exe = os.path.join(build.BIN_DIR, "phase-rotate")
    r = subprocess.run([exe, "-v", "-s", "1", "--sections", "1.3", wav], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    with capi.Phaserot(n_channels=2, blksiz=8192) as h:
        al = h.shard_align()
        S = -(-62400 // al) * al                    # 1.3 s = 62400 frames, rounded up to the alignment
        assert f"Section length  : {S / 48000:.3f} s ({S} frames)" in r.stdout
        h.sweep_sections(x, S)
        T = h.section_peaks()
        MS = h.maxsample
        lines = r.stdout.splitlines()
        assert lines.count("# Result -- Minimize digital peak") == 1
        heads = [i for i, l in enumerate(lines) if l.startswith("# Section ")]
        assert len(heads) == T.shape[0] == -(-x.shape[0] // S)
        render_ang = []
        for k, i in enumerate(heads):
            t1 = min(x.shape[0], (k + 1) * S)
            assert lines[i] == f"# Section {k + 1}: {k * S / 48000:.3f} - {t1 / 48000:.3f} s"
            want = _replay_stride1(T[k], 2)
            row = []
            for c in range(2):
                got = lines[i + 1 + c]
                if want[c] is None:
                    assert got == f"Channel: {c + 1:2d} Phase:   0 deg # cannot find min."
                    a = 0
                else:
                    assert got.startswith(f"Channel: {c + 1:2d} Phase: {want[c] / 2:5.2f} deg"), (got, want[c])
                    a = want[c]
                a = a % MS
                if k:
                    a += MS * _lround((render_ang[-1][c] - a) / MS)
                    assert abs(a - render_ang[-1][c]) <= MS // 2
                row.append(a)
            render_ang.append(row)
        r = subprocess.run([exe, "-s", "1", "--sections", "1.3", wav, out], capture_output=True, text=True)
        assert r.returncode == 0, r.stderr
        y = h.render_sections(x, S, np.array(render_ang, np.int32), 1)
    got = O.read_wav_f32(out)
    got = got[0] if isinstance(got, tuple) else got
    assert got.shape == x.shape
    assert np.array_equal(got, y[4096:4096 + x.shape[0]])
