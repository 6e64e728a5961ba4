"""GPU parity tests: the CUDA path (through the C ABI of libphaserot_cuda) against
the oracle, the golden vectors of the reference build, and size-independent
properties at full BASELINE sizes.  Run with `-m gpu` on a B200.

Tolerances (north_star): rendered audio and per-angle peaks within 1e-5
relative of the reference's fp32/FFTW path; selected angle identical where peaks
are not tied within tolerance."""
import os
import subprocess

import numpy as np
import pytest

import oracle_lib as O
from phaserotate.lv2_b200 import build, capi

pytestmark = pytest.mark.gpu

PEAK_TOL = 1e-5   # relative
AUDIO_TOL = 1e-5  # relative to the signal's full scale (peak of the reference output)


def rel(a, b):
    return float(np.max(np.abs(a - b) / np.maximum(np.abs(b), 1e-30)))


def argmin_equal_unless_tied(pg, po, tol=PEAK_TOL):
    """Identical argmin, except where the oracle's runner-up is within tolerance of its minimum."""
    for c in range(po.shape[0]):
        ag, ao = int(pg[c].argmin()), int(po[c].argmin())
        if ag != ao:
            assert abs(po[c, ag] - po[c, ao]) <= tol * po[c, ao], (c, ag, ao)


@pytest.fixture(scope="module", autouse=True)
def _built():
    build.build_library()
    build.build_host()
    O.build_oracle()


# ---------------------------------------------------------------------------
# sweep
# ---------------------------------------------------------------------------

SWEEP_CASES = {
    "two_sine_2ch_L8192": (lambda: O.two_sine(48000, 3.0, 2), 8192),
    "pink_mono_L8192": (lambda: O.pink_noise(120000, 7)[:, None], 8192),
    "programme_2ch_L4096": (lambda: O.programme(48000, 2.0, 2), 4096),
    "harmonic_3ch_L16384": (lambda: O.harmonic(96000, 1.0, 3), 16384),
    "short_2ch_L8192": (lambda: O.two_sine(48000, 1000 / 48000, 2), 8192),
    "odd_len_2ch_L1024": (lambda: O.harmonic(48000, 0.5, 2)[:23999], 1024),
    "one_frame_L2048": (lambda: np.array([[0.5, -0.25]], np.float32), 2048),
    "eight_ch_L1024": (lambda: O.harmonic(48000, 0.25, 8), 1024),
    # FIR length 32768 (192 kHz files, cli:749-755): two tap partitions on the device
    "harmonic_2ch_L32768": (lambda: O.harmonic(192000, 0.9, 2), 32768),
    "short_mono_L32768": (lambda: O.pink_noise(5000, 11)[:, None], 32768),
    # BASELINE config 5's shape: 8 interleaved channels AND the 32768-tap FIR (two tap partitions) together
    "eight_ch_L32768": (lambda: O.harmonic(192000, 0.22, 8), 32768),
}


@pytest.mark.parametrize("name", sorted(SWEEP_CASES))
@pytest.mark.parametrize("flags", [0, capi.FLAG_NO_PRUNE])
def test_sweep_matches_oracle(name, flags):
    gen, L = SWEEP_CASES[name]
    x = gen()
    po = O.oracle_analyze(x, L)
    with capi.Phaserot(n_channels=x.shape[1], blksiz=L, flags=flags) as h:
        h.sweep(x)
        pg = h.peaks()
        assert h.stats()["kernel_launches"] > 0
    assert rel(pg, po) <= PEAK_TOL
    assert np.array_equal(pg[:, 0], po[:, 0])  # raw input peak is exact
    argmin_equal_unless_tied(pg, po)


def test_sweep_empty_file():
    with capi.Phaserot(n_channels=2, blksiz=1024) as h:
        h.sweep(np.zeros((0, 2), np.float32))
        assert np.all(h.peaks() == 0)


def test_sweep_golden_reference_vectors(golden):
    g = golden["cli_analyze"]
    x, L = g["x"], int(g["blksiz"])
    with capi.Phaserot(n_channels=2, blksiz=L) as h:
        s, c = h.lut()
        assert np.array_equal(s, g["lut_sin"]) and np.array_equal(c, g["lut_cos"])
        for key, (a0, a1, st, ch) in {"full": (0, 360, 1, -1), "coarse": (0, 360, 24, -1), "refine": (-12, 13, 1, -1), "single": (36, 61, 1, 1)}.items():
            h.reset()
            h.sweep(x, a0, a1, st, ch)
            pg = h.peaks()
            assert np.array_equal(pg == 0, g[key] == 0), key  # same entries touched
            assert rel(pg, g[key]) <= PEAK_TOL, key
        h.reset()
        h.sweep(x)
        assert np.array_equal(h.peaks().argmin(1), g["full"].argmin(1))


def test_sweep_accumulates_like_peak_table():
    """PhaseRotate::_peak is a running max until reset (cli:414-421, 355-366)."""
    x = O.harmonic(48000, 0.6, 2)
    with capi.Phaserot(n_channels=2, blksiz=2048) as h:
        h.sweep(x, 0, 360, 24)
        h.sweep(0.5 * x, 0, 360, 1)
        pg = h.peaks()
        po = O.oracle_analyze(x, 2048, 2, 0, 360, 24)
        po = O.oracle_analyze(0.5 * x, 2048, 2, 0, 360, 1, -1, po)
        assert rel(pg, po) <= PEAK_TOL
        assert h.peak(-1, 24) == max(pg[0, 24], pg[1, 24])  # peak_all
        assert h.peak(1, -12) == pg[1, 348]                  # negative index wraps (cli:281-284)
        h.reset()
        assert np.all(h.peaks() == 0)


def test_sweep_fine_grid_and_subgrid_identity():
    """Subsample 10 (0.1 deg) against the oracle; its every-5th entry is the reference's 0.5 deg grid."""
    x = O.programme(48000, 1.5, 2)
    po = O.oracle_analyze(x, 8192, 10)
    with capi.Phaserot(n_channels=2, blksiz=8192, subsample=10) as h:
        h.sweep(x)
        p10 = h.peaks()
    with capi.Phaserot(n_channels=2, blksiz=8192, subsample=2) as h:
        h.sweep(x)
        p2 = h.peaks()
    assert rel(p10, po) <= PEAK_TOL
    argmin_equal_unless_tied(p10, po)
    assert rel(p10[:, ::5], p2) <= 2e-6  # same angles, independently rounded LUT arguments


def test_streaming_analyze_is_drop_in():
    x = O.harmonic(48000, 1.0, 2)
    L = 4096
    nblk = (x.shape[0] + L - 1) // L
    xp = np.zeros(((nblk + 1) * L, 2), np.float32)
    xp[: x.shape[0]] = x
    with capi.Phaserot(n_channels=2, blksiz=L) as h:
        for b in range(nblk + 1):  # analyze_file: real blocks then the zero flush block
            h.analyze(xp[b * L:(b + 1) * L], 0, 360, 1, -1, b == 0)
            if b == nblk // 2:
                h.sync()           # reading mid-stream must not disturb the stream
        pg = h.peaks()
        h2 = capi.Phaserot(n_channels=2, blksiz=L)
        h2.sweep(x)
        assert np.array_equal(pg, h2.peaks())
        h2.close()
    assert rel(pg, O.oracle_analyze(x, L)) <= PEAK_TOL


def test_first_block_quirk_flag():
    L = 1024
    x = np.zeros((4 * L, 1), np.float32)
    x[: L // 2, 0] = O.pink_noise(L // 2, 9, 0.9)
    with capi.Phaserot(n_channels=1, blksiz=L) as h:
        h.sweep(x)
        quirk = h.peaks()
    with capi.Phaserot(n_channels=1, blksiz=L, flags=capi.FLAG_NO_FIRST_BLOCK_QUIRK) as h:
        h.sweep(x)
        fixed = h.peaks()
    assert rel(quirk, O.oracle_analyze(x, L)) <= PEAK_TOL
    assert quirk[0, 1] < 0.2 * quirk[0, 0] and fixed[0, 1] > 0.9 * fixed[0, 0]


# ---------------------------------------------------------------------------
# properties at BASELINE sizes (no oracle needed)
# ---------------------------------------------------------------------------

def _device_programme(seconds, seed=43):
    import torch
    import bench
    dev = torch.device("cuda", 0)
    frames = int(seconds * bench.SR)
    frames -= frames % bench.BLKSIZ
    n_chunks = (frames + bench.GEN_CHUNK - 1) // bench.GEN_CHUNK
    x = torch.cat([bench.gen_chunk_torch(torch, k, dev, seed) for k in range(n_chunks)])[:frames].contiguous()
    torch.cuda.synchronize()
    return x, frames


def test_full_size_pruned_equals_brute_force_and_shards_combine():
    """10 min stereo at 0.1 deg: exact pruning leaves every peak bit-identical to brute force, and
    two sample-range shards combined by max equal the single pass bit for bit (SURVEY 8e)."""
    import bench
    x, frames = _device_programme(600.0)
    with capi.Phaserot(n_channels=2, blksiz=bench.BLKSIZ, subsample=10) as h:
        h.sweep_device(x.data_ptr(), frames)
        pruned = h.peaks()
        st = h.stats()
        assert st["points_evaluated"] < 0.2 * st["points_total"]
        # two shards
        al = h.shard_align()            # shards cut on the FFT segment grid -> bit-identical
        assert al % bench.BLKSIZ == 0
        half = (frames // 2) - ((frames // 2) % al)
        h.reset()
        h.sweep_shard_device(x.data_ptr(), half, None, True, False)
        a = h.peaks()
        hist = x[half - bench.BLKSIZ:half].cpu().numpy()
        h.reset()
        h.sweep_shard_device(x[half:].data_ptr(), frames - half, hist, False, True)
        b = h.peaks()
    with capi.Phaserot(n_channels=2, blksiz=bench.BLKSIZ, subsample=10, flags=capi.FLAG_NO_PRUNE) as h:
        h.sweep_device(x.data_ptr(), frames)
        brute = h.peaks()
    assert np.array_equal(pruned, brute)
    assert np.array_equal(np.maximum(a, b), brute)
    assert np.all(brute[:, 1:] > 0)
    # an unaligned cut still agrees to FFT rounding
    with capi.Phaserot(n_channels=2, blksiz=bench.BLKSIZ, subsample=10) as h:
        cut = half + bench.BLKSIZ
        h.sweep_shard_device(x.data_ptr(), cut, None, True, False)
        a = h.peaks()
        hist = x[cut - bench.BLKSIZ:cut].cpu().numpy()
        h.reset()
        h.sweep_shard_device(x[cut:].data_ptr(), frames - cut, hist, False, True)
        assert rel(np.maximum(a, h.peaks()), brute) <= 2e-6


def test_pending_table_on_device_and_device_history():
    """phaserot_pending_table: the device-resident table (per-angle maxima, then raw peaks) is what
    phaserot_peaks reads back; combining two shards by an element-wise max written INTO the second
    handle's device table (what the NCCL max all-reduce does in place) yields the whole-stream table.
    The shard history may be a device pointer."""
    import torch
    import bench
    x, frames = _device_programme(120.0)
    with capi.Phaserot(n_channels=2, blksiz=bench.BLKSIZ, subsample=10) as h:
        with pytest.raises(capi.PhaserotError):
            h.pending_table()              # nothing pending
        h.sweep_device(x.data_ptr(), frames)
        ptr, nc, na = h.pending_table()
        assert (nc, na) == (2, h.maxsample - 1)

        class _Dev:
            __cuda_array_interface__ = {"shape": (nc * na + nc,), "typestr": "<f4", "data": (ptr, False), "version": 2}
        t = torch.as_tensor(_Dev(), device=x.device)
        torch.cuda.synchronize()
        snap = t.clone().cpu().numpy()
        whole = h.peaks()
        assert np.array_equal(snap[:nc * na].reshape(nc, na), whole[:, 1:])
        assert np.array_equal(snap[nc * na:], whole[:, 0])
        al = h.shard_align()
        half = (frames // 2) - ((frames // 2) % al)
        h.reset()
        h.sweep_shard_device(x.data_ptr(), half, None, True, False)
        ptr_a, _, _ = h.pending_table()

        class _DevA:
            __cuda_array_interface__ = {"shape": (nc * na + nc,), "typestr": "<f4", "data": (ptr_a, False), "version": 2}
        torch.cuda.synchronize()
        first = torch.as_tensor(_DevA(), device=x.device).clone()
        h.peaks()
        h.reset()
        hist = x[half - bench.BLKSIZ:half].contiguous()
        h.sweep_shard_device(x[half:].data_ptr(), frames - half, hist.data_ptr(), False, True)   # device history
        ptr_b, _, _ = h.pending_table()

        class _DevB:
            __cuda_array_interface__ = {"shape": (nc * na + nc,), "typestr": "<f4", "data": (ptr_b, False), "version": 2}
        torch.cuda.synchronize()
        tb = torch.as_tensor(_DevB(), device=x.device)
        tb.copy_(torch.maximum(tb, first))     # in-place combine on the device
        torch.cuda.synchronize()
        assert np.array_equal(h.peaks(), whole)


def test_multichannel_paths_agree():
    """Four interleaved channels: host input (chunked upload), device input and two shards (host and
    device history) all give the table of the oracle / of one another; pruned == brute force bit for bit."""
    import torch
    x = O.programme(48000, 4.0, 2)
    x4 = np.ascontiguousarray(np.stack([x[:, 0], x[:, 1], 0.7 * x[::-1, 0], 0.5 * (x[:, 0] - x[:, 1])], 1).astype(np.float32))
    L = 8192
    frames = x4.shape[0] - x4.shape[0] % L
    x4 = x4[:frames]
    po = O.oracle_analyze(x4, L)
    xd = torch.from_numpy(x4).cuda()
    with capi.Phaserot(n_channels=4, blksiz=L) as h:
        h.sweep(x4)
        host = h.peaks()
        h.reset()
        h.sweep_device(xd.data_ptr(), frames)
        dev = h.peaks()
        al = h.shard_align()
        half = (frames // 2) - ((frames // 2) % al)
        tabs = []
        for hist_dev in (False, True):
            h.reset()
            h.sweep_shard_device(xd.data_ptr(), half, None, True, False)
            a = h.peaks()
            hist = xd[half - L:half].contiguous()
            h.reset()
            h.sweep_shard_device(xd[half:].data_ptr(), frames - half, hist.data_ptr() if hist_dev else hist.cpu().numpy(), False, True)
            tabs.append(np.maximum(a, h.peaks()))
    with capi.Phaserot(n_channels=4, blksiz=L, flags=capi.FLAG_NO_PRUNE) as h:
        h.sweep_device(xd.data_ptr(), frames)
        brute = h.peaks()
    assert rel(dev, po) <= PEAK_TOL
    assert np.array_equal(host, dev) and np.array_equal(dev, brute)
    assert np.array_equal(tabs[0], dev) and np.array_equal(tabs[1], dev)
    assert np.array_equal(dev.argmin(1), po.argmin(1))


def test_blksiz_32768_pruned_equals_brute_force_and_shards_combine():
    """FIR length 32768 (two tap partitions): 2 min stereo at 0.1 deg, same properties as above."""
    L = 32768
    x, frames = _device_programme(120.0)
    frames -= frames % L
    with capi.Phaserot(n_channels=2, blksiz=L, subsample=10) as h:
        h.sweep_device(x.data_ptr(), frames)
        pruned = h.peaks()
        al = h.shard_align()
        assert al % L == 0
        half = (frames // 2) - ((frames // 2) % al)
        h.reset()
        h.sweep_shard_device(x.data_ptr(), half, None, True, False)
        a = h.peaks()
        hist = x[half - L:half].cpu().numpy()
        h.reset()
        h.sweep_shard_device(x[half:].data_ptr(), frames - half, hist, False, True)
        b = h.peaks()
    with capi.Phaserot(n_channels=2, blksiz=L, subsample=10, flags=capi.FLAG_NO_PRUNE) as h:
        h.sweep_device(x.data_ptr(), frames)
        brute = h.peaks()
    assert np.array_equal(pruned, brute)
    assert np.array_equal(np.maximum(a, b), brute)
    assert np.all(brute[:, 1:] > 0)


# ---------------------------------------------------------------------------
# oversampled true-peak sweep (new capability, not in the reference: parity is
# against this repo's own CPU restatement of the definition in phaserot_cuda.h)
# ---------------------------------------------------------------------------

TP_CASES = {
    "two_sine_2ch_L8192": (lambda: O.two_sine(48000, 2.0, 2), 8192),
    "pink_mono_L4096": (lambda: O.pink_noise(90000, 5)[:, None], 4096),
    "programme_2ch_L16384": (lambda: O.programme(96000, 1.0, 2), 16384),
    "odd_len_3ch_L1024": (lambda: O.harmonic(48000, 0.5, 3)[:23999], 1024),
    "one_frame_L2048": (lambda: np.array([[0.5, -0.25]], np.float32), 2048),
    "harmonic_2ch_L32768": (lambda: O.harmonic(192000, 0.6, 2), 32768),
}


@pytest.mark.parametrize("name", sorted(TP_CASES))
@pytest.mark.parametrize("os_", [2, 4])
@pytest.mark.parametrize("flags", [0, capi.FLAG_NO_PRUNE])
def test_true_peak_sweep_matches_oracle(name, os_, flags):
    gen, L = TP_CASES[name]
    x = gen()
    po = O.oracle_analyze_tp(x, L, os_)
    pd = O.oracle_analyze(x, L)
    with capi.Phaserot(n_channels=x.shape[1], blksiz=L, flags=flags, oversample=os_) as h:
        h.sweep(x)
        pg = h.peaks()
        kt = h.stats()
    assert kt["kernel_launches"] > 0
    assert rel(pg, po) <= PEAK_TOL
    assert np.array_equal(pg[:, 0], po[:, 0])        # raw-input detector: same fp32 operations on both sides
    assert np.all(pg >= pd * (1 - 1e-6))             # the digital peak is part of the true-peak detector
    argmin_equal_unless_tied(pg, po)


def test_true_peak_quirk_flag_ranges_and_streaming():
    x = O.programme(48000, 1.5, 2)
    L = 4096
    # first-block rule switched off
    with capi.Phaserot(n_channels=2, blksiz=L, oversample=4, flags=capi.FLAG_NO_FIRST_BLOCK_QUIRK) as h:
        h.sweep(x)
        fixed = h.peaks()
    with capi.Phaserot(n_channels=2, blksiz=L, oversample=4) as h:
        h.sweep(x)
        quirk = h.peaks()
        assert np.all(fixed >= quirk)
        # a refine-style window on one channel
        h.reset()
        h.sweep(x, 30, 55, 1, 1)
        win = h.peaks()
        po = O.oracle_analyze_tp(x, L, 4, ang_start=30, ang_end=55, stride=1, only_chn=1)
        assert rel(win[po > 0], po[po > 0]) <= PEAK_TOL and np.all(win[po == 0] == 0)
        # block streaming (PhaseRotate::analyze drop-in) continues the interpolator across batches
        h.reset()
        nb = (x.shape[0] + L - 1) // L
        xp = np.zeros((nb * L, 2), np.float32)
        xp[:x.shape[0]] = x
        for b in range(nb):
            h.analyze(xp[b * L:(b + 1) * L], 0, 360, 1, -1, b == 0)
            if b == 3:
                h.sync()   # forces a batch boundary: the next batch continues from history
        h.analyze(np.zeros((L, 2), np.float32), 0, 360, 1, -1, False)
        assert rel(h.peaks(), quirk) <= 2e-6


def test_true_peak_full_size_pruned_equals_brute_force_and_shards_combine():
    """5 min stereo at 0.1 deg, 4x true-peak: pruning is exact, shards combine (to FFT rounding: the
    shard with history computes the 11 interpolator samples before its start from that history)."""
    import bench
    x, frames = _device_programme(300.0)
    with capi.Phaserot(n_channels=2, blksiz=bench.BLKSIZ, subsample=10, oversample=4) as h:
        h.sweep_device(x.data_ptr(), frames)
        pruned = h.peaks()
        st = h.stats()
        assert st["points_evaluated"] < 0.2 * st["points_total"]
        al = h.shard_align()
        half = (frames // 2) - ((frames // 2) % al)
        h.reset()
        h.sweep_shard_device(x.data_ptr(), half, None, True, False)
        a = h.peaks()
        hist = x[half - bench.BLKSIZ:half].cpu().numpy()
        h.reset()
        h.sweep_shard_device(x[half:].data_ptr(), frames - half, hist, False, True)
        b = h.peaks()
    with capi.Phaserot(n_channels=2, blksiz=bench.BLKSIZ, subsample=10, oversample=4, flags=capi.FLAG_NO_PRUNE) as h:
        h.sweep_device(x.data_ptr(), frames)
        brute = h.peaks()
    with capi.Phaserot(n_channels=2, blksiz=bench.BLKSIZ, subsample=10) as h:
        h.sweep_device(x.data_ptr(), frames)
        digital = h.peaks()
    assert np.array_equal(pruned, brute)
    assert rel(np.maximum(a, b), brute) <= 2e-6
    assert np.all(brute >= digital) and np.any(brute > digital)
    assert np.all(brute <= digital * 1.5)


def test_full_size_render_properties():
    """3 min stereo: angle 0 is a pure delay of blksiz/2; rendering is linear; +90 then the
    matching -90 rotation restores the (twice delayed) input away from DC/Nyquist effects."""
    import torch
    import bench
    x, frames = _device_programme(180.0)
    L = bench.BLKSIZ
    n_out = (frames // L + 1) * L
    y0 = torch.empty((n_out, 2), device=x.device)
    ya = torch.empty_like(y0)
    yb = torch.empty_like(y0)
    with capi.Phaserot(n_channels=2, blksiz=L) as h:
        h.render_device(x.data_ptr(), frames, [0, 0], 1, y0.data_ptr())
        h.render_device(x.data_ptr(), frames, [61, 250], 1, ya.data_ptr())
        x2 = (0.5 * x).contiguous()
        h.render_device(x2.data_ptr(), frames, [61, 250], 1, yb.data_ptr())
        torch.cuda.synchronize()
    assert torch.equal(y0[L // 2:frames + L // 2], x[:frames])        # ca = 1, sa = -0: exact delay
    assert float((ya * 0.5 - yb).abs().max()) <= 1e-6                   # linearity (power-of-two scale: near exact)
    assert float(ya.abs().max()) > 0.1


# ---------------------------------------------------------------------------
# render
# ---------------------------------------------------------------------------

@pytest.mark.parametrize("name,L,ang", [("two_sine", 8192, [37, 181]), ("pink", 8192, [180]), ("programme", 2048, [-45, 359]), ("harmonic", 16384, [90, 270, 1]),
                                         ("harmonic192", 32768, [33, 300])])
def test_render_matches_oracle(name, L, ang):
    x = {"two_sine": lambda: O.two_sine(48000, 1.3, 2), "pink": lambda: O.pink_noise(100000, 3)[:, None],
         "programme": lambda: O.programme(48000, 0.7, 2), "harmonic": lambda: O.harmonic(96000, 0.9, 3),
         "harmonic192": lambda: O.harmonic(192000, 0.8, 2)}[name]()
    yo = O.oracle_apply(x, L, ang, 1)
    scale = float(np.abs(yo).max())
    with capi.Phaserot(n_channels=x.shape[1], blksiz=L) as h:
        yg = h.render(x, ang, 1)
        assert np.max(np.abs(yg - yo)) <= AUDIO_TOL * scale
        # block streaming PhaseRotate::apply drop-in, continuing after reset
        h.reset()
        nblk = yo.shape[0] // L
        xp = np.zeros((nblk * L, x.shape[1]), np.float32)
        xp[: x.shape[0]] = x
        ys = np.concatenate([h.apply(xp[b * L:(b + 1) * L].copy(), ang) for b in range(nblk)])
        assert np.max(np.abs(ys - yo)) <= AUDIO_TOL * scale


def test_render_golden_reference_vectors(golden):
    g = golden["cli_render"]
    x, L, ang = g["x"], int(g["blksiz"]), g["angles"]
    with capi.Phaserot(n_channels=2, blksiz=L) as h:
        y = h.render(x, ang, 1)
    assert np.max(np.abs(y - g["stream"])) <= AUDIO_TOL * float(np.abs(g["stream"]).max())


# ---------------------------------------------------------------------------
# plugin: C ABI and the LV2 binary
# ---------------------------------------------------------------------------

@pytest.mark.parametrize("rate,blk,n", [(48000, 1024, 40000), (48000, 333, 20000), (44100, 64, 6000), (96000, 1024, 40000), (192000, 4096, 60000)])
def test_plugin_process_matches_oracle(rate, blk, n):
    x = O.pink_noise(n, 42)
    ncalls = (n + blk - 1) // blk
    ang = np.full(ncalls, 90.0, np.float32)
    ang[ncalls // 2:] = -135.0
    ang[-3:] = 200.0  # clamped to 180 (src:566-571)
    yo = O.oracle_plugin_run(x, rate, blk, ang)
    with capi.Phaserot(mode=capi.MODE_PLUGIN, n_channels=1, sample_rate=rate) as h:
        assert h.latency() == {44100: 1792, 48000: 1792, 96000: 2560, 192000: 5120}[rate]
        yg = np.concatenate([h.process(x[None, i * blk:(i + 1) * blk], ang[i])[0] for i in range(ncalls)])
    assert np.max(np.abs(yg - yo)) <= AUDIO_TOL * float(np.abs(yo).max())


def test_plugin_bulk_and_mixed_call_sizes():
    rate, n1, blk = 48000, 100000, 1024
    x = O.pink_noise(n1 + 10 * blk, 5)
    calls = [n1] + [blk] * 10
    angs = np.array([45.0] + [45.0] * 5 + [-90.0] * 5, np.float32)
    with capi.Phaserot(mode=capi.MODE_PLUGIN, n_channels=1, sample_rate=rate) as h:
        outs, pos = [], 0
        for k, nn in enumerate(calls):
            outs.append(h.process(x[None, pos:pos + nn], angs[k])[0])
            pos += nn
        yg = np.concatenate(outs)
    g = 32  # the oracle takes one fixed call size: emulate with the gcd, repeating each call's angle
    per = np.concatenate([np.full(nn // g, angs[k], np.float32) for k, nn in enumerate(calls)])
    yo = O.oracle_plugin_run(x, rate, g, per)
    assert np.max(np.abs(yg - yo)) <= AUDIO_TOL * float(np.abs(yo).max())
    # stereo, one bulk call, different angles per channel
    xs = np.stack([O.pink_noise(300000, 1), O.pink_noise(300000, 2)])
    with capi.Phaserot(mode=capi.MODE_PLUGIN, n_channels=2, sample_rate=96000) as h:
        yg = h.process(xs, [90.0, -30.0])
    for c, a in enumerate([90.0, -30.0]):
        yo = O.oracle_plugin_run(xs[c], 96000, 300000, np.array([a], np.float32))
        assert np.max(np.abs(yg[c] - yo)) <= AUDIO_TOL * float(np.abs(yo).max())


def test_plugin_levels_reduced_on_device():
    """phaserot_process_levels (SURVEY 8f rank 3): the meter inputs of run() come back from the device -
    max |input delayed by the latency| and max |output| of each call - for small (streaming kernel) and
    bulk (FFT path) calls alike; the audio is that of phaserot_process."""
    rng = np.random.default_rng(11)
    for nch, sizes in [(1, [1024] * 6 + [100, 7, 333]), (2, [256, 256, 40000, 1024, 20000])]:
        x = (0.3 * rng.standard_normal((nch, sum(sizes)))).astype(np.float32)
        x[0, 1500] = np.nan                      # the meters ignore NaNs (fmax)
        with capi.Phaserot(mode=capi.MODE_PLUGIN, n_channels=nch, sample_rate=48000.0) as h, \
             capi.Phaserot(mode=capi.MODE_PLUGIN, n_channels=nch, sample_rate=48000.0) as h2:
            lat = h.latency()
            xd = np.concatenate([np.zeros((nch, lat), np.float32), x], 1)   # delayed input: xd[:, t] = x[:, t - lat]
            pos = 0
            for n in sizes:
                y, li, lo = h.process_levels(x[:, pos:pos + n], 33.0)
                y2 = h2.process(x[:, pos:pos + n], 33.0)
                assert np.array_equal(y, y2, equal_nan=True)
                for c in range(nch):
                    want_in = np.nanmax(np.abs(xd[c, pos:pos + n]), initial=0.0)
                    yy = np.abs(y[c])
                    want_out = np.nanmax(yy, initial=0.0) if np.isfinite(yy).any() else 0.0
                    assert li[c] == np.float32(want_in), (nch, pos, n, c)
                    assert lo[c] == np.float32(want_out), (nch, pos, n, c)
                pos += n


def test_plugin_golden_reference_vectors(golden):
    g = golden["plugin"]
    for rate, blk in [(48000, 256), (48000, 1000), (96000, 1024), (192000, 2048)]:
        k = f"r{rate}_b{blk}"
        x, ang, yr = g[k + "_x"], g[k + "_ang"], g[k + "_y"]
        ncalls = len(ang)
        with capi.Phaserot(mode=capi.MODE_PLUGIN, n_channels=1, sample_rate=rate) as h:
            assert h.latency() == int(g[k + "_lat"])
            yg = np.concatenate([h.process(x[None, i * blk:(i + 1) * blk], ang[i])[0] for i in range(ncalls)])
        assert np.max(np.abs(yg - yr)) <= AUDIO_TOL * float(np.abs(yr).max()), k


def test_lv2_plugin_binary_through_host_harness(golden):
    """The CUDA-backed LV2 binary driven by the same minimal LV2 host as the reference plugin."""
    so = os.path.join(build.BIN_DIR, "phaserotate_cuda.so")
    assert os.path.exists(so)
    g = golden["plugin"]
    y, lat, _ = O.lv2_render(so, g["stereo_x"], 48000, 1000, g["stereo_ang"])
    assert lat == 1792
    assert np.max(np.abs(y - g["stereo_y"])) <= AUDIO_TOL * float(np.abs(g["stereo_y"]).max())
    x, ang = g["r48000_b256_x"], g["r48000_b256_ang"]
    for inplace in (False, True):
        y, lat, _ = O.lv2_render(so, x, 48000, 256, ang[:, None], inplace=inplace)
        assert np.max(np.abs(y[0] - g["r48000_b256_y"])) <= AUDIO_TOL * float(np.abs(g["r48000_b256_y"]).max())
    # a long noise render (config 2 style, shortened, last call partial) against the oracle's plugin loop
    xm = O.pink_noise(48000 * 5, 42)
    ncalls = (len(xm) + 1023) // 1024
    a90 = np.full((ncalls, 1), 90.0, np.float32)
    yg, _, _ = O.lv2_render(so, xm, 48000, 1024, a90)
    yo = O.oracle_plugin_run(xm, 48000, 1024, a90[:, 0].copy())
    assert np.max(np.abs(yg[0] - yo)) <= AUDIO_TOL * float(np.abs(yo).max())
    if O.have_ref():  # and against the reference binary itself, where it is built
        yr, _, _ = O.lv2_render(os.path.join(O.REF_DIR, "phaserotate_ref.so"), xm, 48000, 1024, a90)
        assert np.max(np.abs(yg - yr)) <= AUDIO_TOL * float(np.abs(yr).max())


# ---------------------------------------------------------------------------
# the phase-rotate CLI binary
# ---------------------------------------------------------------------------

def _cli(*argv):
    exe = os.path.join(build.BIN_DIR, "phase-rotate")
    return subprocess.run([exe] + list(argv), capture_output=True, text=True)


def test_cli_search_output_matches_reference_text(golden, tmp_path):
    g = golden["cli_text"]
    wav = str(tmp_path / "in.wav")
    O.write_wav_f32(wav, g["x"], 48000)
    for key, argv in {"default": [], "stride2": ["-s", "2"], "stride1": ["-s", "1"], "link": ["-l"], "f4096_s6": ["-f", "4096", "-s", "6"]}.items():
        r = _cli(*argv, wav)
        assert r.returncode == 0, r.stderr
        assert r.stdout == str(g[key]), key
    # verbose tables (-vv): every peak printed is the oracle's at the printed angle, within print precision
    our = _cli("-vv", "-s", "12", wav)
    assert our.returncode == 0, our.stderr
    blk = [int(l.split()[-1]) for l in our.stderr.splitlines() if l.startswith("Process block-size")]
    assert len(blk) == 1, our.stderr
    po = O.oracle_analyze(g["x"], blk[0])

    def db(p):
        return 20.0 * np.log10(p) if p >= 1e-15 else -np.inf

    rows = 0
    for line in our.stdout.splitlines():
        if line.startswith("#"):
            continue
        tok = [float(t) for t in line.split()]
        a = int(round(tok[0] * 2)) % 360
        chans = tok[2:]
        assert len(chans) == po.shape[0], line
        for c, v in enumerate(chans):
            if v != -np.inf:     # -inf: a channel the refine pass leaves out (mask)
                assert abs(v - db(po[c, a])) <= 2e-4, (line, c)
        if -np.inf not in chans:
            assert abs(tok[1] - db(po[:, a].max())) <= 2e-4, line
        rows += 1
    assert rows >= 30 + 2 * 13, our.stdout    # coarse table (every 6 deg) and at least two refine windows
    considered = 0
    for line in our.stderr.splitlines():
        if line.startswith("Consider min:"):  # "Consider min: p (< thr) chn: c @ deg deg", c counted from 0
            p, c, deg = float(line.split()[2]), int(line.split("chn:")[1].split()[0]), float(line.split("@")[1].split()[0])
            assert abs(p - po[c, int(round(deg * 2)) % 360]) <= 1e-5 * p + 1e-6, line
            considered += 1
    assert considered >= 2
    if O.have_ref():  # verbose tables: same lines, numbers within print precision
        ref = subprocess.run([os.path.join(O.REF_DIR, "phase-rotate"), "-vv", "-s", "12", wav], capture_output=True, text=True)
        assert our.stderr == ref.stderr
        assert len(our.stdout.splitlines()) == len(ref.stdout.splitlines())
        for a, b in zip(our.stdout.splitlines(), ref.stdout.splitlines()):
            if a != b:
                fa, fb = [float(t) for t in a.split()], [float(t) for t in b.split()]
                assert np.allclose(fa, fb, atol=2e-4), (a, b)


def test_sweep_pcm_is_bit_identical_to_float_sweep():
    """phaserot_sweep_pcm (SURVEY 8f rank 1): int16 / int32 PCM widened on the device gives the table of
    phaserot_sweep on the floats libsndfile would deliver (sample / 2^15, / 2^31), bit for bit; ragged
    length (not a multiple of 4 samples) and a pinned source included."""
    rng = np.random.default_rng(5)
    x = O.programme(48000, 3.0, 2)[:143999]
    q16 = np.clip(np.round(x * 32768.0), -32768, 32767).astype(np.int16)
    q24 = (np.clip(np.round(x * 8388608.0), -8388608, 8388607).astype(np.int32)) << 8      # left-justified 24 bit
    q32 = rng.integers(-2**31, 2**31 - 1, size=x.shape, dtype=np.int64).astype(np.int32) >> 2  # needs rounding to float
    with capi.Phaserot(n_channels=2, blksiz=8192) as h:
        for q, scale in [(q16, 1.0 / 32768.0), (q24, 1.0 / 2147483648.0), (q32, 1.0 / 2147483648.0)]:
            xf = (q.astype(np.float32) * np.float32(scale)).astype(np.float32)
            h.reset()
            h.sweep(xf)
            ref = h.peaks()
            h.reset()
            h.sweep_pcm(q)
            assert np.array_equal(h.peaks(), ref), q.dtype
        # pinned source: the chunks go out without the staging copy
        import ctypes
        lib = capi.load()
        p = lib.phaserot_alloc_host(q16.nbytes)
        ctypes.memmove(p, q16.ctypes.data, q16.nbytes)
        h.reset()
        h.sweep_pcm((p, q16.shape[0], np.int16))
        got = h.peaks()
        lib.phaserot_free_host(p)
        h.reset()
        h.sweep((q16.astype(np.float32) / np.float32(32768.0)).astype(np.float32))
        assert np.array_equal(got, h.peaks())
        st = h.stats()
    assert st["h2d_bytes"] > 0
    with pytest.raises(capi.PhaserotError):
        with capi.Phaserot(n_channels=2, blksiz=8192) as h:
            h._ck(h._lib.phaserot_sweep_pcm(h._h, q16.ctypes.data, 7, 10, 0, 360, 1, -1), "bad format")


def test_cli_on_pcm_files_matches_float_file(tmp_path):
    """The CLI keeps 16/24-bit PCM files integer up to the device (analysis only); its report equals
    the one for the float file holding the same sample values."""
    x = O.two_sine(48000, 2.0, 2)
    q16 = np.clip(np.round(x * 32768.0), -32768, 32767).astype(np.int16)
    q24 = np.clip(np.round(x * 8388608.0), -8388608, 8388607).astype(np.int32)
    for bits, q, scale in [(16, q16, 32768.0), (24, q24, 8388608.0)]:
        wf, wp = str(tmp_path / f"f{bits}.wav"), str(tmp_path / f"p{bits}.wav")
        O.write_wav_f32(wf, (q.astype(np.float64) / scale).astype(np.float32), 48000)
        O.write_wav_pcm(wp, q, 48000, bits)
        for argv in ([], ["-s", "1"], ["-vv", "-s", "12"]):
            a, b = _cli(*argv, wf), _cli(*argv, wp)
            assert a.returncode == 0 and b.returncode == 0, (a.stderr, b.stderr)
            assert a.stdout == b.stdout, (bits, argv)


def test_cli_render_matches_reference_files(golden, tmp_path):
    g = golden["cli_render"]
    L = int(g["blksiz"])
    for nm, sig, ang in [("stereo", g["x"], "18.5,90.5"), ("mono", g["x"][:, :1].copy(), "18.5"), ("short", g["x"][:700], "18.5,90.5"), ("exact", g["x_exact"], "18.5,90.5")]:
        wav, out = str(tmp_path / f"{nm}.wav"), str(tmp_path / f"{nm}_out.wav")
        O.write_wav_f32(wav, sig, 48000)
        r = _cli("-f", str(L), "-a", ang, wav, out)
        assert r.returncode == 0, r.stderr
        y, _ = O.read_wav_f32(out)
        yr = g["file_" + nm]
        assert y.shape == yr.shape, nm
        assert np.max(np.abs(y - yr)) <= AUDIO_TOL * max(1e-3, float(np.abs(yr).max())), nm
    # analysis + render in one go writes a file of the input's length
    wav, out = str(tmp_path / "a.wav"), str(tmp_path / "a_out.wav")
    O.write_wav_f32(wav, O.harmonic(48000, 1.0, 2), 48000)
    r = _cli("-v", wav, out)
    assert r.returncode == 0 and "# Result -- Minimize digital peak" in r.stdout
    y, _ = O.read_wav_f32(out)
    assert y.shape == (48000, 2)


def test_cli_argument_errors(tmp_path):
    wav = str(tmp_path / "x.wav")
    O.write_wav_f32(wav, O.two_sine(48000, 0.1, 2), 48000)
    for argv, msg in [(["-s", "7", wav], "Error: 180 deg is not evenly dividable by given stride.\n"),
                      (["-f", "100", wav], "Error: fft-len is out of bounds; valid range 1024..32768\n"),
                      (["-a", "10", wav], "Error: -a, --angle option requires an output file to be given.\n"),
                      ([], "Error: Missing parameter. See --help for usage information.\n"),
                      (["-a", "200", wav, str(tmp_path / "o.wav")], "Error: Invalid angle speficied, value needs to be -180 .. +180.\n")]:
        r = _cli(*argv)
        assert r.returncode == 1 and r.stderr == msg, (argv, r.stderr)
    assert _cli("--help").stdout.startswith("phase-rotate - Audio File Phase Rotation Util.")
