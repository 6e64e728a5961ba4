"""The FFT convolution on streams long enough that a CTA walks runs of segments, pinned against float64.

Short streams give every CTA of fftconv_kernel one segment, so the paths that only run inside a run - the
overlap rows a segment takes from the previous one's TMEM stash, the two-partition spectrum (L = 32768) the
CTA carries from segment to segment, the true-peak carry between contiguous launches, launches that start on
partially landed host input, and angle grids of more than one sweep tile - are compared here with the
independent float64 reference of tests/stream_ref.py:

* render: every output sample, at five (channels, FIR length) shapes, aligned and unaligned input;
* sweep: one loud burst per channel, moved over every segment boundary (every launch boundary included), so
  that the samples next to each boundary decide the table; the quiet bed elsewhere cannot;
* host input landing in several chunks, every sample format, against the device-resident sweep bit for bit;
* overs at the burst positions; peak and overs tables on grids of 2160, 2880 and 18000 angles.

Every test asserts the geometry it relies on (runs of >= 3 segments, two contiguous launches, >= 3 chunks),
so that a change of the launch geometry fails here instead of silently testing less."""
import ctypes as C

import numpy as np
import pytest
import scipy.signal as sg

import stream_ref as R
from phaserotate.lv2_b200 import build, capi
from test_gpu_overs import _schedule
from test_gpu_parity import AUDIO_TOL, PEAK_TOL, argmin_equal_unless_tied, rel
from test_truepeak_independent import ITU_PHASES

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module", autouse=True)
def _built():
    build.build_library()


@pytest.fixture(scope="module")
def n_sm():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


def _bed(n, nc, seed, peak):
    """Broadband noise (pink-ish) plus three tones per channel, scaled to `peak`."""
    rng = np.random.default_rng(seed)
    t = np.arange(n, dtype=np.float64)
    out = np.empty((n, nc), np.float32)
    for c in range(nc):
        y = sg.lfilter([0.049922035, -0.095993537, 0.050612699, -0.004408786], [1, -2.494956002, 2.017265875, -0.522189400],
                       rng.standard_normal(n))
        y /= np.abs(y).max()
        for f, ph in zip(rng.uniform(0.001, 0.1, 3), rng.uniform(0, 2 * np.pi, 3)):
            y += 0.4 * np.sin(2 * np.pi * f * t + ph)
        out[:, c] = peak * y / np.abs(y).max()
    return out


def _ragged_frames(L, nc, n_sm, min_run=3, at_least=0):
    """(F, nseg): the shortest stream of at least `at_least` segments whose one-launch pass gives every CTA a run
    of >= min_run segments, with a ragged end: F neither a multiple of L nor of 2V."""
    V2 = R.seg_samples(L)
    for nseg in range(max(at_least, min_run * (n_sm // nc)), 20 * n_sm):
        runs = R.cta_runs(nseg, nc, n_sm)
        if min(runs) < min_run:
            continue
        for F in range(nseg * V2 - 1, (nseg - 1) * V2 - 2 * L, -997):
            if R.n_segments(F, L) == nseg and F % L and F % V2:
                return F, nseg
    raise AssertionError("no stream length found")


# ---------------------------------------------------------------------------
# 1. render, every sample
# ---------------------------------------------------------------------------

# 0, 90 degrees (the Hilbert branch alone), odd grid indices, and indices outside [0, MS) that wrap
ANGLES = [0, 180, 37, 359, 541, -91, 181, 719]


@pytest.mark.parametrize("nc,L,sr", [(1, 1024, 48000), (2, 4096, 48000), (2, 8192, 48000), (3, 16384, 96000), (8, 32768, 192000)])
def test_render_every_sample(nc, L, sr, n_sm):
    import torch
    F, nseg = _ragged_frames(L, nc, n_sm)
    assert min(R.cta_runs(nseg, nc, n_sm)) >= 3 and F % L and F % R.seg_samples(L)
    x = _bed(F, nc, 100 + nc, 0.7)
    pairs = R.analytic_pair(x, L, first_block=False)
    T = len(pairs[0][0])
    sets = [[ANGLES[(c + k) % len(ANGLES)] for c in range(nc)] for k in (0, 1, 2)]
    with capi.Phaserot(n_channels=nc, blksiz=L, sample_rate=sr) as h:
        lut = h.lut()

        def check(y, ang):
            ref = R.render_ref(None, L, ang, lut=lut, pairs=pairs)
            err = np.abs(y.astype(np.float64) - ref)
            scale = float(np.abs(ref).max())
            assert err.max() <= AUDIO_TOL * scale, ang
            # the error does not grow with the segment index
            e1, e3 = err[:T // 3].max(), err[2 * T // 3:].max()
            assert e3 <= 2 * e1 + 1e-9 * scale, (ang, e1, e3)

        check(h.render(x, sets[0], 1), sets[0])
        xa = torch.from_numpy(x).cuda()
        xb = torch.zeros((F + 1) * nc, dtype=torch.float32, device="cuda")
        xb[nc:] = xa.reshape(-1)
        pb = xb.data_ptr() + 4 * nc               # one frame in: not 16 (stereo) / 8 (mono) byte aligned
        if nc <= 2:
            assert pb % (8 * nc) != 0 and xa.data_ptr() % 16 == 0
        for ang in sets[1:]:
            ya = torch.empty((T, nc), dtype=torch.float32, device="cuda")
            yb = torch.full((T, nc), float("nan"), dtype=torch.float32, device="cuda")
            h.render_device(xa.data_ptr(), F, ang, 1, ya.data_ptr())
            h.render_device(pb, F, ang, 1, yb.data_ptr())
            torch.cuda.synchronize()
            assert torch.equal(ya, yb), ang                        # the N-channel loader gives the same bits
            check(ya.cpu().numpy(), ang)


# ---------------------------------------------------------------------------
# 2. sweep with a burst at every segment boundary
# ---------------------------------------------------------------------------

BURST_LEN = 64
BURST_OFF = 4         # loudest output samples at 2 s V + 4: the interpolator's 11 samples back cross the boundary
PAD = 16              # samples before a window the true-peak interpolator reads
TP_GAIN = 1.0 + np.abs(ITU_PHASES).sum(1).max()   # a true-peak row is at most this times the largest radius


def _burst():
    n = np.arange(BURST_LEN)
    return 0.5 * np.hanning(BURST_LEN + 2)[1:-1] * np.sin(2 * np.pi * n / 4.35 + 0.3)   # tone near fs / 4.35


class Stream:
    """A quiet bed (-40 dBFS) on the device and its host mirror; one burst per channel patched in place."""

    def __init__(self, F, nc, L, seed):
        import torch
        self.F, self.nc, self.L = F, nc, L
        self.bed = _bed(F, nc, seed, 0.01)
        self.cur = self.bed.copy()
        self.dev = torch.from_numpy(self.bed).cuda()
        self.patched = []
        # the bed's largest radius over the whole stream bounds every sample outside a burst's window
        self.r_bed = max(np.hypot(xd, H).max() for xd, H in R.analytic_pair(self.bed, L, first_block=False))

    def place(self, starts):
        """starts[c]: input frame of channel c's burst (None: no burst)."""
        import torch
        for c, b0 in self.patched:
            self.cur[b0:b0 + BURST_LEN, c] = self.bed[b0:b0 + BURST_LEN, c]
            self.dev[b0:b0 + BURST_LEN, c] = torch.from_numpy(self.bed[b0:b0 + BURST_LEN, c].copy()).cuda()
        self.patched = []
        for c, b0 in enumerate(starts):
            if b0 is None:
                continue
            v = (self.bed[b0:b0 + BURST_LEN, c].astype(np.float64) + _burst()).astype(np.float32)
            self.cur[b0:b0 + BURST_LEN, c] = v
            self.dev[b0:b0 + BURST_LEN, c] = torch.from_numpy(v).cuda()
            self.patched.append((c, b0))

    def window(self, c, b0, os_):
        """Detector rows of x_d and H over the output samples a burst at b0 reaches, and of the raw input there."""
        w0, w1 = b0 - PAD, b0 + BURST_LEN + self.L + PAD
        xd, H = R.pair_window(self.cur[:, c], self.L, w0, w1)
        rx, ry = R.detector_rows(xd, os_)[:, PAD:], R.detector_rows(H, os_)[:, PAD:]
        raw = R.detector_rows(self.cur[b0 - PAD:b0 + BURST_LEN + PAD, c], os_)[:, PAD:]
        return rx, ry, np.abs(raw).max(0)

    def ref_table(self, starts, os_, lut):
        MS = len(lut[0])
        out = np.zeros((self.nc, MS))
        for c, b0 in enumerate(starts):
            rx, ry, vraw = self.window(c, b0, os_)
            px, py = rx.reshape(-1), ry.reshape(-1)
            out[c, 1:] = R.support_table(px, py, lut, np.arange(1, MS), R.hull_candidates(px, py))
            out[c, 0] = vraw.max()
            # nothing outside the window can reach the table
            bound = self.r_bed * (TP_GAIN if os_ > 1 else 1.0)
            assert bound < 0.5 * out[c].min(), (c, bound, out[c].min())
        return out


def _burst_start(s, L):
    """Input frame of a burst whose loudest output samples straddle the boundary t = 2 s V."""
    return s * R.seg_samples(L) - L // 2 + BURST_OFF - BURST_LEN // 2


def _valid_boundaries(F, L):
    T = (-(-F // L) + 1) * L
    return [s for s in range(1, R.n_segments(F, L))
            if _burst_start(s, L) - PAD >= L and _burst_start(s, L) + BURST_LEN + L + PAD <= min(T, F)]


def _groups(bounds, nc):
    """One boundary per channel per call; the last call repeats early boundaries on its spare channels."""
    k = -(-len(bounds) // nc)
    padded = list(bounds) + list(bounds[:k * nc - len(bounds)])
    return [padded[i * nc:(i + 1) * nc] for i in range(k)]


def _launches(h, os_):
    kt = h.kernel_times()
    return kt["truepeak_filter"]["launches"] // 2 if os_ > 1 else kt["fftconv_filter"]["launches"]


def _check_table(pg, ref, os_):
    assert rel(pg, ref) <= PEAK_TOL
    if os_ <= 1:
        assert np.array_equal(pg[:, 0].astype(np.float64), ref[:, 0])     # raw input peak: no arithmetic
    argmin_equal_unless_tied(pg, ref)


def _check_overs(cnt, st, starts, os_, T, lut):
    MS = len(lut[0])
    for c, b0 in enumerate(starts):
        rx, ry, vraw = st.window(c, b0, os_)
        lo, hi = R.count_overs(rx, ry, vraw, T, lut, np.arange(MS))
        assert np.all(cnt[c] >= lo) and np.all(cnt[c] <= hi), c


def _ceilings(ref):
    """Between the bursts' peak levels (a few samples over, at some angles only), and at half the lowest of them
    (dozens of samples of every burst over), both far above the bed."""
    return [float(np.float32(0.5 * (ref[:, 1:].min() + ref[:, 1:].max()))), float(np.float32(0.5 * ref.min()))]


# (channels, FIR length, rate, sampled boundaries: None = every one)
SWEEP_CONFIGS = {"stereo_L8192": (2, 8192, 48000, 48), "8ch_L32768": (8, 32768, 192000, None)}


@pytest.mark.parametrize("os_", [0, 4])
@pytest.mark.parametrize("cfg", sorted(SWEEP_CONFIGS))
def test_sweep_burst_at_every_boundary(cfg, os_, n_sm):
    nc, L, sr, n_sample = SWEEP_CONFIGS[cfg]
    sf = R.segs_first(nc, n_sm)
    F, nseg = _ragged_frames(L, nc, n_sm, at_least=2 * sf + 3)
    assert nseg > 2 * sf                      # a device sweep of true-peak makes two contiguous launches (or more)
    bounds = _valid_boundaries(F, L)
    assert sf in bounds and sf + 1 in bounds  # the boundary between the first two contiguous launches
    first_run = max(R.cta_runs(sf, nc, n_sm))
    assert first_run >= 3                     # CTAs of the contiguous launches walk runs with reused rows
    if n_sample is not None:
        rng = np.random.default_rng(7)
        forced = {bounds[0], first_run, 2 * first_run, sf - 1, sf, sf + 1, sf + first_run, bounds[-1]}
        rest = [s for s in bounds if s not in forced]
        bounds = sorted(forced | set(rng.choice(rest, n_sample - len(forced), replace=False).tolist()))
    st = Stream(F, nc, L, seed=11)
    with capi.Phaserot(n_channels=nc, blksiz=L, sample_rate=sr, oversample=os_) as h:
        lut = h.lut()
        for k, group in enumerate(_groups(bounds, nc)):
            starts = [_burst_start(s, L) for s in group]
            st.place(starts)
            h.reset()
            if k == 0:
                h.set_profiling(1)
            h.sweep_device(st.dev.data_ptr(), F)
            pg = h.peaks()
            if k == 0:
                assert _launches(h, os_) >= 3, h.kernel_times()     # bootstrap + at least two contiguous launches
                h.set_profiling(0)
            ref = st.ref_table(starts, os_, lut)
            _check_table(pg, ref, os_)
            if k % 4 == 0:
                # 4. overs at the same positions
                for T in _ceilings(ref):
                    cnt, _ = h.overs_device(st.dev.data_ptr(), F, T)
                    _check_overs(cnt, st, starts, os_, T, lut)


# ---------------------------------------------------------------------------
# 3. host input landing in several chunks
# ---------------------------------------------------------------------------

LANDING = {"stereo_4min": (2, 8192), "8ch_70s": (8, 32768)}


def _formats(x):
    """(name, payload, the floats the library converts it to)."""
    q16 = np.round(x * 32767).astype(np.int16)
    v24 = np.round(x * 8388607).astype(np.int32)
    b24 = np.ascontiguousarray(v24.astype("<i4").view(np.uint8).reshape(-1, 4)[:, :3]).reshape(-1)
    q32 = np.round(x.astype(np.float64) * 2147483647.0).astype(np.int32)
    return [("f32", x, x), ("f32_pinned", x, x),
            ("s16", q16, q16.astype(np.float32) / np.float32(32768)),
            ("s24", b24, v24.astype(np.float32) / np.float32(1 << 23)),
            ("s32", q32, q32.astype(np.float32) * np.float32(2.0 ** -31))]


@pytest.mark.parametrize("os_", [0, 4])
@pytest.mark.parametrize("cfg", sorted(LANDING))
def test_host_landing_in_chunks(cfg, os_, n_sm):
    import torch
    nc, L = LANDING[cfg]
    ch = R.chunk_frames(nc)
    F = 3 * ch + 12345
    assert -(-F // ch) >= 4 and F % L                             # three full chunks and a ragged fourth
    nseg = R.n_segments(F, L)
    assert max(R.cta_runs(min(nseg, R.segs_first(nc, n_sm)), nc, n_sm)) >= 3
    st = Stream(F, nc, L, seed=23)
    starts = [(1 + c % 3) * ch - BURST_LEN // 2 for c in range(nc)]   # bursts across chunk boundaries
    st.place(starts)
    x = st.cur
    loud = np.ascontiguousarray(4 * x[::-1])
    lib = capi.load()
    with capi.Phaserot(n_channels=nc, blksiz=L, oversample=os_) as h:
        lut = h.lut()
        ref = st.ref_table(starts, os_, lut)
        for name, payload, xf in _formats(x):
            h.reset()
            xt = torch.from_numpy(np.ascontiguousarray(xf)).cuda()
            h.sweep_device(xt.data_ptr(), F)
            want = h.peaks()
            del xt
            h.reset()
            h.sweep(loud)                    # leaves louder frames where the next stream lands
            h.peaks()
            h.reset()
            if name == "f32":
                h.sweep(payload)
            elif name == "f32_pinned":
                p = lib.phaserot_alloc_host(payload.nbytes)
                assert p
                try:
                    C.memmove(p, payload.ctypes.data, payload.nbytes)
                    h.sweep((p, F))
                    got = h.peaks()
                finally:
                    lib.phaserot_free_host(p)
            else:
                h.sweep_pcm(payload)
            if name != "f32_pinned":
                got = h.peaks()
            assert np.array_equal(got, want), name
            if name == "f32":
                _check_table(got, ref, os_)
        for T in _ceilings(ref):
            cnt, _ = h.overs(x, T)
            _check_overs(cnt, st, starts, os_, T, lut)


# ---------------------------------------------------------------------------
# 5. angle grids wider than one sweep tile
# ---------------------------------------------------------------------------

def test_wide_grids(n_sm):
    from test_gpu_parity import _device_programme
    L = 8192
    xdev, F = _device_programme(120.0)
    nseg = R.n_segments(F, L)
    assert max(R.cta_runs(nseg, 2, n_sm)) >= 3
    x = xdev.cpu().numpy()
    pairs = R.analytic_pair(x, L)
    for os_ in (0, 4):
        pts = []
        for c, (xd, H) in enumerate(pairs):
            px = R.detector_rows(xd, os_)[:, L // 2:].reshape(-1)
            py = R.detector_rows(H, os_)[:, L // 2:].reshape(-1)
            cand = R.hull_candidates(px, py)
            pts.append((px[cand], py[cand], np.abs(R.detector_rows(x[:, c], os_)).max()))
        for S in (12, 16, 100):
            MS = 180 * S
            assert MS - 1 > 2048                       # more than one tile of angles per row
            with capi.Phaserot(n_channels=2, blksiz=L, subsample=S, oversample=os_) as h:
                lut = h.lut()
                ref = np.zeros((2, MS))
                for c, (px, py, raw) in enumerate(pts):
                    ref[c, 1:] = R.support_table(px, py, lut, np.arange(1, MS))
                    ref[c, 0] = raw
                h.sweep_device(xdev.data_ptr(), F)
                _check_table(h.peaks(), ref, os_)
                T = float(np.float32(0.5 * (ref[:, 1:].min() + ref[:, 1:].max())))
                if S == 100:
                    a0, a1, stride, chn = 1000, 17000, 7, 1
                    sched = _schedule(MS, a0, a1, stride)
                    assert len(sched) > 2048
                    h.reset()
                    h.sweep_device(xdev.data_ptr(), F, a0, a1, stride, chn)
                    pg = h.peaks()
                    mask = np.zeros((2, MS), bool)
                    mask[chn, sched] = True
                    assert rel(pg[mask], ref[mask]) <= PEAK_TOL and not pg[~mask].any()
                    cnt, _ = h.overs_device(xdev.data_ptr(), F, T, a0, a1, stride, chn)
                    ang = sched
                else:
                    cnt, _ = h.overs_device(xdev.data_ptr(), F, T)
                    chn, ang = -1, np.arange(MS)
                lo, hi = R.overs_counts(x, L, T, S, os_, lut, pairs, ang)
                for c in ([0, 1] if chn < 0 else [chn]):
                    assert np.all(cnt[c, ang] >= lo[c, ang]) and np.all(cnt[c, ang] <= hi[c, ang]), (S, c)
                assert lo[:, ang].max() > 0 and hi[:, ang].min() < lo[:, ang].max()
