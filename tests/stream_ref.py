"""Float64 reference of the rotated stream and the stream geometry of the FFT convolution, for long streams.

The analytic pair of a channel is (x_d, H): x_d[t] = x[t - L/2] and H = the closed-form Hilbert FIR over x
(test_truepeak_independent.hilbert_taps), both in float64 with scipy.  The rotated output at angle a is
ca x_d + sa H.  A peak table is a maximum over that set: for a != 0 it is the support function of the symmetric
point set {+-(x_d[t], H[t])} in the direction (ca, sa), so it is evaluated over the vertices of the convex hull
of that set only (plus the points qhull found on its boundary), which makes a table of minutes of audio cost
seconds.  Nothing here calls the library or its C restatement.

The geometry follows the sizes documented in include/phaserot_cuda.h and phaserot_create: half FIR Lh = L/2,
NP = 2 tap partitions when Lh > 8192, partition length Lp = Lh / NP, V = 16384 - Lp new complex points per
segment; segment s yields the output samples [2 s V, 2 (s + 1) V).
"""
import numpy as np
import scipy.signal as sg
from scipy.spatial import ConvexHull, QhullError

from test_truepeak_independent import hilbert_taps, interpolated

# ---------------------------------------------------------------------------
# geometry
# ---------------------------------------------------------------------------


def seg_V(L):
    """New complex points per FFT segment (V = 16384 - Lp)."""
    Lh = L // 2
    NP = 2 if Lh > 8192 else 1
    return 16384 - Lh // NP


def seg_samples(L):
    """Output samples per segment: 2 V."""
    return 2 * seg_V(L)


def n_segments(F, L, flush_blocks=1):
    """Segments of a pass over F frames followed by `flush_blocks` zero blocks."""
    t_end = (-(-F // L) + flush_blocks) * L
    m_end = (t_end + 1) // 2
    return -(-m_end // seg_V(L))


def cta_runs(nseg, nchan, n_sm):
    """Segments each CTA of one fftconv_kernel launch over nseg segments per channel walks, for every CTA that
    has work: the grid is min(nseg * nchan, n_sm) CTAs, channel fastest, and the CTAs of a channel split its
    segments into contiguous runs of ceil(nseg / nb)."""
    grid = min(nseg * nchan, n_sm)
    out = []
    for b in range(grid):
        ci, jb = b % nchan, b // nchan
        nb = (grid - ci + nchan - 1) // nchan
        run = -(-nseg // nb)
        n = min(nseg, jb * run + run) - jb * run
        if n > 0:
            out.append(n)
    return out


def chunk_frames(C):
    """Frames per host upload chunk: ~32 MB of floats, a multiple of 4 frames."""
    return max(4, ((8 << 20) // C) & ~3)


def segs_first(nchan, n_sm):
    """Segments per channel of the first contiguous launch of a sweep (8 per CTA)."""
    return max(1, n_sm * 8 // nchan)


# ---------------------------------------------------------------------------
# analytic pair, render
# ---------------------------------------------------------------------------


def _chan(x):
    x = np.asarray(x)
    return x[:, None] if x.ndim == 1 else x


def analytic_pair(x, L, first_block=True, flush_blocks=1):
    """[(x_d, H)] per channel in float64 over the T = (ceil(F / L) + flush_blocks) L output samples of a pass.
    first_block: the CLI's first-block rule (x_d is zero under the first block, cli:418-419)."""
    x = _chan(x)
    F, C = x.shape
    T = (-(-F // L) + flush_blocks) * L
    taps = hilbert_taps(L)
    out = []
    for c in range(C):
        xc = np.zeros(T)
        xc[:F] = x[:, c]
        H = sg.oaconvolve(xc, taps)[:T]
        xd = np.concatenate([np.zeros(L // 2), xc])[:T]
        if first_block:
            xd[:L] = 0.0
        out.append((xd, H))
    return out


def pair_window(xc, L, t0, t1):
    """(x_d, H) of one channel (float64 input xc, the whole stream) at output samples [t0, t1), from the inputs
    they depend on only (no first-block rule)."""
    lo = max(0, t0 - L + 1)
    seg = np.asarray(xc[lo:min(len(xc), t1)], np.float64)
    H = np.zeros(t1 - t0)
    if len(seg):
        full = sg.fftconvolve(seg, hilbert_taps(L))          # full[i] is output lo + i
        a, b = t0 - lo, min(t1 - lo, len(full))
        H[:max(0, b - a)] = full[a:b]
    xd = np.zeros(t1 - t0)
    s0, s1 = max(t0 - L // 2, 0), min(t1 - L // 2, len(xc))
    if s1 > s0:
        xd[s0 + L // 2 - t0:s1 + L // 2 - t0] = xc[s0:s1]
    return xd, H


def closed_form_lut(S):
    """(sin, cos) of -a / S degrees, a = 0 .. 180 S - 1, rounded to float32 like the library's table."""
    ang = -np.arange(180 * S) * np.pi / (180 * S)
    return np.sin(ang).astype(np.float32), np.cos(ang).astype(np.float32)


def render_cs(lut, a):
    """(sa, ca) in float64 of a render angle: any grid index, wrapped to [0, MS) like the CLI (cli:463)."""
    s, c = lut
    i = int(a) % len(s)
    return float(s[i]), float(c[i])


def render_ref(x, L, angles, flush_blocks=1, lut=None, S=2, pairs=None):
    """out[t][c] = ca x_d + sa H in float64 over the T samples of the render (no first-block rule).
    pairs: analytic_pair(x, L, first_block=False, flush_blocks=flush_blocks), when already at hand."""
    lut = closed_form_lut(S) if lut is None else lut
    pairs = analytic_pair(x, L, first_block=False, flush_blocks=flush_blocks) if pairs is None else pairs
    out = np.zeros((len(pairs[0][0]), len(pairs)))
    for c, (xd, H) in enumerate(pairs):
        sa, ca = render_cs(lut, angles[c])
        out[:, c] = ca * xd + sa * H
    return out


# ---------------------------------------------------------------------------
# peak tables
# ---------------------------------------------------------------------------


def detector_rows(s, os_):
    """Rows a detector examines per sample: the sample alone (os_ <= 1) or the sample and its interpolated points."""
    s = np.asarray(s, np.float64)
    return s[None, :] if os_ <= 1 else interpolated(s, os_)


def hull_candidates(px, py, brute_below=64):
    """Indices of the points that can hold the support function of {+-(px, py)} in some direction: the hull
    vertices of the symmetric set and the points qhull found on its boundary.  Degenerate (collinear, all
    zero) or tiny sets return every index."""
    n = len(px)
    if n < brute_below:
        return np.arange(n)

    def hull_of(sel):
        pts = np.concatenate([np.stack([px[sel], py[sel]], 1), -np.stack([px[sel], py[sel]], 1)])
        try:
            return ConvexHull(pts)
        except (QhullError, ValueError):
            return None

    sel = np.arange(n)
    if n > 1 << 16:
        # Long streams: the hull of the 4096 points of largest radius contains the disc of its inradius, and so
        # does the whole hull; no point inside that disc can be on the boundary.
        r = np.hypot(px, py)
        top = np.argpartition(r, n - 4096)[n - 4096:]
        sub = hull_of(top)
        if sub is not None:
            r_in = float(np.min(-sub.equations[:, 2]))   # unit normals: distance of each edge from the origin
            sel = np.nonzero(r >= r_in * (1 - 1e-9))[0]
    hull = hull_of(sel)
    if hull is None:
        return sel
    idx = np.concatenate([hull.vertices, hull.coplanar[:, 0] if len(hull.coplanar) else np.zeros(0, int)])
    return sel[np.unique(idx % len(sel))]


def exact_candidates(px, py, lut, ang_idx):
    """Hull candidates widened so that the table over them is the brute-force table bit for bit: a point whose
    radius is below the smallest table entry (less a margin far above rounding) cannot reach any entry, since
    |ca px + sa py| <= its radius; every other point is kept.  (qhull drops points within its precision of the
    boundary, which can round a hair above a vertex.)"""
    cand = hull_candidates(px, py)
    h_min = support_table(px, py, lut, ang_idx, cand).min() if len(ang_idx) else 0.0
    r = np.hypot(px, py)
    near = np.nonzero(r >= h_min * (1 - 1e-9) if h_min > 0 else r > 0)[0]
    return np.union1d(cand, near)


def support_table(px, py, lut, ang_idx, candidates=None):
    """max_t |ca px + sa py| at each grid index of ang_idx (float64 evaluation of the float32 LUT)."""
    s, c = lut
    if candidates is not None:
        px, py = px[candidates], py[candidates]
    sa = np.asarray(s, np.float64)[ang_idx][:, None]
    ca = np.asarray(c, np.float64)[ang_idx][:, None]
    out = np.zeros(len(ang_idx))
    step = max(1, (1 << 22) // max(1, len(ang_idx)))
    for i in range(0, len(px), step):
        v = np.abs(ca * px[None, i:i + step] + sa * py[None, i:i + step]).max(1)
        out = np.maximum(out, v)
    return out


def peak_table(x, L, S=2, os_=0, lut=None, pairs=None, hull=True):
    """peak[c][a] of a sweep over x (CLI analysis: first-block rule, one flush block), float64.  Index 0 is the
    detector over the raw input blocks; a >= 1 the rotated set over the samples t >= L/2.  os_ = 2 or 4: the
    true-peak detector of include/phaserot_cuda.h.  hull=False: brute force over every point."""
    x = _chan(x)
    F, C = x.shape
    MS = 180 * S
    lut = closed_form_lut(S) if lut is None else lut
    pairs = analytic_pair(x, L) if pairs is None else pairs
    B = -(-F // L)
    out = np.zeros((C, MS))
    for c, (xd, H) in enumerate(pairs):
        px = detector_rows(xd, os_)[:, L // 2:].reshape(-1)
        py = detector_rows(H, os_)[:, L // 2:].reshape(-1)
        ang = np.arange(1, MS)
        if hull:
            out[c, 1:] = support_table(px, py, lut, ang, exact_candidates(px, py, lut, ang))
        else:
            out[c, 1:] = support_table(px, py, lut, ang)
        raw = np.zeros(B * L)
        raw[:F] = x[:, c]
        out[c, 0] = np.abs(detector_rows(raw, os_)).max() if B else 0.0
    return out


def overs_counts(x, L, T, S=2, os_=0, lut=None, pairs=None, ang_idx=None, rel=2e-6):
    """(lo, hi) per [c][a]: samples t whose detector value v = max over the sample's rows of |ca x_d + sa H|
    is above T (1 + rel), resp. above T (1 - rel).  Only samples whose largest radius reaches T (1 - rel) can
    count, so only those are evaluated."""
    x = _chan(x)
    F, C = x.shape
    MS = 180 * S
    lut = closed_form_lut(S) if lut is None else lut
    pairs = analytic_pair(x, L) if pairs is None else pairs
    ang_idx = np.arange(MS) if ang_idx is None else np.asarray(ang_idx)
    B = -(-F // L)
    lo = np.zeros((C, MS), np.int64)
    hi = np.zeros((C, MS), np.int64)
    for c, (xd, H) in enumerate(pairs):
        raw = np.zeros(B * L)
        raw[:F] = x[:, c]
        lo[c], hi[c] = count_overs(detector_rows(xd, os_)[:, L // 2:], detector_rows(H, os_)[:, L // 2:],
                                   np.abs(detector_rows(raw, os_)).max(0), T, lut, ang_idx, rel)
    return lo, hi


def count_overs(rx, ry, vraw, T, lut, ang_idx, rel=2e-6):
    """(lo, hi) [MS] of one channel: rx, ry [rows][samples] the detector rows of x_d and H, vraw the detector
    value of each raw input sample (grid index 0)."""
    s, c = (np.asarray(v, np.float64) for v in lut)
    keep = np.nonzero(np.hypot(rx, ry).max(0) > T * (1 - rel))[0]
    rx, ry = rx[:, keep], ry[:, keep]
    lo = np.zeros(len(s), np.int64)
    hi = np.zeros(len(s), np.int64)
    for a in ang_idx:
        v = vraw if a == 0 else np.abs(c[a] * rx + s[a] * ry).max(0)
        lo[a] = np.count_nonzero(v > T * (1 + rel))
        hi[a] = np.count_nonzero(v > T * (1 - rel))
    return lo, hi
