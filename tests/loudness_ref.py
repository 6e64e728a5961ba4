"""Float64 restatement of ITU-R BS.1770-4 integrated loudness, the oracle of the loudness tests.

K-weighting: the two biquads of BS.1770-4 (high shelf, then high pass) with coefficients derived for any
rate as libebur128 derives them, run with scipy's lfilter from zero state.  Gating: 100 ms sub-blocks of
floor(fs / 10 + 0.5) frames, 400 ms blocks of four sub-blocks with a hop of one (complete blocks only),
absolute gate at -70 LUFS, relative gate at -10 LU."""
import numpy as np
from scipy.signal import lfilter

# BS.1770-4 Table 1 (pre-filter, high shelf) and Table 2 (RLB, high pass) at 48 kHz: (b, a)
TABLE_48K = (
    ((1.53512485958697, -2.69169618940638, 1.19839281085285), (1.0, -1.69065929318241, 0.73248077421585)),
    ((1.0, -2.0, 1.0), (1.0, -1.99004745483398, 0.99007225036621)),
)

WEIGHTS_5_1 = (1.0, 1.0, 1.0, 0.0, 1.41, 1.41)  # WAV order L R C LFE Ls Rs


def kweight_coefs(fs):
    """[(b, a) of the shelf, (b, a) of the high pass] at sample rate fs."""
    K = np.tan(np.pi * 1681.974450955533 / fs)
    Q = 0.7071752369554196
    Vh = 10.0 ** (3.999843853973347 / 20.0)
    Vb = Vh ** 0.4996667741545416
    a0 = 1.0 + K / Q + K * K
    shelf = ((Vh + Vb * K / Q + K * K) / a0, 2.0 * (K * K - Vh) / a0, (Vh - Vb * K / Q + K * K) / a0), \
            (1.0, 2.0 * (K * K - 1.0) / a0, (1.0 - K / Q + K * K) / a0)
    K = np.tan(np.pi * 38.13547087602444 / fs)
    Q = 0.5003270373238773
    a0 = 1.0 + K / Q + K * K
    hp = (1.0, -2.0, 1.0), (1.0, 2.0 * (K * K - 1.0) / a0, (1.0 - K / Q + K * K) / a0)
    return [shelf, hp]


def kweight(x, fs):
    y = np.asarray(x, np.float64)
    for b, a in kweight_coefs(fs):
        y = lfilter(b, a, y, axis=0)
    return y


def integrated(x, fs, weights=None):
    """Integrated loudness in LUFS of x [frames] or [frames, channels]; -inf when no block passes."""
    x = np.asarray(x, np.float64)
    if x.ndim == 1:
        x = x[:, None]
    n, C = x.shape
    G = np.ones(C) if weights is None else np.asarray(weights, np.float64)
    step = int(np.floor(fs / 10.0 + 0.5))
    n_sub = n // step
    if n_sub < 4:
        return -np.inf
    y = kweight(x[:n_sub * step], fs)
    S = (y * y).reshape(n_sub, step, C).sum(1)
    z = (S[:-3] + S[1:-2] + S[2:-1] + S[3:]) / (4.0 * step)
    e = z @ G
    sel = e > 10.0 ** ((-70.0 + 0.691) / 10.0)
    if not sel.any():
        return -np.inf
    sel &= e > 0.1 * e[sel].mean()
    if not sel.any():
        return -np.inf
    return -0.691 + 10.0 * np.log10(e[sel].mean())


def sine_segments(fs, parts, freq=1000.0, channels=2):
    """EBU Tech 3341 test signals: a 1 kHz sine in consecutive segments [(seconds, dBFS peak), ...] on every channel."""
    out = []
    t0 = 0
    for sec, db in parts:
        n = int(round(sec * fs))
        t = (np.arange(n) + t0) / fs
        out.append(10.0 ** (db / 20.0) * np.sin(2 * np.pi * freq * t))
        t0 += n
    y = np.concatenate(out)
    return np.repeat(y[:, None], channels, 1).astype(np.float32)


TECH3341 = {
    1: [(20.0, -23.0)],
    2: [(20.0, -33.0)],
    3: [(10.0, -36.0), (60.0, -23.0), (10.0, -36.0)],
    4: [(10.0, -72.0), (10.0, -36.0), (60.0, -23.0), (10.0, -36.0), (10.0, -72.0)],
    5: [(20.0, -26.0), (20.1, -20.0), (20.0, -26.0)],
}
TECH3341_EXPECTED = {1: -23.0, 2: -33.0, 3: -23.0, 4: -23.0, 5: -23.0}
