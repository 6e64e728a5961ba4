"""ctypes binding of libphaserot_cuda (include/phaserot_cuda.h).

This is plumbing for tests and bench.py: it forwards to the C ABI and never
computes audio itself.  If the library is missing or no sm_100 GPU is present
every entry point fails loudly (PhaserotError) — there is no CPU fallback.
"""
import ctypes as C
import os

import numpy as np

from . import build as _build

OK = 0
E_INVAL, E_NO_DEVICE, E_CUDA, E_NOMEM, E_UNSUPPORTED, E_STATE, E_AGAIN = -1, -2, -3, -4, -5, -6, -7
MODE_CLI, MODE_PLUGIN = 0, 1
FLAG_NO_FIRST_BLOCK_QUIRK = 1
FLAG_NO_PRUNE = 2
PCM_F32, PCM_S16, PCM_S32, PCM_S24 = 0, 1, 2, 3
ABI_VERSION = 4

SYMBOLS = [
    "phaserot_create", "phaserot_destroy", "phaserot_reset", "phaserot_set_stream",
    "phaserot_sweep", "phaserot_sweep_pcm", "phaserot_sweep_device", "phaserot_analyze", "phaserot_peak", "phaserot_peaks", "phaserot_lut",
    "phaserot_apply", "phaserot_render", "phaserot_render_device",
    "phaserot_process", "phaserot_process_levels", "phaserot_latency",
    "phaserot_sweep_shard_device", "phaserot_sweep_shard", "phaserot_shard_align", "phaserot_plugin_angle",
    "phaserot_sweep_shard_boot_device", "phaserot_sweep_shard_resume",
    "phaserot_sweep_sections", "phaserot_sweep_sections_device", "phaserot_section_peaks",
    "phaserot_render_sections", "phaserot_render_sections_device",
    "phaserot_loudness", "phaserot_loudness_device", "phaserot_overs", "phaserot_overs_device",
    "phaserot_nth_peaks", "phaserot_nth_peaks_device",
    "phaserot_group_create", "phaserot_group_destroy", "phaserot_group_size", "phaserot_group_handle", "phaserot_group_sweep",
    "phaserot_group_peaks", "phaserot_group_reset", "phaserot_pending_table", "phaserot_set_profiling", "phaserot_get_kernel_times",
    "phaserot_sync", "phaserot_get_stats", "phaserot_reset_stats",
    "phaserot_alloc_host", "phaserot_free_host",
    "phaserot_strerror", "phaserot_last_error", "phaserot_abi_version",
]


class Cfg(C.Structure):
    _fields_ = [
        ("abi_version", C.c_uint32), ("mode", C.c_int32), ("n_channels", C.c_int32), ("blksiz", C.c_int32),
        ("sample_rate", C.c_double), ("subsample", C.c_int32), ("device", C.c_int32), ("flags", C.c_uint32),
        ("oversample", C.c_int32),
    ]


class Stats(C.Structure):
    _fields_ = [("kernel_launches", C.c_uint64), ("points_total", C.c_uint64), ("points_evaluated", C.c_uint64),
                ("h2d_bytes", C.c_uint64), ("d2h_bytes", C.c_uint64), ("dense_repeats", C.c_uint64)]


NKERNELS = 7
KERNEL_NAMES = ["fftconv_filter", "sweep", "deinterleave", "fftconv_render", "fir_stream", "other", "truepeak_filter"]


class KTimes(C.Structure):
    _fields_ = [("ms", C.c_double * NKERNELS), ("launches", C.c_uint64 * NKERNELS)]


class PhaserotError(RuntimeError):
    def __init__(self, code, what, detail=""):
        self.code = code
        super().__init__(f"{what}: {code} ({detail})")


_lib = None


def lib_path():
    return _build.LIB


def load():
    """Load (building first if the sources are newer) libphaserot_cuda.so."""
    global _lib
    if _lib is not None:
        return _lib
    path = os.environ.get("PHASEROT_LIB") or _build.LIB  # PHASEROT_LIB: A/B runs of two builds (tools/ab_kernel.sh)
    if not os.path.exists(path):
        _build.build_library()
    lib = C.CDLL(path)
    vp, fp, ip = C.c_void_p, C.POINTER(C.c_float), C.POINTER(C.c_int)
    lib.phaserot_create.argtypes = [C.POINTER(vp), C.POINTER(Cfg)]
    lib.phaserot_destroy.argtypes = [vp]
    lib.phaserot_destroy.restype = None
    lib.phaserot_reset.argtypes = [vp]
    lib.phaserot_set_stream.argtypes = [vp, vp]
    lib.phaserot_sweep.argtypes = [vp, vp, C.c_uint64, C.c_int, C.c_int, C.c_int, C.c_int]
    lib.phaserot_sweep_pcm.argtypes = [vp, vp, C.c_int, C.c_uint64, C.c_int, C.c_int, C.c_int, C.c_int]
    lib.phaserot_sweep_device.argtypes = [vp, vp, C.c_uint64, C.c_int, C.c_int, C.c_int, C.c_int]
    lib.phaserot_analyze.argtypes = [vp, vp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int]
    lib.phaserot_peak.argtypes = [vp, C.c_int, C.c_int]
    lib.phaserot_peak.restype = C.c_float
    lib.phaserot_peaks.argtypes = [vp, vp]
    lib.phaserot_lut.argtypes = [vp, vp, vp]
    lib.phaserot_apply.argtypes = [vp, vp, vp]
    lib.phaserot_render.argtypes = [vp, vp, C.c_uint64, vp, C.c_int, vp]
    lib.phaserot_render_device.argtypes = [vp, vp, C.c_uint64, vp, C.c_int, vp]
    lib.phaserot_process.argtypes = [vp, C.POINTER(vp), C.POINTER(vp), C.c_uint32, vp]
    lib.phaserot_process_levels.argtypes = [vp, C.POINTER(vp), C.POINTER(vp), C.c_uint32, vp, vp, vp]
    lib.phaserot_latency.argtypes = [vp]
    lib.phaserot_latency.restype = C.c_uint32
    lib.phaserot_sweep_shard_device.argtypes = [vp, vp, C.c_uint64, vp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int]
    lib.phaserot_sweep_shard.argtypes = [vp, vp, C.c_int, C.c_uint64, vp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int]
    lib.phaserot_plugin_angle.argtypes = [vp, vp]
    lib.phaserot_sweep_shard_boot_device.argtypes = [vp, vp, C.c_uint64, vp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int]
    lib.phaserot_sweep_shard_resume.argtypes = [vp]
    lib.phaserot_sweep_sections.argtypes = [vp, vp, C.c_int, C.c_uint64, C.c_uint64, C.c_int, C.c_int, C.c_int, C.c_int]
    lib.phaserot_sweep_sections_device.argtypes = [vp, vp, C.c_uint64, C.c_uint64, C.c_int, C.c_int, C.c_int, C.c_int]
    lib.phaserot_section_peaks.argtypes = [vp, C.POINTER(C.c_int), vp]
    lib.phaserot_render_sections.argtypes = [vp, vp, C.c_uint64, C.c_uint64, vp, C.c_int, vp]
    lib.phaserot_render_sections_device.argtypes = [vp, vp, C.c_uint64, C.c_uint64, vp, C.c_int, vp]
    lib.phaserot_loudness.argtypes = [vp, vp, C.c_int, C.c_uint64, C.c_double, vp, vp, C.c_int, vp]
    lib.phaserot_loudness_device.argtypes = [vp, vp, C.c_uint64, C.c_double, vp, vp, C.c_int, vp]
    lib.phaserot_overs.argtypes = [vp, vp, C.c_int, C.c_uint64, C.c_float, C.c_int, C.c_int, C.c_int, C.c_int, vp, vp]
    lib.phaserot_overs_device.argtypes = [vp, vp, C.c_uint64, C.c_float, C.c_int, C.c_int, C.c_int, C.c_int, vp, vp]
    lib.phaserot_nth_peaks.argtypes = [vp, vp, C.c_int, C.c_uint64, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, vp]
    lib.phaserot_nth_peaks_device.argtypes = [vp, vp, C.c_uint64, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, vp]
    lib.phaserot_group_create.argtypes = [C.POINTER(vp), C.POINTER(Cfg), vp, C.c_int]
    lib.phaserot_group_destroy.argtypes = [vp]
    lib.phaserot_group_destroy.restype = None
    lib.phaserot_group_size.argtypes = [vp]
    lib.phaserot_group_handle.argtypes = [vp, C.c_int]
    lib.phaserot_group_handle.restype = vp
    lib.phaserot_group_sweep.argtypes = [vp, vp, C.c_int, C.c_uint64, C.c_int, C.c_int, C.c_int, C.c_int]
    lib.phaserot_group_peaks.argtypes = [vp, vp]
    lib.phaserot_group_reset.argtypes = [vp]
    lib.phaserot_shard_align.argtypes = [vp]
    lib.phaserot_pending_table.argtypes = [vp, C.POINTER(C.POINTER(C.c_float)), C.POINTER(C.c_int), C.POINTER(C.c_int)]
    lib.phaserot_shard_align.restype = C.c_uint32
    lib.phaserot_set_profiling.argtypes = [vp, C.c_int]
    lib.phaserot_get_kernel_times.argtypes = [vp, C.POINTER(KTimes)]
    lib.phaserot_sync.argtypes = [vp]
    lib.phaserot_get_stats.argtypes = [vp, C.POINTER(Stats)]
    lib.phaserot_reset_stats.argtypes = [vp]
    lib.phaserot_alloc_host.argtypes = [C.c_uint64]
    lib.phaserot_alloc_host.restype = C.c_void_p
    lib.phaserot_free_host.argtypes = [vp]
    lib.phaserot_free_host.restype = None
    lib.phaserot_strerror.argtypes = [C.c_int]
    lib.phaserot_strerror.restype = C.c_char_p
    lib.phaserot_last_error.restype = C.c_char_p
    lib.phaserot_abi_version.restype = C.c_int
    _lib = lib
    return lib


def _ptr(a):
    return a.ctypes.data_as(C.c_void_p)


class Phaserot:
    """Thin RAII wrapper: one libphaserot_cuda handle."""

    def __init__(self, mode=MODE_CLI, n_channels=1, blksiz=8192, sample_rate=48000.0, subsample=2, device=-1, flags=0, oversample=0):
        self._lib = load()
        self._h = C.c_void_p()
        self.n_channels, self.blksiz, self.subsample, self.mode = n_channels, blksiz, subsample or 2, mode
        self.maxsample = 180 * self.subsample
        cfg = Cfg(ABI_VERSION, mode, n_channels, blksiz, float(sample_rate), subsample, device, flags, oversample)
        rc = self._lib.phaserot_create(C.byref(self._h), C.byref(cfg))
        if rc != OK:
            self._h = C.c_void_p()
            raise PhaserotError(rc, "phaserot_create", self._detail(rc))

    def _detail(self, rc):
        return self._lib.phaserot_strerror(rc).decode() + "; " + self._lib.phaserot_last_error().decode()

    def _ck(self, rc, what):
        if rc != OK:
            raise PhaserotError(rc, what, self._detail(rc))

    def close(self):
        if self._h:
            self._lib.phaserot_destroy(self._h)
            self._h = C.c_void_p()

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # -- CLI analysis ------------------------------------------------------
    def reset(self):
        self._ck(self._lib.phaserot_reset(self._h), "phaserot_reset")

    def set_stream(self, stream_ptr):
        self._ck(self._lib.phaserot_set_stream(self._h, C.c_void_p(stream_ptr)), "phaserot_set_stream")

    def sweep(self, x, ang_start=0, ang_end=None, stride=1, chn=-1):
        """x: host array [frames, channels] float32 (C-contiguous) or a raw host pointer tuple (ptr, frames)."""
        if ang_end is None:
            ang_end = self.maxsample
        if isinstance(x, tuple):
            ptr, n = x
        else:
            x = np.ascontiguousarray(x, np.float32).reshape(-1, self.n_channels)
            ptr, n = x.ctypes.data, x.shape[0]
        self._ck(self._lib.phaserot_sweep(self._h, C.c_void_p(ptr), n, ang_start, ang_end, stride, chn), "phaserot_sweep")

    def sweep_pcm(self, pcm, ang_start=0, ang_end=None, stride=1, chn=-1):
        """pcm: int16 / int32 array [frames, channels], or (host pointer, n_frames, numpy dtype)."""
        if ang_end is None:
            ang_end = self.maxsample
        if isinstance(pcm, tuple):
            ptr, n_frames, dt = C.c_void_p(pcm[0]), pcm[1], np.dtype(pcm[2])
        else:
            pcm = np.ascontiguousarray(pcm)
            assert pcm.size % self.n_channels == 0
            ptr, n_frames, dt = _ptr(pcm), pcm.size // self.n_channels, pcm.dtype
        fmt = {np.dtype(np.int16): PCM_S16, np.dtype(np.int32): PCM_S32, np.dtype(np.uint8): PCM_S24}[dt]
        if fmt == PCM_S24 and not isinstance(pcm, tuple):
            n_frames //= 3  # packed 24-bit: uint8 array of 3 bytes per sample
        self._ck(self._lib.phaserot_sweep_pcm(self._h, ptr, fmt, n_frames, ang_start, ang_end, stride, chn), "phaserot_sweep_pcm")

    def sweep_shard(self, data, n_frames, hist, first, last, fmt=PCM_F32, ang_start=0, ang_end=None, stride=1, chn=-1):
        """Host-memory shard (phaserot_sweep_shard): data = numpy array or raw host pointer; hist like sweep_shard_device."""
        if ang_end is None:
            ang_end = self.maxsample
        dp = C.c_void_p(data) if isinstance(data, int) else _ptr(data)
        hp = None
        if isinstance(hist, int):
            hp = C.c_void_p(hist)
        elif hist is not None:
            hist = np.ascontiguousarray(hist, np.float32)
            assert hist.size == self.blksiz * self.n_channels
            hp = _ptr(hist)
        self._ck(self._lib.phaserot_sweep_shard(self._h, dp, fmt, n_frames, hp, int(first), int(last), ang_start, ang_end, stride, chn),
                 "phaserot_sweep_shard")

    def plugin_angle(self):
        out = np.zeros(self.n_channels, np.float32)
        self._ck(self._lib.phaserot_plugin_angle(self._h, _ptr(out)), "phaserot_plugin_angle")
        return out

    def sweep_device(self, dev_ptr, n_frames, ang_start=0, ang_end=None, stride=1, chn=-1):
        if ang_end is None:
            ang_end = self.maxsample
        self._ck(self._lib.phaserot_sweep_device(self._h, C.c_void_p(dev_ptr), n_frames, ang_start, ang_end, stride, chn), "phaserot_sweep_device")

    def sweep_shard_device(self, dev_ptr, n_frames, hist, first, last, ang_start=0, ang_end=None, stride=1, chn=-1):
        """hist: host array [blksiz, channels] float32, an int (device pointer to the same) or None."""
        if ang_end is None:
            ang_end = self.maxsample
        hp = None
        if isinstance(hist, int):
            hp = C.c_void_p(hist)
        elif hist is not None:
            hist = np.ascontiguousarray(hist, np.float32)
            assert hist.size == self.blksiz * self.n_channels
            hp = _ptr(hist)
        self._ck(self._lib.phaserot_sweep_shard_device(self._h, C.c_void_p(dev_ptr), n_frames, hp, int(first), int(last),
                                                       ang_start, ang_end, stride, chn), "phaserot_sweep_shard_device")

    def sweep_shard_boot_device(self, dev_ptr, n_frames, hist, first, last, ang_start=0, ang_end=None, stride=1, chn=-1):
        """Phase 1 of the two-phase sharded sweep: the bootstrap wave only (hist like sweep_shard_device)."""
        if ang_end is None:
            ang_end = self.maxsample
        hp = None
        if isinstance(hist, int):
            hp = C.c_void_p(hist)
        elif hist is not None:
            hist = np.ascontiguousarray(hist, np.float32)
            hp = _ptr(hist)
        self._ck(self._lib.phaserot_sweep_shard_boot_device(self._h, C.c_void_p(dev_ptr), n_frames, hp, int(first), int(last),
                                                            ang_start, ang_end, stride, chn), "phaserot_sweep_shard_boot_device")

    def sweep_shard_resume(self):
        """Phase 2: the contiguous passes on top of the (combined) pending table."""
        self._ck(self._lib.phaserot_sweep_shard_resume(self._h), "phaserot_sweep_shard_resume")

    def pending_table(self):
        """(device pointer, n_channels, n_angles) of the pending sweep's table: n_channels * n_angles + n_channels + 1 floats
        (maxima, raw peaks, the library's overflow flag: reduce ALL of them; peaks() raising E_AGAIN means: combine once more)."""
        p, nc, na = C.POINTER(C.c_float)(), C.c_int(), C.c_int()
        self._ck(self._lib.phaserot_pending_table(self._h, C.byref(p), C.byref(nc), C.byref(na)), "phaserot_pending_table")
        return C.cast(p, C.c_void_p).value, nc.value, na.value

    def shard_align(self):
        return int(self._lib.phaserot_shard_align(self._h))

    def set_profiling(self, on):
        self._ck(self._lib.phaserot_set_profiling(self._h, int(on)), "phaserot_set_profiling")

    def kernel_times(self):
        k = KTimes()
        self._ck(self._lib.phaserot_get_kernel_times(self._h, C.byref(k)), "phaserot_get_kernel_times")
        return {KERNEL_NAMES[i]: {"ms": float(k.ms[i]), "launches": int(k.launches[i])} for i in range(NKERNELS)}

    def analyze(self, block, ang_start=0, ang_end=180, stride=1, chn=-1, start=False):
        block = np.ascontiguousarray(block, np.float32)
        assert block.size == self.blksiz * self.n_channels
        self._ck(self._lib.phaserot_analyze(self._h, _ptr(block), ang_start, ang_end, stride, chn, int(start)), "phaserot_analyze")

    def peak(self, c, a):
        return float(self._lib.phaserot_peak(self._h, c, a))

    def peaks(self):
        out = np.zeros((self.n_channels, self.maxsample), np.float32)
        self._ck(self._lib.phaserot_peaks(self._h, _ptr(out)), "phaserot_peaks")
        return out

    def lut(self):
        s = np.zeros(self.maxsample, np.float32)
        c = np.zeros(self.maxsample, np.float32)
        self._ck(self._lib.phaserot_lut(self._h, _ptr(s), _ptr(c)), "phaserot_lut")
        return s, c

    def sync(self):
        self._ck(self._lib.phaserot_sync(self._h), "phaserot_sync")

    # -- per-section analysis and render ------------------------------------
    def sweep_sections(self, x, section_frames, ang_start=0, ang_end=None, stride=1, chn=-1):
        """x: host array [frames, channels] of float32, int16 or int32 (PCM_S32), or packed 24-bit uint8 bytes."""
        if ang_end is None:
            ang_end = self.maxsample
        x = np.ascontiguousarray(x)
        fmt = {np.dtype(np.float32): PCM_F32, np.dtype(np.int16): PCM_S16, np.dtype(np.int32): PCM_S32, np.dtype(np.uint8): PCM_S24}[x.dtype]
        n = x.size // self.n_channels // (3 if fmt == PCM_S24 else 1)
        self._ck(self._lib.phaserot_sweep_sections(self._h, _ptr(x), fmt, n, section_frames, ang_start, ang_end, stride, chn),
                 "phaserot_sweep_sections")

    def sweep_sections_device(self, dev_ptr, n_frames, section_frames, ang_start=0, ang_end=None, stride=1, chn=-1):
        if ang_end is None:
            ang_end = self.maxsample
        self._ck(self._lib.phaserot_sweep_sections_device(self._h, C.c_void_p(dev_ptr), n_frames, section_frames, ang_start, ang_end, stride, chn),
                 "phaserot_sweep_sections_device")

    def section_peaks(self):
        """Tables of the last sections sweep: [n_sections, channels, 180 * subsample]."""
        n = C.c_int()
        self._ck(self._lib.phaserot_section_peaks(self._h, C.byref(n), None), "phaserot_section_peaks")
        out = np.zeros((n.value, self.n_channels, self.maxsample), np.float32)
        self._ck(self._lib.phaserot_section_peaks(self._h, C.byref(n), _ptr(out)), "phaserot_section_peaks")
        return out

    def render_sections(self, x, section_frames, angles, flush_blocks=1):
        """angles: [n_sections, channels] grid steps on the full circle."""
        x = np.ascontiguousarray(x, np.float32).reshape(-1, self.n_channels)
        n = x.shape[0]
        nblk = (n + self.blksiz - 1) // self.blksiz + flush_blocks
        out = np.zeros((nblk * self.blksiz, self.n_channels), np.float32)
        ang = np.ascontiguousarray(angles, np.int32)
        self._ck(self._lib.phaserot_render_sections(self._h, _ptr(x), n, section_frames, _ptr(ang), flush_blocks, _ptr(out)),
                 "phaserot_render_sections")
        return out

    def render_sections_device(self, d_in, n_frames, section_frames, angles, flush_blocks, d_out):
        ang = np.ascontiguousarray(angles, np.int32)
        self._ck(self._lib.phaserot_render_sections_device(self._h, C.c_void_p(d_in), n_frames, section_frames, _ptr(ang), flush_blocks,
                                                           C.c_void_p(d_out)), "phaserot_render_sections_device")

    # -- integrated loudness -------------------------------------------------
    def _loudness_args(self, angle_sets, weights):
        ang = np.ascontiguousarray(angle_sets, np.int32).reshape(-1, self.n_channels)
        w = None if weights is None else np.ascontiguousarray(weights, np.float32).reshape(self.n_channels)
        return ang, w, np.zeros(ang.shape[0], np.float64)

    def loudness(self, x, angle_sets, sample_rate, weights=None):
        """BS.1770-4 integrated loudness (LUFS) of the trimmed render at each angle set.
        x: host array [frames, channels] of float32, int16 or int32 (PCM_S32), or packed 24-bit uint8 bytes;
        angle_sets: [n_sets, channels] grid steps on the full circle; weights: [channels] or None (1.0)."""
        x = np.ascontiguousarray(x)
        fmt = {np.dtype(np.float32): PCM_F32, np.dtype(np.int16): PCM_S16, np.dtype(np.int32): PCM_S32, np.dtype(np.uint8): PCM_S24}[x.dtype]
        n = x.size // self.n_channels // (3 if fmt == PCM_S24 else 1)
        ang, w, out = self._loudness_args(angle_sets, weights)
        self._ck(self._lib.phaserot_loudness(self._h, _ptr(x), fmt, n, float(sample_rate), None if w is None else _ptr(w), _ptr(ang),
                                             ang.shape[0], _ptr(out)), "phaserot_loudness")
        return out

    def loudness_device(self, ptr, n_frames, angle_sets, sample_rate, weights=None):
        """The same over interleaved float32 audio in device memory."""
        ang, w, out = self._loudness_args(angle_sets, weights)
        self._ck(self._lib.phaserot_loudness_device(self._h, C.c_void_p(ptr), n_frames, float(sample_rate), None if w is None else _ptr(w),
                                                    _ptr(ang), ang.shape[0], _ptr(out)), "phaserot_loudness_device")
        return out

    # -- overs above a ceiling ---------------------------------------------------
    def _overs_out(self):
        return np.zeros((self.n_channels, self.maxsample), np.uint64), np.zeros((self.n_channels, self.maxsample), np.float64)

    def overs(self, x, ceiling, ang_start=0, ang_end=None, ang_stride=1, chn=-1):
        """Per-angle count and excess of the samples above `ceiling` (linear): (counts uint64 [C][MS], excess float64 [C][MS]).
        x: host array [frames, channels] of float32, int16 or int32 (PCM_S32), or packed 24-bit uint8 bytes."""
        if ang_end is None:
            ang_end = self.maxsample
        x = np.ascontiguousarray(x)
        fmt = {np.dtype(np.float32): PCM_F32, np.dtype(np.int16): PCM_S16, np.dtype(np.int32): PCM_S32, np.dtype(np.uint8): PCM_S24}[x.dtype]
        n = x.size // self.n_channels // (3 if fmt == PCM_S24 else 1)
        counts, excess = self._overs_out()
        self._ck(self._lib.phaserot_overs(self._h, _ptr(x), fmt, n, float(ceiling), ang_start, ang_end, ang_stride, chn, _ptr(counts), _ptr(excess)),
                 "phaserot_overs")
        return counts, excess

    def overs_device(self, ptr, n_frames, ceiling, ang_start=0, ang_end=None, ang_stride=1, chn=-1):
        """The same over interleaved float32 audio in device memory."""
        if ang_end is None:
            ang_end = self.maxsample
        counts, excess = self._overs_out()
        self._ck(self._lib.phaserot_overs_device(self._h, C.c_void_p(ptr), n_frames, float(ceiling), ang_start, ang_end, ang_stride, chn, _ptr(counts),
                                                 _ptr(excess)), "phaserot_overs_device")
        return counts, excess

    # -- rank table ------------------------------------------------------------
    def nth_peaks(self, x, n_rank, ang_start=0, ang_end=None, ang_stride=1, chn=-1):
        """The n_rank largest values of the rotated output at every angle: float32 [C][MS][n_rank], each row non-increasing.
        x: host array [frames, channels] of float32, int16 or int32 (PCM_S32), or packed 24-bit uint8 bytes."""
        if ang_end is None:
            ang_end = self.maxsample
        x = np.ascontiguousarray(x)
        fmt = {np.dtype(np.float32): PCM_F32, np.dtype(np.int16): PCM_S16, np.dtype(np.int32): PCM_S32, np.dtype(np.uint8): PCM_S24}[x.dtype]
        n = x.size // self.n_channels // (3 if fmt == PCM_S24 else 1)
        out = np.zeros((self.n_channels, self.maxsample, max(int(n_rank), 1)), np.float32)
        self._ck(self._lib.phaserot_nth_peaks(self._h, _ptr(x), fmt, n, int(n_rank), ang_start, ang_end, ang_stride, chn, _ptr(out)),
                 "phaserot_nth_peaks")
        return out

    def nth_peaks_device(self, ptr, n_frames, n_rank, ang_start=0, ang_end=None, ang_stride=1, chn=-1):
        """The same over interleaved float32 audio in device memory."""
        if ang_end is None:
            ang_end = self.maxsample
        out = np.zeros((self.n_channels, self.maxsample, max(int(n_rank), 1)), np.float32)
        self._ck(self._lib.phaserot_nth_peaks_device(self._h, C.c_void_p(ptr), n_frames, int(n_rank), ang_start, ang_end, ang_stride, chn, _ptr(out)),
                 "phaserot_nth_peaks_device")
        return out

    # -- CLI render --------------------------------------------------------
    def apply(self, buf, angles):
        buf = np.ascontiguousarray(buf, np.float32)
        ang = np.ascontiguousarray(angles, np.int32)
        self._ck(self._lib.phaserot_apply(self._h, _ptr(buf), _ptr(ang)), "phaserot_apply")
        return buf

    def render(self, x, angles, flush_blocks=1):
        x = np.ascontiguousarray(x, np.float32).reshape(-1, self.n_channels)
        n = x.shape[0]
        nblk = (n + self.blksiz - 1) // self.blksiz + flush_blocks
        out = np.zeros((nblk * self.blksiz, self.n_channels), np.float32)
        ang = np.ascontiguousarray(angles, np.int32)
        self._ck(self._lib.phaserot_render(self._h, _ptr(x), n, _ptr(ang), flush_blocks, _ptr(out)), "phaserot_render")
        return out

    def render_device(self, d_in, n_frames, angles, flush_blocks, d_out):
        ang = np.ascontiguousarray(angles, np.int32)
        self._ck(self._lib.phaserot_render_device(self._h, C.c_void_p(d_in), n_frames, _ptr(ang), flush_blocks, C.c_void_p(d_out)), "phaserot_render_device")

    # -- plugin ------------------------------------------------------------
    def process(self, x_planar, angle_deg):
        """x_planar: [channels, n] float32; returns output of the same shape."""
        x = np.ascontiguousarray(x_planar, np.float32).reshape(self.n_channels, -1)
        out = np.zeros_like(x)
        n = x.shape[1]
        ins = (C.c_void_p * self.n_channels)(*[x[c].ctypes.data for c in range(self.n_channels)])
        outs = (C.c_void_p * self.n_channels)(*[out[c].ctypes.data for c in range(self.n_channels)])
        ang = np.ascontiguousarray(np.broadcast_to(np.asarray(angle_deg, np.float32), (self.n_channels,)))
        self._ck(self._lib.phaserot_process(self._h, ins, outs, n, _ptr(ang)), "phaserot_process")
        return out

    def process_levels(self, x_planar, angle_deg):
        """Like process(); returns (output, level_in[channels], level_out[channels])."""
        x = np.ascontiguousarray(x_planar, np.float32).reshape(self.n_channels, -1)
        out = np.zeros_like(x)
        n = x.shape[1]
        ins = (C.c_void_p * self.n_channels)(*[x[c].ctypes.data for c in range(self.n_channels)])
        outs = (C.c_void_p * self.n_channels)(*[out[c].ctypes.data for c in range(self.n_channels)])
        ang = np.ascontiguousarray(np.broadcast_to(np.asarray(angle_deg, np.float32), (self.n_channels,)))
        li = np.zeros(self.n_channels, np.float32)
        lo = np.zeros(self.n_channels, np.float32)
        self._ck(self._lib.phaserot_process_levels(self._h, ins, outs, n, _ptr(ang), _ptr(li), _ptr(lo)), "phaserot_process_levels")
        return out, li, lo

    def process_raw(self, in_ptrs, out_ptrs, n, ang):
        self._ck(self._lib.phaserot_process(self._h, in_ptrs, out_ptrs, n, _ptr(ang)), "phaserot_process")

    def latency(self):
        return int(self._lib.phaserot_latency(self._h))

    def stats(self):
        s = Stats()
        self._ck(self._lib.phaserot_get_stats(self._h, C.byref(s)), "phaserot_get_stats")
        return {k: int(getattr(s, k)) for k, _ in Stats._fields_}

    def reset_stats(self):
        self._ck(self._lib.phaserot_reset_stats(self._h), "phaserot_reset_stats")


class PhaserotGroup:
    """One stream analysed by several devices of this process (phaserot_group_*)."""

    def __init__(self, n_devices, devices=None, n_channels=1, blksiz=8192, subsample=2, flags=0, oversample=0):
        self._lib = load()
        self._g = C.c_void_p()
        self.n_channels, self.blksiz, self.subsample = n_channels, blksiz, subsample or 2
        self.maxsample = 180 * self.subsample
        cfg = Cfg(ABI_VERSION, MODE_CLI, n_channels, blksiz, 48000.0, subsample, -1, flags, oversample)
        dv = None
        if devices is not None:
            self._dev = np.ascontiguousarray(devices, np.int32)
            dv = _ptr(self._dev)
        rc = self._lib.phaserot_group_create(C.byref(self._g), C.byref(cfg), dv, n_devices)
        if rc != OK:
            self._g = C.c_void_p()
            raise PhaserotError(rc, "phaserot_group_create", self._lib.phaserot_strerror(rc).decode() + "; " + self._lib.phaserot_last_error().decode())

    def _ck(self, rc, what):
        if rc != OK:
            raise PhaserotError(rc, what, self._lib.phaserot_strerror(rc).decode() + "; " + self._lib.phaserot_last_error().decode())

    def size(self):
        return int(self._lib.phaserot_group_size(self._g))

    def sweep(self, data, n_frames=None, fmt=PCM_F32, ang_start=0, ang_end=None, stride=1, chn=-1):
        if ang_end is None:
            ang_end = self.maxsample
        if isinstance(data, int):
            dp = C.c_void_p(data)
        else:
            data = np.ascontiguousarray(data)
            dp = _ptr(data)
            if n_frames is None:
                n_frames = data.size // self.n_channels // (3 if fmt == PCM_S24 else 1)
        self._ck(self._lib.phaserot_group_sweep(self._g, dp, fmt, n_frames, ang_start, ang_end, stride, chn), "phaserot_group_sweep")

    def peaks(self):
        out = np.zeros((self.n_channels, self.maxsample), np.float32)
        self._ck(self._lib.phaserot_group_peaks(self._g, _ptr(out)), "phaserot_group_peaks")
        return out

    def reset(self):
        self._ck(self._lib.phaserot_group_reset(self._g), "phaserot_group_reset")

    def close(self):
        if self._g:
            self._lib.phaserot_group_destroy(self._g)
            self._g = C.c_void_p()

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
