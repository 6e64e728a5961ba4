/*
 * libphaserot_cuda — C ABI of the B200 (sm_100a) backend for the phase-rotation
 * hot path of x42/phaserotate.lv2.
 *
 * Plain C, plain pointers and sizes.  Every entry point names the reference
 * interface it replaces (paths relative to the reference tree, commit 00fece1).
 * There is no CPU fallback: phaserot_create() fails with PHASEROT_E_NO_DEVICE
 * when no sm_100 device is usable, and every other call fails on a handle that
 * could not be created.
 *
 * Threading: create/destroy may be called concurrently from any thread (the
 * reference serialises FFTW planning with a mutex for the same reason,
 * src/phaserotate.c:43,198-220,358-365).  All other calls on one handle must
 * come from one thread at a time (an LV2 run() thread, or the CLI main thread).
 *
 * Memory: the caller owns every host buffer passed in; the library owns device
 * memory, pinned staging buffers and streams.  Pointers documented as "device"
 * must be CUDA device pointers on the handle's device.
 */
#ifndef PHASEROT_CUDA_H
#define PHASEROT_CUDA_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(_WIN32)
#define PHASEROT_API __declspec(dllexport)
#else
#define PHASEROT_API __attribute__ ((visibility ("default")))
#endif

#define PHASEROT_ABI_VERSION 4

typedef struct phaserot phaserot_t;

enum {
	PHASEROT_OK            = 0,
	PHASEROT_E_INVAL       = -1, /* bad argument */
	PHASEROT_E_NO_DEVICE   = -2, /* no usable sm_100 GPU: there is no CPU fallback */
	PHASEROT_E_CUDA        = -3, /* a CUDA call failed; see phaserot_last_error() */
	PHASEROT_E_NOMEM       = -4, /* host or device allocation failed */
	PHASEROT_E_UNSUPPORTED = -5, /* valid for the reference but not implemented on the device path yet */
	PHASEROT_E_STATE       = -6, /* call not valid for this handle's mode */
	PHASEROT_E_AGAIN       = -7  /* sharded sweep only, see phaserot_pending_table(): combine the pending tables once more */
};

enum {
	/* Mirrors cli/phase-rotate.cc: FIR length = block size, PhaseRotate semantics. */
	PHASEROT_MODE_CLI = 0,
	/* Mirrors src/phaserotate.c: sizes from the sample rate (src:278-297), run() semantics. */
	PHASEROT_MODE_PLUGIN = 1
};

enum {
	/* Default (0): bug-compatible with the reference.  Flags switch single
	 * quirks off (SURVEY 3.3). */
	PHASEROT_FLAG_NO_FIRST_BLOCK_QUIRK = 1u << 0, /* Q1: test the first L/2 outputs against the real history */
	PHASEROT_FLAG_NO_PRUNE             = 1u << 1  /* evaluate every sample at every angle (no exact pruning) */
};

typedef struct phaserot_cfg {
	uint32_t abi_version; /* PHASEROT_ABI_VERSION */
	int32_t  mode;        /* PHASEROT_MODE_* */
	int32_t  n_channels;  /* CLI: SF_INFO.channels (cli:770-777); plugin: 1 or 2 (src/phaserotate.h:97) */
	int32_t  blksiz;      /* CLI: process block = FIR length, power of two in [1024, 32768] (cli:749-755) */
	double   sample_rate; /* plugin: rate passed to instantiate() (src:278-289) */
	int32_t  subsample;   /* angle grid: MAXSAMPLE = 180 * subsample; 0 -> 2 = the reference grid (cli:38-39) */
	int32_t  device;      /* CUDA device ordinal, -1 = current device */
	uint32_t flags;       /* PHASEROT_FLAG_* */
	int32_t  oversample;  /* analysis peak detector: 0 or 1 = digital (sample) peak like the reference
	                       * (cli:98-121, cli/dsp_peak_calc.h); 2 or 4 = oversampled true-peak, see below */
} phaserot_cfg_t;

/*
 * Oversampled true-peak (cfg.oversample = 2 or 4) is NOT a reference feature
 * (the reference measures the digital peak only; SURVEY 0.4) - parity is
 * unpinned and the definition below is this library's own, restated on the CPU
 * in oracle/phaserot_oracle.c (pro_cli_analyze_tp) for the tests.
 *
 * Interpolator: the 48-tap, 4-phase polyphase FIR of ITU-R BS.1770-4 Annex 2,
 *     s^[t, ph] = sum_{k = 0..11} c[ph][k] * s[t - k],   ph = 0..3
 * (oversample 2 uses phases 0 and 2).  Interpolation is linear, so the pair
 * (x_d, H) is interpolated once and every angle is evaluated on the result:
 *     peak[c][a] = max over the samples t the reference examines of
 *                  max ( |ca x_d[t] + sa H[t]|,  max_ph |ca x_d^[t, ph] + sa H^[t, ph]| )
 * i.e. the digital peak is always included (true-peak >= digital peak), x_d
 * carries the first-block rule (cli:418-419: zero for t < blksiz), and samples
 * before the stream start are zero.  For un-wrapped angle 0 (cli:413-414) the
 * same detector runs on the raw input.
 */

/* ---- lifetime ---------------------------------------------------------- */

/* Replaces: PhaseRotateProc + PhaseRotate construction (cli:128-165, 314-335,
 * 768-777) in CLI mode; the DSP part of instantiate() (src:278-404) in plugin
 * mode.  Designs the Hilbert FIR (same taps as the reference), uploads its
 * spectrum and allocates stream state.  Returns PHASEROT_OK or a negative
 * error; *out is NULL on failure. */
PHASEROT_API int phaserot_create (phaserot_t** out, const phaserot_cfg_t* cfg);

/* Replaces: ~PhaseRotate / ~PhaseRotateProc (cli:167-173, 337-353); cleanup() (src:179-223). */
PHASEROT_API void phaserot_destroy (phaserot_t* h);

/* Replaces: PhaseRotate::reset (cli:355-366) / activate() (src:511-520):
 * clears stream history, overlap state and the peak table.  The plugin's angle
 * state is NOT reset, like the reference (src:147,169-177). */
PHASEROT_API int phaserot_reset (phaserot_t* h);

/* Run all work of this handle on a caller-owned CUDA stream (cudaStream_t),
 * e.g. the stream a framework times with its own events and orders its
 * collectives against.  NULL restores the handle's private (non-blocking)
 * stream - so the legacy default stream, whose handle IS 0, cannot be selected
 * by passing it: use a created stream, or the special handles cudaStreamLegacy /
 * cudaStreamPerThread. */
PHASEROT_API int phaserot_set_stream (phaserot_t* h, void* cuda_stream);

/* ---- CLI analysis: min-peak sweep -------------------------------------- */

/* Replaces: one analyze_file() pass (cli:565-587) = PhaseRotate::analyze over
 * every block of the file plus the zero flush block, including the first-block
 * rule (cli:418-419) and the raw-peak rule for un-wrapped angle 0 (cli:413-414).
 *
 *   interleaved : n_frames * n_channels floats, host memory (pinned is faster)
 *   ang_start, ang_end, ang_stride : the angle loop of thr_process (cli:409-428),
 *                 in grid steps (half degrees for subsample 2)
 *   chn         : -1 = all channels, else only that channel (cli:434-435)
 *
 * Results accumulate (max) into the handle's peak table exactly like
 * PhaseRotate::_peak; read them with phaserot_peak()/phaserot_peaks().
 * Synchronous: the table is final when the call returns.
 *
 * Cost model: exact pruning drops every sample that cannot raise any angle's
 * running maximum; what survives goes on a list sized for programme material
 * (1/32 of a launch's samples).  Few-tone or constant-envelope input, where most
 * samples lie on the hull of the (x_d, H) point set, overflows it: the pass is
 * then repeated once in dense mode (launches sized to the list, and every
 * survivor evaluated only at the few angles it can still raise), the handle
 * stays in dense mode while the material needs it, and the table is the same
 * bit for bit either way (phaserot_stats_t.dense_repeats counts the repeats).
 * A handle also starts its NEXT sweep in dense mode, without a repeat, when a
 * finished sweep put more than 0.5 % of its samples on the lists, and returns
 * to normal mode once the lists hold less than 0.1 %. */
PHASEROT_API int phaserot_sweep (phaserot_t* h, const float* interleaved, uint64_t n_frames,
                                 int ang_start, int ang_end, int ang_stride, int chn);

/* The same pass over integer PCM as it sits in the file: `pcm` is HOST memory,
 * interleaved, PHASEROT_PCM_S16 (int16_t) or PHASEROT_PCM_S32 (int32_t; 24-bit
 * samples left-justified, as sf_readf_int delivers them).  The samples cross
 * PCIe as integers and are widened on the device with the conversion
 * libsndfile applies inside sf_readf_float (sample / 2^15, / 2^31), which is
 * what the reference reads with (cli/phase-rotate.cc:573): the result is
 * bit-identical to phaserot_sweep() on the converted floats, at half (or the
 * same) the host traffic.  Replaces sf_readf_float + de-interleave of
 * analyze_file / thr_process (cli:573, 397-401) for PCM files. */
#define PHASEROT_PCM_S16 1
#define PHASEROT_PCM_S32 2
/* packed 24-bit little-endian samples exactly as they sit in a WAV / RF64 / W64 data chunk
 * (what sf_read_raw returns): 3 bytes per sample on the host and on the bus, widened on the
 * device to the value sf_readf_float delivers (sample / 2^23) */
#define PHASEROT_PCM_S24 3
/* interleaved float32 (the format of phaserot_sweep), for the calls below that take a format */
#define PHASEROT_PCM_F32 0
PHASEROT_API int phaserot_sweep_pcm (phaserot_t* h, const void* pcm, int format, uint64_t n_frames,
                                     int ang_start, int ang_end, int ang_stride, int chn);

/* Same pass over audio that is already resident in device memory
 * (interleaved, n_frames * n_channels floats).  Work is enqueued on the
 * handle's stream; the peak table is brought back by the next
 * phaserot_peak()/phaserot_peaks()/phaserot_sync() call. */
PHASEROT_API int phaserot_sweep_device (phaserot_t* h, const float* d_interleaved, uint64_t n_frames,
                                        int ang_start, int ang_end, int ang_stride, int chn);

/* One shard of a longer stream, for sample-range sharding across GPUs: this
 * handle examines output samples of frames [0, n_frames) of the shard, where
 * the shard is preceded in the full stream by `hist` (blksiz frames,
 * interleaved, host or device memory; NULL = silence / start of stream; a
 * device pointer is read in place and must stay valid until the table is read).
 *   first != 0 : the shard starts the stream (first-block rule applies)
 *   last  != 0 : the shard ends it (short block zero padded + zero flush block)
 * Non-last shards must be a multiple of blksiz long.  Because a per-angle peak
 * is a maximum over samples, the element-wise max of all shards' tables is the
 * table of the whole stream (combine with an NCCL max all-reduce).  It equals
 * the single-pass table bit for bit when every shard starts at a multiple of
 * phaserot_shard_align() frames (the shards then cut the stream on the same
 * FFT segment grid); otherwise it agrees to fp32 FFT rounding (~1e-6). */
PHASEROT_API int phaserot_sweep_shard_device (phaserot_t* h, const float* d_interleaved, uint64_t n_frames,
                                              const float* hist, int first, int last,
                                              int ang_start, int ang_end, int ang_stride, int chn);

/* Two-phase form of phaserot_sweep_shard_device() for strong scaling (many ranks, each with a small
 * part of one stream).  A rank that bootstraps its filter radius from its own shard only prunes
 * against the peaks of that shard, which can be far below those of the whole stream: more survivors,
 * more sweep work, and the step waits for the worst rank.  Split the call:
 *     phaserot_sweep_shard_boot_device (h, ...);    enqueue the bootstrap wave of this shard only
 *     phaserot_pending_table + max all-reduce       the union of all ranks' waves = a sparse sample of the WHOLE stream
 *     phaserot_sweep_shard_resume (h);              the contiguous passes, pruning with the combined thresholds
 *     phaserot_pending_table + max all-reduce + phaserot_peaks   as for the one-call form
 * The result is the same table bit for bit (a running maximum; pruning is exact either way). */
PHASEROT_API int phaserot_sweep_shard_boot_device (phaserot_t* h, const float* d_interleaved, uint64_t n_frames,
                                                   const float* hist, int first, int last,
                                                   int ang_start, int ang_end, int ang_stride, int chn);
PHASEROT_API int phaserot_sweep_shard_resume (phaserot_t* h);

/* The same shard from HOST memory (`data`: interleaved, `format` = PHASEROT_PCM_*;
 * pinned is faster): uploaded in chunks on a copy stream while the compute stream
 * works on what has landed, like phaserot_sweep().  `hist`: blksiz frames of
 * float32 history (host or device) or NULL.  Asynchronous like the device form:
 * the table comes back with the next phaserot_peak()/phaserot_peaks()/phaserot_sync(),
 * so phaserot_pending_table() can be combined across ranks first.  Replaces the
 * read loop of analyze_file (cli:565-587) for one rank's part of the file. */
PHASEROT_API int phaserot_sweep_shard (phaserot_t* h, const void* data, int format, uint64_t n_frames,
                                       const float* hist, int first, int last,
                                       int ang_start, int ang_end, int ang_stride, int chn);

PHASEROT_API uint32_t phaserot_shard_align (const phaserot_t* h);

/* ---- per-section analysis and render ------------------------------------ */

/* Extends phaserot_sweep() / phaserot_sweep_pcm() (one analyze_file() pass, cli:565-587) with one min-peak
 * table per section of the stream, for material whose best angle changes along the file (an album or a
 * mix as one file, a broadcast, a film stem).  Same arguments, first-block and flush rules as
 * phaserot_sweep(); `data` is host memory in `format` = PHASEROT_PCM_*.  The stream is cut into sections
 * of section_frames frames, a positive multiple of phaserot_shard_align(h); the last section is the
 * remainder and the zero flush block belongs to it: ceil(n_frames / section_frames) sections.
 * The table of section k equals, bit for bit, the table phaserot_sweep_shard_device() gives for frames
 * [k S, (k+1) S) with the blksiz frames before them as history, first = (k == 0), last = (k == last
 * section); the element-wise max over the sections is the table of phaserot_sweep() bit for bit.  Grid
 * index 0 is the raw input peak of the section (cli:413-414).
 * One FFT pass over the whole stream, whose rows are (section, channel) pairs, each with its own filter
 * radius and survivor list: the launches do not grow with the number of sections.  A section whose list
 * overflows (few-tone material) is repeated through the shard path with dense mode
 * (phaserot_stats_t.dense_repeats counts these repeats).
 * At most 65535 (section, channel) rows per call (one hour of 48 kHz stereo in sections down to 0.11 s);
 * more is PHASEROT_E_INVAL with a phaserot_last_error() text, as is a section length off the alignment.
 * The handle's own peak table is not touched; every call starts from zeros.  Synchronous.
 * PHASEROT_E_STATE for plugin handles, PHASEROT_E_UNSUPPORTED for true-peak handles (oversample > 1). */
PHASEROT_API int phaserot_sweep_sections (phaserot_t* h, const void* data, int format, uint64_t n_frames, uint64_t section_frames,
                                          int ang_start, int ang_end, int ang_stride, int chn);
/* The same over audio resident in device memory (interleaved float32). */
PHASEROT_API int phaserot_sweep_sections_device (phaserot_t* h, const float* d_interleaved, uint64_t n_frames, uint64_t section_frames,
                                                 int ang_start, int ang_end, int ang_stride, int chn);
/* Tables of the last sections sweep: out[n_sections][n_channels][180 * subsample] (NULL: only
 * *n_sections is returned; 0 before the first sections sweep).  Extends phaserot_peaks(). */
PHASEROT_API int phaserot_section_peaks (phaserot_t* h, int* n_sections, float* out);

/* Extends phaserot_render() / phaserot_render_device() (PhaseRotate::apply over the stream, cli:467-485)
 * with one angle per section and channel: angles[k * n_channels + c], in grid steps on the FULL circle
 * (a + 2 * 180 * subsample renders the same output as a; a + 180 * subsample renders its negation).
 * Unlike phaserot_render(), the angles are not wrapped (cli:463).  Output sample t of section k is
 * rendered at angle a[k][c], except the first blksiz frames of every section k > 0, where the angle moves
 * linearly from a[k-1][c] to a[k][c]: at sample j of that ramp the angle is
 *     phi = a[k-1] + (a[k] - a[k-1]) * (j + 1) / blksiz grid steps
 * and (sa, ca) = sincos of phi times the SinCosLut constant (cli:41-72).  Outside the ramps every sample
 * equals phaserot_render() at that section's angle bit for bit.  Sections are those of
 * phaserot_sweep_sections() (same section_frames rule and row limit); flush_blocks and the output layout
 * are those of phaserot_render(); the apply() stream state is not changed.  Synchronous. */
PHASEROT_API int phaserot_render_sections (phaserot_t* h, const float* interleaved, uint64_t n_frames, uint64_t section_frames,
                                           const int* angles, int flush_blocks, float* out);
PHASEROT_API int phaserot_render_sections_device (phaserot_t* h, const float* d_interleaved, uint64_t n_frames, uint64_t section_frames,
                                                  const int* angles, int flush_blocks, float* d_out);

/* ---- integrated loudness of the rotated output ----------------------------- */

/* Extends the report of analyze_file (cli:931-947), which gives the peak before and after rotation, with the
 * integrated loudness of ITU-R BS.1770-4 before and after: the peak-to-loudness ratio a loudness target with a
 * true-peak ceiling (EBU R128: -23 LUFS / -1 dBTP) is met with, and a check that rotation kept the loudness.
 * For each of n_sets angle sets, lufs[k] is the integrated loudness of the output phaserot_render() writes after
 * the latency trim at those angles (the --fixed-write render):
 *     out[t] = ca[c] x[t] + sa[c] H'[t],   t in [0, n_frames),   H' = Hilbert branch aligned to x
 * with (sa, ca) the SinCosLut pair (cli:41-72) of angles[k * n_channels + c], in grid steps on the FULL circle as
 * in phaserot_render_sections() (a + 180 * subsample is the negation of a, which measures the same).  Set 0 at
 * angle 0 is the input itself.  No first-block rule applies: that rule belongs to the analysis only.
 *   K-weighting : the two biquads of BS.1770-4 (high shelf, then high pass), coefficients for any rate derived
 *                 as libebur128 does - at 48 kHz they are those of Tables 1 and 2
 *   gating      : sub-blocks of step = floor(sample_rate / 10 + 0.5) frames; 400 ms blocks of 4 sub-blocks,
 *                 hop 1 sub-block, complete blocks only; l_j = -0.691 + 10 log10 sum_c G_c z_cj; absolute gate
 *                 -70 LUFS, then the relative gate -10 LU; lufs = -0.691 + 10 log10 (gated mean)
 *                 -INFINITY when no block passes or the stream is shorter than 400 ms
 *   weights     : G_c per channel (NULL = 1.0 each; BS.1770 5.1 in WAV order: 1, 1, 1, 0, 1.41, 1.41)
 * Rotation and K-weighting are linear, so every 100 ms sub-block's mean square is a quadratic form in (ca, sa);
 * one pass gives its three sums and any number of angle sets costs only the gate.
 * `data` and `format` as phaserot_sweep_pcm() / PHASEROT_PCM_F32, with the same widening; host memory.
 * Synchronous; deterministic (the same doubles on every call, and from the host and device forms on the same
 * float input).  The peak table, section tables and apply() stream state are not changed (the host form
 * completes a pending device sweep first, as phaserot_peaks() would).  Valid for true-peak handles too.
 * PHASEROT_E_STATE for plugin handles; PHASEROT_E_INVAL with a phaserot_last_error() text for n_sets < 1, NULL
 * angles or lufs, a negative or non-finite weight, n_frames == 0 or a sample_rate outside [8000, 768000]. */
PHASEROT_API int phaserot_loudness (phaserot_t* h, const void* data, int format, uint64_t n_frames, double sample_rate,
                                    const float* weights, const int* angles, int n_sets, double* lufs);
/* The same over audio resident in device memory (interleaved float32, n_frames * n_channels). */
PHASEROT_API int phaserot_loudness_device (phaserot_t* h, const float* d_interleaved, uint64_t n_frames, double sample_rate,
                                           const float* weights, const int* angles, int n_sets, double* lufs);

/* ---- overs above a ceiling ------------------------------------------------- */

/* Extends the min-peak sweep, which says at which angle the single largest sample is smallest, with how much
 * of the rotated output a limiter or clipper after a ceiling T (linear, e.g. -1 dBTP) would have to work on:
 * for every angle, the number of samples above T and by how much, from one pass.
 *   sample set : exactly the samples and detector points phaserot_sweep() evaluates on the same handle and input
 *                (first-block rule cli:418-419, the zero flush block, chn, the digital peak or the oversample =
 *                2 / 4 detector of the true-peak definition above); grid index 0 is the raw input under the
 *                same detector (cli:413-414)
 *   digital    : sample t is over at angle a when |y| > T, y = fmaf (ca, x_d, sa * H) - the expression of the
 *                sweep, so counts[c][a] > 0 exactly when phaserot_sweep()'s peak[c][a] > T, index 0 included
 *   true-peak  : sample t is over when the largest |y| over its detector points exceeds T; samples are counted,
 *                not points
 *   excess     : excess[c][a] = sum over the overs of (v - T), v the value that made the sample over; every term is
 *                truncated to a multiple of 2^-32 and summed in 64-bit integers, so repeated calls and the host and
 *                device forms return the same doubles.  The sum of one entry must stay below 2^32 (full scale = 1.0):
 *                audio within full scale cannot reach it (an hour of 48 kHz audio is 1.7e8 samples, each term a few units at most);
 *                float input far outside [-1, 1] with a low ceiling can, and its excess is then not defined (the
 *                counts are)
 *   output     : full tables counts[n_channels][180 * subsample], excess[n_channels][180 * subsample] (excess may be
 *                NULL); entries outside the requested angles and channel are 0.  Should the angle loop reach grid
 *                index 0 both as angle 0 (raw input) and wrapped (a multiple of 180 * subsample), the entry holds
 *                whichever of the two has more overs.
 * A point whose radius sqrt(x_d^2 + H^2) is below T cannot be over T at any angle: T is the fixed radius of the
 * sweep's exact pruning, and PHASEROT_FLAG_NO_PRUNE (radius 0: every examined point listed) gives the same tables.  Low ceilings
 * put most samples on the survivor lists; an FFT launch whose list overflows is re-run in pieces that fit
 * (phaserot_stats_t.dense_repeats counts these re-runs) - the tables do not depend on it.
 * `data` and `format` as phaserot_sweep_pcm() / PHASEROT_PCM_F32, with the same widening; host memory.
 * Synchronous.  The peak table, section tables and apply() stream state are not changed (the host form completes
 * a pending device sweep first, as phaserot_peaks() would).  PHASEROT_E_STATE for plugin handles;
 * PHASEROT_E_INVAL with a phaserot_last_error() text for a ceiling <= 0 or not finite, n_frames == 0, NULL counts,
 * and the angle and channel arguments phaserot_sweep() rejects. */
PHASEROT_API int phaserot_overs (phaserot_t* h, const void* data, int format, uint64_t n_frames, float ceiling,
                                 int ang_start, int ang_end, int ang_stride, int chn,
                                 uint64_t* counts, double* excess);
/* The same over audio resident in device memory (interleaved float32, n_frames * n_channels). */
PHASEROT_API int phaserot_overs_device (phaserot_t* h, const float* d_interleaved, uint64_t n_frames, float ceiling,
                                        int ang_start, int ang_end, int ang_stride, int chn,
                                        uint64_t* counts, double* excess);

/* ---- rank table: the N largest samples at every angle --------------------- */

/* The level that N samples of the rotated output reach, at every angle, from one pass: a limiter or clipper after
 * the rotation has to act on the samples above it, so the angle where it is lowest is the angle to pick for such a
 * stage (the sweep's peak is rank 1).
 *   samples    : exactly those phaserot_overs() examines on the same handle and input (first-block rule
 *                cli:418-419, the zero flush block, chn, the digital or oversample = 2 / 4 true-peak detector);
 *                grid index 0 is the raw input under the same detector over the frames of the raw-peak rule
 *                (cli:413-414)
 *   value      : v_t(a) = fabsf (fmaf (ca, x_d, sa * H)), the sweep's expression; true-peak: the largest of these
 *                over the sample's detector points (samples are ranked, not points)
 *   output     : out[n_channels][180 * subsample][n_rank]; out[c][a][k] is the (k+1)-th largest v_t(a) over the
 *                examined samples, a multiset (equal values of different samples repeat), so each row is
 *                non-increasing.  Entries beyond the number of examined samples are 0, and so are the rows outside
 *                the requested angles and channel.  Should the angle loop reach grid index 0 both as angle 0 (raw
 *                input) and wrapped, the row is whichever of the two has the larger rank-1 value (ties: the raw
 *                row), so that out[c][a][0] == peak[c][a] of phaserot_sweep() for every (c, a), index 0 included.
 * For every ceiling T, min (counts[c][a], n_rank) of phaserot_overs() at T equals the number of k with
 * out[c][a][k] > T.  A sample whose radius sqrt(x_d^2 + H^2) is below the N-th value of every angle cannot change
 * any row: the running N-th values are the radius of the sweep's exact pruning, and PHASEROT_FLAG_NO_PRUNE (radius
 * 0) gives the same table.  The table is a sorted multiset: it does not depend on how the work is split, and
 * repeated calls and the host and device forms return the same floats.  Material on which most samples stay near
 * the N-th value (pure tones) keeps most samples listed; the launches whose lists or candidate buffers overflow
 * are re-run in pieces that fit (phaserot_stats_t.dense_repeats counts them).
 * 1 <= n_rank <= 256.  `data` and `format` as phaserot_sweep_pcm() / PHASEROT_PCM_F32, with the same widening;
 * host memory.  Synchronous.  The peak table, section tables and apply() stream state are not changed (the host
 * form completes a pending device sweep first).  PHASEROT_E_STATE for plugin handles; PHASEROT_E_INVAL with a
 * phaserot_last_error() text for n_rank out of range, NULL out, n_frames == 0, and the angle and channel arguments
 * phaserot_sweep() rejects. */
PHASEROT_API int phaserot_nth_peaks (phaserot_t* h, const void* data, int format, uint64_t n_frames, int n_rank,
                                     int ang_start, int ang_end, int ang_stride, int chn, float* out);
/* The same over audio resident in device memory (interleaved float32, n_frames * n_channels). */
PHASEROT_API int phaserot_nth_peaks_device (phaserot_t* h, const float* d_interleaved, uint64_t n_frames, int n_rank,
                                            int ang_start, int ang_end, int ang_stride, int chn, float* out);

/* ---- several GPUs in one process ---------------------------------------- */

/* A group of handles, one per device, that analyses ONE stream: the file is cut
 * on phaserot_shard_align() into one contiguous shard per device (sample-range
 * sharding; every shard reads blksiz frames of history in front), every device
 * uploads and sweeps its shard concurrently, and the per-angle maxima are
 * combined on the first device by a kernel that reads the other devices'
 * tables through NVLink peer memory (element-wise max; exact and associative,
 * so the result equals the single-device table bit for bit).  No NCCL
 * bootstrap: a CLI run is over before a communicator would be up.  Replaces
 * analyze_file + the merge of the per-thread `_peak` rows (cli:431-444,
 * 565-587) for `phase-rotate --gpus N`.
 *   devices   : n_devices CUDA ordinals (NULL = 0 .. n_devices - 1); cfg->device is ignored
 * The group's peak table is read with phaserot_group_peaks(); handle 0 of the
 * group (phaserot_group_handle) serves render / lut / latency queries. */
typedef struct phaserot_group phaserot_group_t;
PHASEROT_API int  phaserot_group_create (phaserot_group_t** out, const phaserot_cfg_t* cfg, const int* devices, int n_devices);
PHASEROT_API void phaserot_group_destroy (phaserot_group_t* g);
PHASEROT_API int  phaserot_group_size (const phaserot_group_t* g);
PHASEROT_API phaserot_t* phaserot_group_handle (phaserot_group_t* g, int i);
/* one analyze_file() pass over host memory (`format` = PHASEROT_PCM_*), same angle arguments as phaserot_sweep() */
PHASEROT_API int  phaserot_group_sweep (phaserot_group_t* g, const void* data, int format, uint64_t n_frames,
                                        int ang_start, int ang_end, int ang_stride, int chn);
PHASEROT_API int  phaserot_group_peaks (phaserot_group_t* g, float* out);
PHASEROT_API int  phaserot_group_reset (phaserot_group_t* g);

/* Device-resident result of the sweep that is still pending (enqueued, not read
 * back yet), for combining shards without a host round trip: *d_table points at
 * n_channels * n_angles + n_channels + 1 floats owned by the handle - the running
 * per-angle maxima [channel][angle slot], the raw input peak of every channel
 * (the value of grid index 0, cli:413-414), and one word of the library's own:
 * non-zero when this shard's survivor list overflowed (see phaserot_sweep).  All
 * values are >= 0, so an element-wise max over the shards' WHOLE buffers (NCCL
 * all-reduce, ncclMax, in place, enqueued after the sweep on the handle's stream;
 * nothing is synchronised here) is the result of the whole stream; the next
 * phaserot_peaks()/phaserot_sync() then reads the combined table back on every
 * rank.  Because the flag is part of the reduced buffer every rank learns in the
 * same step that some shard was incomplete: phaserot_peaks()/phaserot_sync()
 * then return PHASEROT_E_AGAIN on EVERY rank after re-enqueueing the rank's
 * shard in dense mode on top of the combined table - the caller repeats
 *     phaserot_pending_table() -> all-reduce -> phaserot_peaks()
 * once (dense launches cannot overflow).  Programme material never takes that
 * path.  Replaces the merge of the per-thread `_peak` rows in
 * PhaseRotate::analyze (cli:431-444) across devices.  PHASEROT_E_STATE when no
 * sweep is pending. */
PHASEROT_API int phaserot_pending_table (phaserot_t* h, float** d_table, int* n_channels, int* n_angles);

/* Block-streaming drop-in for PhaseRotate::analyze (cli:431-444): feed one
 * block of blksiz frames at a time (`start` != 0 for the first block of a
 * file, cli:571-582).  Blocks are staged and processed in large batches; the
 * peak table is completed by the next phaserot_peak()/phaserot_peaks() call.
 * The angle range must stay the same between two reads of the table. */
PHASEROT_API int phaserot_analyze (phaserot_t* h, const float* block, int ang_start, int ang_end,
                                   int ang_stride, int chn, int start);

/* Replaces: PhaseRotate::peak (cli:275-285), incl. c < 0 -> peak_all (cli:287-299). */
PHASEROT_API float phaserot_peak (phaserot_t* h, int c, int a);

/* Whole table: out[n_channels][180 * subsample]. */
PHASEROT_API int phaserot_peaks (phaserot_t* h, float* out);

/* sin/cos of the angle grid as used for every rotation: the reference's
 * SinCosLut (cli:41-72).  s, c: [180 * subsample]. */
PHASEROT_API int phaserot_lut (phaserot_t* h, float* s, float* c);

/* ---- CLI render -------------------------------------------------------- */

/* Replaces: PhaseRotate::apply (cli:467-485) — one block of blksiz frames,
 * in place, interleaved; angles[c] in grid steps, wrapped like cli:463.
 * Stateful (history + overlap), synchronous. */
PHASEROT_API int phaserot_apply (phaserot_t* h, float* buf, const int* angles);

/* Bulk form of the same stream: processes ceil(n_frames / blksiz) zero padded
 * blocks plus `flush_blocks` zero blocks from reset state in one device pass.
 * out: (ceil(n_frames / blksiz) + flush_blocks) * blksiz frames, interleaved,
 * no latency trim (the trim stays in the host write loop, cli:963-1001). */
PHASEROT_API int phaserot_render (phaserot_t* h, const float* interleaved, uint64_t n_frames,
                                  const int* angles, int flush_blocks, float* out);

/* After phaserot_render() the handle's apply() stream state is that of the
 * last block processed (the zero flush block, or the last input block when
 * flush_blocks == 0), so phaserot_apply() can continue the same stream. */

/* Device-resident form: d_in / d_out are device pointers (same shapes). */
PHASEROT_API int phaserot_render_device (phaserot_t* h, const float* d_interleaved, uint64_t n_frames,
                                         const int* angles, int flush_blocks, float* d_out);

/* ---- plugin ------------------------------------------------------------ */

/* Replaces: the audio path of run() -> process_channel() (src:538-725, 774-852)
 * for all channels of the instance: planar in[c] / out[c] of n_frames floats
 * (in[c] == out[c] allowed, src:780-785), angle_deg[c] = value of the angle
 * control port for this call (src:564-571).  Keeps the reference's latency
 * (phaserot_latency()) and its per-partition angle ramp (src:673-717).
 * Synchronous; no host allocation in steady state. */
PHASEROT_API int phaserot_process (phaserot_t* h, const float* const* in, float* const* out,
                                   uint32_t n_frames, const float* angle_deg);

/* phaserot_process() that also returns the two level-meter inputs of the
 * plugin's run() for this call, reduced on the device: level_in[c] = max |x|
 * over the input delayed by the plugin latency (the samples that line up with
 * this call's output; src/phaserotate.c:573-609), level_out[c] = max |y| over
 * the n_frames outputs (src:727-739).  NaNs are ignored (fmax).  Either pointer
 * NULL = plain phaserot_process().  The meter ballistics (hold, fall-off,
 * peak-hold, `levels` notification) stay on the host: they are per call, not
 * per sample. */
PHASEROT_API int phaserot_process_levels (phaserot_t* h, const float* const* in, float* const* out, uint32_t n_frames,
                                          const float* angle_deg, float* level_in, float* level_out);

/* Angle state of every channel in turns (Channel::angle, src/phaserotate.c:53), as
 * process_channel() finds it at the start of the NEXT call: the reference re-arms
 * its delayed meter reset while `target_angle != angle` (src:564-571, 611), i.e.
 * for as long as the ramp is still moving.  angle_turns: [n_channels]. */
PHASEROT_API int phaserot_plugin_angle (phaserot_t* h, float* angle_turns);

/* Replaces: FFTiProc::latency = parsiz + firlat (src:297); CLI: blksiz / 2 (cli:963). */
PHASEROT_API uint32_t phaserot_latency (const phaserot_t* h);

/* ---- misc -------------------------------------------------------------- */

/* Page-locked host memory for audio buffers handed to sweep/render (makes the
 * H2D/D2H copies asynchronous and full speed).  Optional: any host pointer is
 * accepted by every call. */
PHASEROT_API void* phaserot_alloc_host (uint64_t bytes);
PHASEROT_API void  phaserot_free_host (void* p);

/* Wait for all enqueued work of this handle and bring the peak table back. */
PHASEROT_API int phaserot_sync (phaserot_t* h);

/* Counters since create/reset_stats: kernels launched by this library and
 * sample-angle pairs actually evaluated after exact pruning. */
typedef struct phaserot_stats {
	uint64_t kernel_launches;
	uint64_t points_total;     /* (channel, sample) pairs examined by the sweep filter */
	uint64_t points_evaluated; /* pairs that survived pruning and were evaluated at every angle */
	uint64_t h2d_bytes;
	uint64_t d2h_bytes;
	uint64_t dense_repeats;    /* passes repeated in dense mode because a survivor list overflowed (see phaserot_sweep) */
} phaserot_stats_t;
PHASEROT_API int phaserot_get_stats (phaserot_t* h, phaserot_stats_t* out);
PHASEROT_API int phaserot_reset_stats (phaserot_t* h);

/* Per-kernel device times, measured with CUDA events recorded on the handle's
 * stream around every launch while profiling is on (bench.py's roofline leg).
 * Index: 0 fftconv+filter (sweep), 1 angle sweep, 2 deinterleave/interleave,
 * 3 fftconv+rotate (render), 4 direct FIR (plugin small calls), 5 other,
 * 6 true-peak sweep front end (fftconv -> Hilbert branch, interpolate + filter). */
#define PHASEROT_NKERNELS 7
typedef struct phaserot_ktimes {
	double   ms[PHASEROT_NKERNELS];
	uint64_t launches[PHASEROT_NKERNELS];
} phaserot_ktimes_t;
PHASEROT_API int phaserot_set_profiling (phaserot_t* h, int on);
PHASEROT_API int phaserot_get_kernel_times (phaserot_t* h, phaserot_ktimes_t* out);

PHASEROT_API const char* phaserot_strerror (int code);
/* Text of the last CUDA failure on this thread ("" if none). */
PHASEROT_API const char* phaserot_last_error (void);
PHASEROT_API int         phaserot_abi_version (void);

#ifdef __cplusplus
}
#endif
#endif
