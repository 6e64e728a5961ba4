// libphaserot_cuda: host side of the C ABI declared in include/phaserot_cuda.h.
//
// What runs where
//   host   : FIR design (once), angle tables, the plugin's per-partition angle
//            ramp state machine, peak-table bookkeeping (PhaseRotate::_peak)
//   device : everything that touches audio samples (kernels.cuh)
//
// There is no CPU fallback in this file: every audio path ends in a kernel
// launch, and create() refuses to hand out a handle without an sm_100 device.
#include "../../../include/phaserot_cuda.h"
#include "kernels.cuh"
#include "loudness.cuh"
#include "fft16k_tables.h"

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <limits>
#include <mutex>
#include <new>
#include <string>
#include <thread>
#include <type_traits>
#include <vector>

#ifndef M_PI
#define M_PI 3.14159265358979323846
#endif

using namespace prk;

namespace {

thread_local char g_last_error[512] = "";
std::mutex        g_create_lock;

int
cuda_fail (cudaError_t e, const char* what, int line)
{
	snprintf (g_last_error, sizeof (g_last_error), "%s failed at phaserot_cuda.cu:%d: %s", what, line, cudaGetErrorString (e));
	return PHASEROT_E_CUDA;
}

#define CK(call)                                              \
	do {                                                      \
		cudaError_t e_ = (call);                              \
		if (e_ != cudaSuccess) {                              \
			return cuda_fail (e_, #call, __LINE__);           \
		}                                                     \
	} while (0)

// ---------------------------------------------------------------------------
// FIR design (host, once per handle)
// ---------------------------------------------------------------------------

// Hilbert FIR taps of length L.
// Reference: cli/phase-rotate.cc:144-161 (window constant 0.5f/L held in float,
// cli:142) and src/phaserotate.c:374-391 (window constant in double).  Both
// inverse-transform the half spectrum F[k] = (0, (-1)^k), k = 0..L/2, whose
// closed form is -2 cot(pi (i - L/2) / L) at odd (i - L/2) and zero elsewhere,
// then apply a Hann window scaled by 0.5/L in double and store float.
void
design_fir (int L, bool plugin, std::vector<float>& taps)
{
	taps.assign ((size_t)L, 0.f);
	const double scale = plugin ? 0.5 / (double)L : (double)(0.5f / (float)L);
	for (int i = 0; i < L; ++i) {
		const int m = i - L / 2;
		if (!(m & 1)) {
			continue;
		}
		const float  raw = (float)(-2.0 / std::tan (M_PI * (double)m / (double)L));
		const double win = scale * (1.0 - std::cos (2.0 * M_PI * (double)i * (1.0 / (double)L)));
		taps[(size_t)i]  = (float)((double)raw * win);
	}
}

// reference SinCosLut (cli/phase-rotate.cc:41-72), generalised to subsample S:
//   float mp = 2.f * M_PI / S / -360.0;  sincosf (mp * i, &s, &c)
void
build_lut (int S, std::vector<float>& s, std::vector<float>& c)
{
	const int   n  = 180 * S;
	const float mp = (float)(2.f * M_PI / S / -360.0);
	s.resize ((size_t)n);
	c.resize ((size_t)n);
	for (int i = 0; i < n; ++i) {
		sincosf (mp * (float)i, &s[(size_t)i], &c[(size_t)i]);
	}
}

struct DevBuf {
	void*  p   = nullptr;
	size_t cap = 0;
	int ensure (size_t bytes)
	{
		if (bytes <= cap) {
			return PHASEROT_OK;
		}
		if (p) {
			cudaFree (p);
			p   = nullptr;
			cap = 0;
		}
		const size_t want = bytes + bytes / 8 + 4096;
		cudaError_t  e    = cudaMalloc (&p, want);
		if (e != cudaSuccess) {
			e = cudaMalloc (&p, bytes);
			if (e != cudaSuccess) {
				cudaGetLastError ();
				snprintf (g_last_error, sizeof (g_last_error), "cudaMalloc(%zu) failed: %s", bytes, cudaGetErrorString (e));
				return PHASEROT_E_NOMEM;
			}
			cap = bytes;
			return PHASEROT_OK;
		}
		cap = want;
		return PHASEROT_OK;
	}
	void release ()
	{
		if (p) {
			cudaFree (p);
		}
		p   = nullptr;
		cap = 0;
	}
};

struct PinBuf {
	void*  p   = nullptr; // host pointer
	void*  d   = nullptr; // device alias (mapped)
	size_t cap = 0;
	int ensure (size_t bytes)
	{
		if (bytes <= cap) {
			return PHASEROT_OK;
		}
		if (p) {
			cudaFreeHost (p);
			p = d = nullptr;
			cap   = 0;
		}
		cudaError_t e = cudaHostAlloc (&p, bytes, cudaHostAllocMapped);
		if (e != cudaSuccess) {
			cudaGetLastError ();
			snprintf (g_last_error, sizeof (g_last_error), "cudaHostAlloc(%zu) failed: %s", bytes, cudaGetErrorString (e));
			return PHASEROT_E_NOMEM;
		}
		e = cudaHostGetDevicePointer (&d, p, 0);
		if (e != cudaSuccess) {
			d = nullptr;
			cudaGetLastError ();
		}
		cap = bytes;
		return PHASEROT_OK;
	}
	void release ()
	{
		if (p) {
			cudaFreeHost (p);
		}
		p = d = nullptr;
		cap   = 0;
	}
};

// per-channel angle state of the plugin (Channel::angle/sa/ca, src:53-55)
struct PluginChan {
	float               angle = 0.f;
	float               sa = 0.f, ca = 1.f;
	std::vector<float2> last;          // coefficients of the last completed partition
	bool                last_is_ramp = false;
	float2              last_const   = make_float2 (1.f, 0.f);
};

// One analysis pass over a stream (sweep_core)
struct SweepJob {
	const void*  src         = nullptr;          // interleaved frames (host or device)
	bool         on_device   = false;            // src is device memory (float32)
	int          fmt         = PHASEROT_PCM_F32; // host src: PHASEROT_PCM_*
	long long    n_frames    = 0;                // frames present in src
	int          flush       = 0;                // zero blocks after the last (partial) block of src (stream_geom)
	bool         first_block = false;            // apply the first-block rule (cli:418-419) to t < L
	const float* hist        = nullptr;          // L frames of history preceding src (interleaved) or null
	int          ang_start = 0, ang_end = 0, ang_stride = 1, chn = -1;
};

// The pass over F frames that are a whole stream (first and last) or one shard of it: the last shard ends with
// one zero flush block (analyze_file, cli:572-586; every other shard is whole blocks, check_sweep), and the
// first-block rule applies to the first shard
SweepJob
shard_job (const void* src, bool on_device, int fmt, long long F, const float* hist, bool first, bool last, int ang_start, int ang_end, int ang_stride,
           int chn)
{
	return { src, on_device, fmt, F, last ? 1 : 0, first && F > 0, hist, ang_start, ang_end, ang_stride, chn };
}

// d_small: per-channel state of the pending sweep and the render
struct SmallState {
	unsigned           count[64];
	float              thr2[64];
	int                ramp_len[64];
	unsigned long long stats[3]; // points listed in dense mode, evaluated points, overflow word of bootstrap launches (nobody reads it)
	unsigned           count_odd[64]; // list counts of odd launches
	unsigned           r2max[64];
	unsigned           wide_count[64];
};

} // namespace

struct phaserot {
	phaserot_cfg_t cfg;
	int            dev   = 0;
	int            n_sm  = 148;
	int            C     = 1;
	int            L     = 0;   // FIR length
	int            Lh    = 0;   // half taps (odd taps of the FIR)
	int            NP    = 1;   // tap partitions of the FFT convolution (2 for L = 32768)
	int            Lp    = 0;   // half taps per partition = overlap of consecutive segments
	int            V     = 0;   // valid complex outputs per segment
	int            padf  = 0;   // front pad of a plane (complex elements)
	int            S     = 2;
	int            MS    = 360; // MAXSAMPLE
	bool           plugin = false;
	// plugin sizes (src:278-297)
	uint32_t P = 0, firlen = 0, firlat = 0;

	cudaStream_t own_stream = nullptr, copy_stream = nullptr, stream = nullptr;
	cudaEvent_t  ev_copy[2] = { nullptr, nullptr }, ev_done[2] = { nullptr, nullptr };

	std::vector<float> taps, lut_s, lut_c;
	std::vector<float> table; // [C][MS]  == PhaseRotate::_peak

	DevBuf d_G, d_G1, d_scratch, d_tw, d_g;
	DevBuf d_plane, d_out, d_list, d_stage[2], d_io, d_inter, d_hist;
	DevBuf d_small; // SmallState
	DevBuf d_cs, d_peaks, d_ramp, d_chancs;
	// dense mode (long survivor lists, see sweep_window_kernel): grid index -> slot, sector thresholds, wide list
	DevBuf d_slot, d_sec, d_wide;
	PinBuf h_slot;
	bool      dense_mode  = false; // sticky: the last sweep overflowed its survivor list (few-tone / constant-envelope material)
	long long list_cap    = 0;     // points per channel the list holds
	SweepJob  redo;                // the pending sweep in device-resident form, for a dense-mode repeat or a resume
	uint64_t pend_points = 0; // points examined by the pending sweep (statistics; dense-mode exit test)
	int      pend_again   = 0;     // PHASEROT_E_AGAIN returned for the pending sweep so far
	bool     pend_exposed = false; // the pending table was handed out (phaserot_pending_table): the caller combines shards
	bool     pend_redone = false; // the pending sweep was repeated in dense mode (its list counts start from a raised table)
	DevBuf d_tpH; // true-peak staging of the Hilbert branch: [C][tp_stride] floats
	long long tp_stride = 0;
	int       OS        = 1; // 1 = digital peak, 2 / 4 = oversampled true-peak
	PinBuf h_stage[2], h_res, h_io, h_cs;
	long long plane_stride = 0, out_stride = 0, list_stride = 0;

	// per-section analysis (phaserot_sweep_sections): device table [rows][A] | raw peaks [rows], row = section * (c1 - c0) + c - c0;
	// d_sect_aux: evaluated points (u64) | thr2 [rows] | count [rows] | overflow flags [rows] | bootstrap flags [rows] | r2max [rows]
	DevBuf                 d_sect, d_sect_aux, d_sect_rt;
	long long              sect_n = 0;
	int                    sect_A = 0, sect_c0 = 0, sect_c1 = 0;
	bool                   sect_raw = false;
	std::vector<int>       sect_idx;
	std::vector<long long> sect_redo_k; // sections whose list overflowed: their tables come from the shard path
	std::vector<float>     sect_redo;   // [redone section][C][MS]

	// integrated loudness (phaserot_loudness): K(x) [frames][C] floats | Hilbert branch of one FFT launch [C][stride]
	// floats | fp64 work: sub-block sums, head correction, chunk states, A powers, weights, results | angle sets
	DevBuf d_kx, d_lH, d_lwork, d_lset;

	// overs table (phaserot_overs): survivor list | true-peak staging of the Hilbert branch | tables, angle table,
	// radii and the list counters of every launch; its own buffers, so that a pending device sweep is not disturbed.
	// The rank table (phaserot_nth_peaks) shares the list and the staging.
	DevBuf d_ovl, d_ovH, d_ovw;
	// rank table: rows, thresholds, counters, radix selection state | candidate buckets
	DevBuf d_nthw, d_nthc;

	// pending (asynchronous) sweep result
	bool             pending = false;
	std::vector<int> pend_idx;
	bool             pend_raw = false;
	int              pend_c0 = 0, pend_c1 = 0;
	int              pend_A = 0;

	// streaming analyze()
	std::vector<float> an_buf;
	int                an_start = 0, an_end = 0, an_stride = 1, an_chn = -1, an_first = 0;
	uint64_t           an_blocks = 0;
	std::vector<float> hist; // last L frames of the previous stream (interleaved)
	bool               hist_valid = false;

	// apply() stream state
	std::vector<float> ap_hist;

	// plugin stream state
	std::vector<PluginChan> pch;
	std::vector<float>      ptail; // [C][firlen + P] newest input last
	uint64_t                ppos = 0;
	DevBuf                  d_ring;             // [C][kRing] input history of the small-call path
	bool                    ring_valid = false; // false: re-seed the ring from ptail before the next small call

	phaserot_stats_t stats {};

	// profiling: event pairs around launches, resolved at the next sync
	bool                     prof = false;
	std::vector<cudaEvent_t> prof_ev;   // pool, pairs
	std::vector<int>         prof_kind; // kind per used pair
	size_t                   prof_used = 0;
	phaserot_ktimes_t        ktimes {};
};

namespace {

struct DevGuard {
	int prev = -1;
	explicit DevGuard (int dev)
	{
		cudaGetDevice (&prev);
		if (prev != dev) {
			cudaSetDevice (dev);
		} else {
			prev = -1;
		}
	}
	~DevGuard ()
	{
		if (prev >= 0) {
			cudaSetDevice (prev);
		}
	}
};

constexpr size_t kSmallBytes = sizeof (SmallState);
struct ProfScope {
	phaserot* h;
	size_t    slot = (size_t)-1;
	ProfScope (phaserot* h_, int kind) : h (h_)
	{
		if (!h->prof) return;
		if ((h->prof_used + 1) * 2 > h->prof_ev.size ()) {
			for (int i = 0; i < 2; ++i) {
				cudaEvent_t e;
				if (cudaEventCreate (&e) != cudaSuccess) return;
				h->prof_ev.push_back (e);
			}
		}
		slot = h->prof_used++;
		h->prof_kind.resize (h->prof_used);
		h->prof_kind[slot] = kind;
		cudaEventRecord (h->prof_ev[2 * slot], h->stream);
	}
	~ProfScope ()
	{
		if (slot != (size_t)-1) cudaEventRecord (h->prof_ev[2 * slot + 1], h->stream);
	}
};

// call after the stream is synchronised
void
prof_resolve (phaserot* h)
{
	for (size_t i = 0; i < h->prof_used; ++i) {
		float ms = 0.f;
		if (cudaEventElapsedTime (&ms, h->prof_ev[2 * i], h->prof_ev[2 * i + 1]) == cudaSuccess) {
			h->ktimes.ms[h->prof_kind[i]] += ms;
			h->ktimes.launches[h->prof_kind[i]] += 1;
		} else {
			cudaGetLastError ();
		}
	}
	h->prof_used = 0;
}

SmallState*         d_small (phaserot* h) { return (SmallState*)h->d_small.p; }
unsigned*           d_count (phaserot* h) { return d_small (h)->count; }
float*              d_thr2 (phaserot* h) { return d_small (h)->thr2; }
// raw input peaks [C]: directly behind the [C][A] table of the pending sweep, so that table and
// raw peaks are one contiguous buffer (one D2H copy, one all-reduce when shards are combined)
unsigned*           d_raw (phaserot* h) { return (unsigned*)h->d_peaks.p + (size_t)std::max (h->pend_A, 1) * h->C; }
int*                d_ramplen (phaserot* h) { return d_small (h)->ramp_len; }
unsigned long long* d_stats (phaserot* h) { return d_small (h)->stats; }
// List-overflow flag of the pending sweep: the word behind the raw peaks, i.e. the LAST element of the
// device table (bits of 1.0f when set).  It travels with the table through an external max all-reduce, so
// every rank of a sharded sweep learns that some shard is incomplete without a second collective.
unsigned*           d_overflow (phaserot* h) { return d_raw (h) + h->C; }
unsigned*           d_overflow_ignored (phaserot* h) { return (unsigned*)&d_small (h)->stats[2]; }
unsigned*           d_count_odd (phaserot* h) { return d_small (h)->count_odd; }
unsigned*           d_r2max (phaserot* h) { return d_small (h)->r2max; }
unsigned*           d_wide_count (phaserot* h) { return d_small (h)->wide_count; }

int
upload_tables (phaserot* h)
{
	// odd taps g[j] = fir[2j + 1]: the complex half-rate convolution kernel
	const int Lh = h->Lh;
	std::vector<float> g ((size_t)Lh);
	for (int j = 0; j < Lh; ++j) {
		g[(size_t)j] = h->taps[(size_t)(2 * j + 1)];
	}
	// filter spectrum / M in MID-pass order, twiddles (fft16k_tables.h)
	const std::vector<float2> G = make_filter_spectrum (g.data (), h->Lp);
	int rc = h->d_G.ensure (sizeof (float2) * kM);
	if (rc) return rc;
	CK (cudaMemcpy (h->d_G.p, G.data (), sizeof (float2) * kM, cudaMemcpyHostToDevice));
	if (h->NP == 2) {
		// second half of the taps and the per-CTA spectrum scratch (see mid_pass())
		const std::vector<float2> G1 = make_filter_spectrum (g.data () + h->Lp, h->Lp);
		rc = h->d_G1.ensure (sizeof (float2) * kM);
		if (rc) return rc;
		CK (cudaMemcpy (h->d_G1.p, G1.data (), sizeof (float2) * kM, cudaMemcpyHostToDevice));
		rc = h->d_scratch.ensure (sizeof (float2) * kM * (size_t)h->n_sm);
		if (rc) return rc;
	}
	const std::vector<float2> tw = make_twiddles ();
	rc = h->d_tw.ensure (sizeof (float2) * tw.size ());
	if (rc) return rc;
	CK (cudaMemcpy (h->d_tw.p, tw.data (), sizeof (float2) * tw.size (), cudaMemcpyHostToDevice));

	// odd taps for the direct-form small-call path
	rc = h->d_g.ensure (sizeof (float) * (size_t)Lh);
	if (rc) return rc;
	CK (cudaMemcpy (h->d_g.p, g.data (), sizeof (float) * (size_t)Lh, cudaMemcpyHostToDevice));
	return PHASEROT_OK;
}

void
fill_conv_common (phaserot* h, ConvParams& p)
{
	memset (&p, 0, sizeof (p));
	p.plane        = (const float2*)h->d_plane.p;
	p.plane_stride = h->plane_stride;
	p.padf         = h->padf;
	p.G            = (const float2*)h->d_G.p;
	p.tw1          = (const float2*)h->d_tw.p;
	p.tw2          = p.tw1 + kTwP1Rows * 512;
	p.Lh           = h->Lp;
	p.V            = h->V;
	p.dl           = h->Lh / 2;
	p.hist_frames  = h->L;
	p.G1           = (const float2*)h->d_G1.p;
	p.scratch      = (float4*)h->d_scratch.p;
	p.seg_stride   = 1;
	p.prefetch     = getenv ("PHASEROT_PREFETCH") ? atoi (getenv ("PHASEROT_PREFETCH")) : 0;
}

// Extent of a pass over F frames followed by `flush_blocks` zero blocks: output samples t < t_end, complex
// outputs m < m_end in nseg FFT segments; with the first-block rule (cli:418-419) m < m_skip is not examined
// and the direct branch is zero for m < m_zero.
struct StreamGeom {
	long long t_end, m_end, nseg, m_skip, m_zero;
	// points a pass over nchan channels examines, G per output sample (true-peak: the sample and OS interpolated points)
	uint64_t points (int nchan, int G) const { return (uint64_t)nchan * (uint64_t)(2 * (m_end - m_skip)) * (uint64_t)G; }
};
StreamGeom
stream_geom (const phaserot* h, long long F, int flush_blocks, bool first_block)
{
	StreamGeom g;
	g.t_end         = ((F + h->L - 1) / h->L + flush_blocks) * h->L;
	g.m_end         = (g.t_end + 1) / 2;
	g.nseg          = (g.m_end + h->V - 1) / h->V;
	const bool rule = first_block && !(h->cfg.flags & PHASEROT_FLAG_NO_FIRST_BLOCK_QUIRK);
	g.m_skip        = rule ? h->Lh / 2 : 0;
	g.m_zero        = rule ? h->Lh : 0;
	return g;
}

// ConvParams of an analysis pass (EPI_POINTS, EPI_HILBERT, EPI_SECT_POINTS) over F interleaved frames at `inter`
// (`hist`: frames [-L, 0) or null), channels [c0, c0 + nchan): survivors of the radius thr2 go to `list`, rows of
// `cap` points counted in `count`
ConvParams
analysis_params (phaserot* h, const float* inter, const float* hist, long long F, const StreamGeom& g, int c0, int nchan, float2* list, long long cap,
                 unsigned* count, unsigned* overflow, const float* thr2, unsigned* rawpeak)
{
	ConvParams p;
	fill_conv_common (h, p);
	p.inter       = inter;
	p.hist        = hist;
	p.n_frames    = F;
	p.C           = h->C;
	p.chan0       = c0;
	p.nchan       = nchan;
	p.m_end       = g.m_end;
	p.m_skip      = g.m_skip;
	p.m_zero      = g.m_zero;
	p.list        = list;
	p.list_stride = cap;
	p.list_cap    = (unsigned)cap;
	p.count       = count;
	p.overflow    = overflow;
	p.thr2        = thr2;
	p.rawpeak     = rawpeak;
	return p;
}

// The true-peak pass over what the analysis pass `p` reads and lists: p's Hilbert branch goes compact to the
// staging H ([channel][h_stride], kTpCarry carried samples first), and truepeak_kernel reads it from there
TpParams
tp_params (const phaserot* h, ConvParams& p, long long t_end, float* H, long long h_stride)
{
	p.out         = (float2*)H;
	p.out_stride  = h_stride / 2;
	p.out_compact = 1;
	TpParams tp;
	memset (&tp, 0, sizeof (tp));
	tp.inter       = p.inter;
	tp.hist        = p.hist;
	tp.n_frames    = p.n_frames;
	tp.C           = p.C;
	tp.hist_frames = h->L;
	tp.H           = H;
	tp.h_stride    = h_stride;
	tp.chan0       = p.chan0;
	tp.seg0        = p.seg0;
	tp.seg_stride  = p.seg_stride;
	tp.V2          = 2 * h->V;
	tp.D           = h->L / 2;
	tp.t_skip      = 2 * p.m_skip;
	tp.t_zero      = 2 * p.m_zero;
	tp.t_end       = t_end;
	tp.os          = h->OS;
	tp.list        = p.list;
	tp.list_stride = p.list_stride;
	tp.count       = p.count;
	tp.list_cap    = p.list_cap;
	tp.overflow    = p.overflow;
	tp.thr2        = p.thr2;
	tp.rawpeak     = p.rawpeak;
	return tp;
}

// Function attributes are per device (per context): phaserot_create() sets them
// for every kernel that needs more than the default 48 KB of dynamic shared
// memory, once per device, under g_create_lock - never on a launch path (an LV2
// run() must not take locks, and a second handle on another device of the same
// process must find its own opt-in).
template <int EPI, int SRC, int NP>
int
set_conv_attr ()
{
	CK (cudaFuncSetAttribute (fftconv_kernel<EPI, SRC, NP>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBytes));
	if (getenv ("PHASEROT_CARVEOUT")) {
		CK (cudaFuncSetAttribute (fftconv_kernel<EPI, SRC, NP>, cudaFuncAttributePreferredSharedMemoryCarveout, atoi (getenv ("PHASEROT_CARVEOUT"))));
	}
	return PHASEROT_OK;
}

// Only the kernels a handle of this shape can launch are touched: setting an
// attribute loads the kernel's code (CUDA loads modules lazily), and a CLI run on
// a 48 kHz file needs three of the twenty-odd kernels in the library - the rest
// would only add to the process start-up time.  Sections and loudness ask for
// theirs when they are first called (phaserot_create() does not know whether they
// will be).
enum {
	KA_POINTS = 1 << 0, KA_RENDER_INTER = 1 << 1, KA_RENDER_PLANE = 1 << 2, KA_HILBERT = 1 << 3, KA_SECT_POINTS = 1 << 4, KA_SECT_RENDER = 1 << 5,
	KA_FIR_STREAM = 1 << 8
};
// `want`: KA_* bits; the fftconv_kernel bits (the low byte) stand for the instantiation with the handle's NP.
// Caller holds g_create_lock and has made `dev` current.
int
set_device_attrs (int dev, int NP, unsigned want)
{
	static std::vector<unsigned> done; // per device; fftconv_kernel bits of NP = 2 are shifted by 16
	if (done.size () <= (size_t)dev) done.resize ((size_t)dev + 1, 0u);
	if (NP == 2) want = ((want & 0xffu) << 16) | (want & ~0xffu);
	const unsigned todo = want & ~done[(size_t)dev];
	int rc;
	if ((todo & KA_POINTS) && (rc = set_conv_attr<EPI_POINTS, SRC_INTER, 1> ())) return rc;
	if ((todo & (KA_POINTS << 16)) && (rc = set_conv_attr<EPI_POINTS, SRC_INTER, 2> ())) return rc;
	if ((todo & KA_RENDER_INTER) && (rc = set_conv_attr<EPI_RENDER, SRC_INTER, 1> ())) return rc;
	if ((todo & (KA_RENDER_INTER << 16)) && (rc = set_conv_attr<EPI_RENDER, SRC_INTER, 2> ())) return rc;
	if ((todo & KA_RENDER_PLANE) && (rc = set_conv_attr<EPI_RENDER, SRC_PLANE, 1> ())) return rc;
	if ((todo & (KA_RENDER_PLANE << 16)) && (rc = set_conv_attr<EPI_RENDER, SRC_PLANE, 2> ())) return rc;
	if ((todo & KA_HILBERT) && (rc = set_conv_attr<EPI_HILBERT, SRC_INTER, 1> ())) return rc;
	if ((todo & (KA_HILBERT << 16)) && (rc = set_conv_attr<EPI_HILBERT, SRC_INTER, 2> ())) return rc;
	if ((todo & KA_SECT_POINTS) && (rc = set_conv_attr<EPI_SECT_POINTS, SRC_INTER, 1> ())) return rc;
	if ((todo & (KA_SECT_POINTS << 16)) && (rc = set_conv_attr<EPI_SECT_POINTS, SRC_INTER, 2> ())) return rc;
	if ((todo & KA_SECT_RENDER) && (rc = set_conv_attr<EPI_SECT_RENDER, SRC_INTER, 1> ())) return rc;
	if ((todo & (KA_SECT_RENDER << 16)) && (rc = set_conv_attr<EPI_SECT_RENDER, SRC_INTER, 2> ())) return rc;
	if (todo & KA_FIR_STREAM) {
		CK (cudaFuncSetAttribute (fir_stream_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 96 * 1024));
	}
	done[(size_t)dev] |= want;
	return PHASEROT_OK;
}

// the same from a call that has not taken g_create_lock (sections, loudness: never a plugin run())
int
load_kernels (phaserot* h, unsigned want)
{
	std::lock_guard<std::mutex> lk (g_create_lock);
	return set_device_attrs (h->dev, h->NP, want);
}

template <int EPI, int SRC, int NP>
int
launch_conv_np (phaserot* h, const ConvParams& p)
{
	const long long total = p.nseg * p.nchan;
	if (total <= 0) {
		return PHASEROT_OK;
	}
	const int grid = (int)std::min<long long> (total, h->n_sm);
	ProfScope ps (h, epi_points (EPI) ? 0 : EPI == EPI_HILBERT ? 6 : 3);
	fftconv_kernel<EPI, SRC, NP><<<grid, kConvThreads, kSmemBytes, h->stream>>> (p);
	CK (cudaGetLastError ());
	++h->stats.kernel_launches;
	return PHASEROT_OK;
}

template <int EPI, int SRC = SRC_PLANE>
int
launch_conv (phaserot* h, const ConvParams& p)
{
	return h->NP == 2 ? launch_conv_np<EPI, SRC, 2> (h, p) : launch_conv_np<EPI, SRC, 1> (h, p);
}

// true-peak: the last kTpCarry samples of a launch's Hilbert branch (n_samples per channel in the staging H) move
// to the front of the staging rows of channels [ch0, ch0 + nch), where the next launch's interpolator reads them
int
launch_tp_carry (phaserot* h, float* H, long long stride, int ch0, int nch, long long n_samples)
{
	ProfScope ps (h, 5);
	tp_carry_kernel<<<nch, 32, 0, h->stream>>> (H, stride, ch0, n_samples);
	CK (cudaGetLastError ());
	++h->stats.kernel_launches;
	return PHASEROT_OK;
}

// true-peak: the carry of channels [ch0, ch0 + nch) for a launch from segment s0 on (the interpolator reaches
// 11 samples back).  At the start of a stream without history it is silence; otherwise one extra segment of
// `p`'s Hilbert branch ending there seeds it (before the stream start it reads history only: with L frames its
// last samples lack taps L-16.. of the window edge, which are below 1e-9 (Hann), far inside fp32 rounding of H).
int
seed_tp_carry (phaserot* h, ConvParams& p, float* H, long long stride, long long s0, int ch0, int nch)
{
	if (s0 == 0 && !p.hist) {
		for (int c = ch0; c < ch0 + nch; ++c) CK (cudaMemsetAsync (H + (long long)c * stride, 0, sizeof (float) * kTpCarry, h->stream));
		return PHASEROT_OK;
	}
	p.chan0      = ch0;
	p.nchan      = nch;
	p.seg0       = s0 - 1;
	p.seg_stride = 1;
	p.nseg       = 1;
	const int rc = launch_conv<EPI_HILBERT, SRC_INTER> (h, p);
	if (rc) return rc;
	return launch_tp_carry (h, H, stride, ch0, nch, 2 * h->V);
}

// plane geometry for `m_end` complex outputs per channel
int
ensure_planes (phaserot* h, long long m_end, long long* nseg_out)
{
	const long long nseg   = (m_end + h->V - 1) / h->V;
	const long long elems  = h->padf + nseg * h->V + 8;
	const long long stride = (elems + 3) & ~3LL;
	const int rc = h->d_plane.ensure ((size_t)stride * h->C * sizeof (float2));
	if (rc) return rc;
	h->plane_stride = stride;
	*nseg_out       = nseg;
	return PHASEROT_OK;
}

int
launch_deinterleave (phaserot* h, const float* d_in, long long frame0, long long n_frames_total, long long n_first, long long n_count)
{
	if (n_count <= 0) {
		return PHASEROT_OK;
	}
	const int       nt = 256;
	const long long nb = (n_count + nt - 1) / nt;
	ProfScope       ps (h, 2);
	deinterleave_kernel<<<(unsigned)nb, nt, 0, h->stream>>> (d_in, frame0, n_frames_total, n_first, n_count, h->C,
	                                                          (float2*)h->d_plane.p, h->plane_stride, h->padf);
	CK (cudaGetLastError ());
	++h->stats.kernel_launches;
	return PHASEROT_OK;
}

// zero (or fill from `hist_frames`: L frames, interleaved, host) the front pad
int
init_front_pad (phaserot* h, const float* hist_frames)
{
	for (int c = 0; c < h->C; ++c) {
		CK (cudaMemsetAsync ((float2*)h->d_plane.p + (long long)c * h->plane_stride, 0, sizeof (float2) * (size_t)h->padf, h->stream));
	}
	if (hist_frames) {
		// history occupies complex indices [-Lh, 0)
		int rc = h->h_io.ensure (sizeof (float) * (size_t)h->L * h->C);
		if (rc) return rc;
		float* st = (float*)h->h_io.p;
		for (int c = 0; c < h->C; ++c) {
			for (int i = 0; i < h->L; ++i) {
				st[(size_t)c * h->L + i] = hist_frames[(size_t)i * h->C + c];
			}
			CK (cudaMemcpyAsync ((float2*)h->d_plane.p + (long long)c * h->plane_stride + h->padf - h->Lh, st + (size_t)c * h->L,
			                     sizeof (float) * (size_t)h->L, cudaMemcpyHostToDevice, h->stream));
		}
		CK (cudaStreamSynchronize (h->stream)); // staging buffer is reused
	}
	return PHASEROT_OK;
}

// bootstrap gate of the digital sweep: keep points with r^2 >= kBootBeta * (largest r^2 seen), i.e. r >= 0.8 r_max
constexpr float kBootBeta = 0.64f;
// Points per channel the bootstrap wave may put on the list.  It must hold what the gate passes on ordinary
// material (the list fills in arrival order: a list that is too small keeps the early, weak points - the gate is
// still low then - and the main passes start from poor peaks); on constant-envelope material the gate passes
// every point of the wave and this cap bounds the brute-force sweep of the bootstrap to ~0.2 ms.
constexpr long long kBootCap = 1 << 20;

inline bool OS_is_digital (const phaserot* h) { return h->OS <= 1; }

struct SweepCfg {
	int nt, R, gy;
};
SweepCfg
pick_sweep_cfg (int A)
{
	SweepCfg best { 256, 8, (A + 2047) / 2048 };
	long long best_slots = (long long)best.gy * 2048;
	for (int R : { 1, 2, 4, 8 }) {
		for (int nt : { 128, 192, 256 }) {
			const int per = nt * R;
			const int gy  = (A + per - 1) / per;
			if (gy > 1 && R < 8) {
				continue; // prefer more angles per thread over re-reading the points
			}
			const long long slots = (long long)gy * per;
			if (slots < best_slots || (slots == best_slots && gy < best.gy)) {
				best       = { nt, R, gy };
				best_slots = slots;
			}
		}
	}
	return best;
}

// Launches a sweep-family kernel (angles in lanes over survivor lists: sweep_kernel, overs_kernel) over `rows`
// rows of A angles: launch (R, grid, threads), R a std::integral_constant of the angles per thread
template <class Launch>
void
dispatch_sweep (const phaserot* h, int A, int rows, Launch&& launch)
{
	const SweepCfg  sc = pick_sweep_cfg (A);
	const long long gx = std::max<long long> (1, (h->n_sm * 8) / std::max<long long> (1, (long long)sc.gy * rows));
	const dim3      grid ((unsigned)gx, (unsigned)sc.gy, (unsigned)rows);
	switch (sc.R) {
		case 1: launch (std::integral_constant<int, 1> (), grid, sc.nt); break;
		case 2: launch (std::integral_constant<int, 2> (), grid, sc.nt); break;
		case 4: launch (std::integral_constant<int, 4> (), grid, sc.nt); break;
		default: launch (std::integral_constant<int, 8> (), grid, sc.nt); break;
	}
}

// Every angle of d_cs over the survivor lists of `rows` rows from row0 on (list, count: [row]), into
// table [row][A] with a running max.  A bootstrap list is swept even when its count ran past cap (the
// excess was dropped); any other flagged row is repeated in dense mode, so its full list is skipped.
int
launch_sweep (phaserot* h, const float2* lst, long long list_stride, const unsigned* count, unsigned cap, bool boot, int row0, int rows, int A,
              unsigned* table, unsigned long long* n_eval)
{
	if (A == 0) return PHASEROT_OK;
	const float2* cs = (const float2*)h->d_cs.p;
	const int     so = boot ? 0 : 1;
	ProfScope     ps (h, 1);
	dispatch_sweep (h, A, rows, [&] (auto R, dim3 grid, int nt) {
		sweep_kernel<decltype (R)::value><<<grid, nt, 0, h->stream>>> (lst, list_stride, count, cap, so, row0, cs, A, table, A, n_eval);
	});
	CK (cudaGetLastError ());
	++h->stats.kernel_launches;
	return PHASEROT_OK;
}

// Contiguous launches of a sweep: the first has PHASEROT_SEGS_FIRST segments per CTA, the following ones up to
// PHASEROT_SEGS_MULT times that (measurement aids, defaults 8 and 16)
struct SegsKnobs {
	int first = getenv ("PHASEROT_SEGS_FIRST") ? std::max (1, atoi (getenv ("PHASEROT_SEGS_FIRST"))) : 8;
	int mult  = getenv ("PHASEROT_SEGS_MULT") ? std::max (1, atoi (getenv ("PHASEROT_SEGS_MULT"))) : 16;
};

// Segments per channel of the next contiguous launch (n_main launches so far, seg_done of nseg segments done).
// The first launch has segs_first as a refresh of the radius - unless what would be left for the second
// launch is less than that and `merge_short_rest` (short streams, shards of a strong-scaling run): then
// everything goes into one launch and a launch + sweep round trip (~35 us) is saved.
long long
next_launch_segs (int n_main, long long seg_done, long long nseg, long long segs_first, long long segs_max, bool merge_short_rest)
{
	const bool short_rest = merge_short_rest && nseg - seg_done <= 2 * segs_first;
	return (n_main == 0 && !short_rest) ? segs_first : segs_max;
}

// Launch sizes and survivor-list capacity of a pass over nseg segments per channel of nchan channels.
struct ListPlan {
	long long ppseg;                // points a segment can put on the list (true-peak: the sample and OS interpolated points)
	long long segs_first, segs_max; // segments per channel of the first contiguous launch and of the following ones
	long long cap;                  // points per channel the list holds
	long long segs_cap;             // segments per channel of the largest launch
};
ListPlan
plan_lists (const phaserot* h, int nchan, long long nseg, bool on_device, bool dense)
{
	// (8 segments per CTA; device-resident digital-peak input: up to 128 from the
	// second contiguous launch on - by then the radius is close to final, a launch
	// leaves a few dozen survivors, and every launch + sweep saved is ~20 us: an hour
	// of stereo is bootstrap + 2 launches.  The list is sized by the stream, at most
	// 3.7 GB.  Host input keeps 8, so that little work is left when the last chunk
	// has landed.)
	static const SegsKnobs knobs;
	ListPlan lp;
	lp.ppseg      = (long long)h->V * 2 * (h->OS > 1 ? h->OS + 1 : 1);
	lp.segs_first = std::max<long long> (1, ((long long)h->n_sm * knobs.first) / nchan);
	lp.segs_max   = !on_device ? lp.segs_first : (OS_is_digital (h) ? knobs.mult : 2) * lp.segs_first;
	// Survivor list, sized by demand.  Normal mode: 1/32 of the points of the
	// largest launch (pruning leaves 1e-4 .. 1e-5 of them on programme material), at
	// least 1 M points per channel; a list that overflows flags the pass and
	// complete_pending() repeats it in dense mode.  Dense mode (and NO_PRUNE, where
	// every point goes on the list): at most kDenseCap points per channel (4 M .. 48 M), and the
	// launches are sized to it, so nothing can overflow.
	// (the list and the wide list: 16 bytes per point and channel; 2 GB between them, 48 M points for stereo)
	const long long kDenseCap = std::min<long long> (48LL << 20, std::max<long long> (4LL << 20, (2LL << 30) / (16LL * std::max (1, nchan))));
	if (dense) {
		const long long fit = std::max<long long> (1, kDenseCap / lp.ppseg);
		lp.segs_first       = std::min (lp.segs_first, fit);
		lp.segs_max         = std::min (lp.segs_max, fit);
		lp.cap              = std::min (std::max (lp.segs_first, lp.segs_max), std::max<long long> (nseg, 1)) * lp.ppseg;
	} else {
		const long long full = std::min (std::max (lp.segs_first, lp.segs_max), std::max<long long> (nseg, 1)) * lp.ppseg;
		// (at least one wave: a stream too short for the bootstrap starts with an unpruned wave that lists every point)
		const long long wave_pts = std::max<long long> (1, (h->n_sm + nchan - 1) / nchan) * lp.ppseg;
		lp.cap                   = std::min (full, std::max ({ 1LL << 20, full / 32, wave_pts }));
	}
	lp.segs_cap = std::min (std::max (lp.segs_first, lp.segs_max), std::max<long long> (nseg, 1));
	return lp;
}

enum class Pass {
	Fresh,    // a new pass: the pending one is finished first, the device table starts empty, bootstrap included
	BootOnly, // Fresh, but only the bootstrap wave and its sweep are enqueued (two-phase sharded sweep)
	Continue, // the pending pass again, on its device table without a bootstrap: dense-mode repeat, or the rest of BootOnly
};
int sweep_core (phaserot* h, SweepJob job, Pass pass);

// Repeats the pending sweep in dense mode on top of the table reached so far (a running maximum only
// grows, and every point evaluated was a real one).  Dense launches are sized to the list, so the repeat
// cannot overflow.  `evaluated`: points the overflowed attempt evaluated.
int
repeat_dense (phaserot* h, unsigned long long evaluated)
{
	h->stats.points_evaluated += evaluated;
	h->dense_mode  = true;
	h->pend_redone = true;
	++h->stats.dense_repeats;
	return sweep_core (h, h->redo, Pass::Continue);
}

// The pending sweep is complete on the device when this returns: waits for it and,
// if a survivor list overflowed (material where most samples survive the radius
// filter), repeats the pass in dense mode.
int
complete_pending (phaserot* h)
{
	if (!h->pending) {
		return PHASEROT_OK;
	}
	int rc = h->h_res.ensure (64);
	if (rc) return rc;
	for (int attempt = 0; attempt < 2; ++attempt) {
		unsigned long long* st = (unsigned long long*)h->h_res.p;
		CK (cudaMemcpyAsync (st, d_stats (h), 2 * sizeof (unsigned long long), cudaMemcpyDeviceToHost, h->stream));
		CK (cudaMemcpyAsync (st + 2, d_overflow (h), sizeof (unsigned), cudaMemcpyDeviceToHost, h->stream));
		CK (cudaStreamSynchronize (h->stream));
		if (getenv ("PHASEROT_DEBUG")) {
			fprintf (stderr, "[phaserot] complete (attempt %d): listed %llu evaluated %llu overflow %llx dense %d cap %lld\n", attempt, st[0], st[1], st[2],
			         (int)h->dense_mode, h->list_cap);
		}
		if ((unsigned)st[2] == 0) {
			return PHASEROT_OK;
		}
		if (attempt == 1 || h->dense_mode) {
			snprintf (g_last_error, sizeof (g_last_error), "survivor list overflow in dense mode");
			return PHASEROT_E_CUDA; // cannot happen: dense launches are sized to the list
		}
		rc = repeat_dense (h, st[1]);
		if (rc) return rc;
	}
	return PHASEROT_OK;
}

// Running max of one row of a device sweep table (maxima in the order of the angle schedule idx) into a
// row of the host grid (PhaseRotate::_peak).  Grid index 0 also takes the raw input peak, if any.
void
merge_row (float* row, const float* tab, const std::vector<int>& idx, const float* raw)
{
	for (size_t k = 0; k < idx.size (); ++k) {
		const int a = idx[k];
		row[a]      = std::max (row[a], tab[k]);
	}
	if (raw) row[0] = std::max (row[0], *raw);
}

// merge a finished device sweep into the host table (PhaseRotate::_peak semantics: running max)
int
finish_pending (phaserot* h)
{
	if (!h->pending) {
		return PHASEROT_OK;
	}
	int rc = PHASEROT_OK;
	if (!h->pend_exposed) {
		rc = complete_pending (h); // repeats the pass in dense mode if a list overflowed
		if (rc) return rc;
	}
	const int    A     = h->pend_A;
	// [C][A] maxima | [C] raw peaks | overflow flag | pad to 8 bytes | 2 x u64 statistics
	const size_t n_tab = (size_t)A * h->C + (size_t)h->C + 1;
	const size_t n_pad = n_tab + (n_tab & 1);
	const size_t bytes = sizeof (unsigned) * n_pad + 2 * sizeof (unsigned long long);
	rc                 = h->h_res.ensure (bytes);
	if (rc) return rc;
	unsigned* res = (unsigned*)h->h_res.p;
	if (A > 0) {
		CK (cudaMemcpyAsync (res, h->d_peaks.p, sizeof (unsigned) * n_tab, cudaMemcpyDeviceToHost, h->stream));
	} else {
		CK (cudaMemcpyAsync (res, d_raw (h), sizeof (unsigned) * ((size_t)h->C + 1), cudaMemcpyDeviceToHost, h->stream));
	}
	unsigned long long* st = (unsigned long long*)(res + n_pad);
	CK (cudaMemcpyAsync (st, d_stats (h), 2 * sizeof (unsigned long long), cudaMemcpyDeviceToHost, h->stream));
	CK (cudaStreamSynchronize (h->stream));
	prof_resolve (h);
	h->stats.d2h_bytes += bytes;
	if (res[n_tab - 1] != 0) {
		// Only reachable for a table that was handed out (phaserot_pending_table) and combined by the
		// caller: this shard, or - the flag is part of the reduced buffer - some other rank's, overflowed
		// its survivor list.  Every rank sees the same flag: each repeats its shard in dense mode on top of
		// the combined table (a running maximum) and the caller reduces once more.
		if (h->pend_again >= 2) {
			snprintf (g_last_error, sizeof (g_last_error), "survivor list overflow flag still set after a dense repeat");
			return PHASEROT_E_CUDA; // cannot happen: dense launches are sized to the list
		}
		++h->pend_again;
		if (h->dense_mode && !h->pend_redone) {
			// this rank's shard ran in dense mode and is complete; it was another rank's flag.  Clear the word
			// and take part in the second reduction with the table as it is.
			CK (cudaMemsetAsync (d_overflow (h), 0, sizeof (unsigned), h->stream));
			return PHASEROT_E_AGAIN;
		}
		rc = repeat_dense (h, st[1]);
		if (rc) return rc;
		return PHASEROT_E_AGAIN;
	}
	const float* tab = (const float*)res; // float bits
	for (int c = h->pend_c0; c < h->pend_c1; ++c) {
		merge_row (h->table.data () + (size_t)c * h->MS, tab + (size_t)c * A, h->pend_idx, h->pend_raw ? tab + (size_t)A * h->C + c : nullptr);
	}
	h->stats.points_evaluated += st[1];
	if (getenv ("PHASEROT_DEBUG")) {
		fprintf (stderr, "[phaserot] finish: listed %llu evaluated %llu points %llu dense %d cap %lld\n", st[0], st[1],
		         (unsigned long long)h->pend_points, (int)h->dense_mode, h->list_cap);
	}
	// leave dense mode when the material no longer needs it (the list stayed far below the normal capacity)
	// (judged on a dense pass that started from an empty table: a repeat starts from the peaks of the failed attempt and lists little)
	if (h->dense_mode && !h->pend_redone && !(h->cfg.flags & PHASEROT_FLAG_NO_PRUNE) && h->pend_points > 0 && (double)st[0] < 1e-3 * (double)h->pend_points) { // st[0]: points the lists held
		h->dense_mode = false;
	}
	else if (!h->dense_mode && !(h->cfg.flags & PHASEROT_FLAG_NO_PRUNE) && h->pend_points >= (4ull << 20) && (double)st[1] > 5e-3 * (double)h->pend_points) {
		// Few-tone material below the overflow limit (config 1's two tones: 1 % of the samples survive the radius
		// filter): in normal mode every survivor was swept at every angle (st[1]).  The next sweep of this handle
		// starts dense - windows instead of every angle - and stays so while its lists hold more than 0.1 % of the
		// samples.  A mode of execution only: the table is the same bit for bit either way.
		h->dense_mode = true;
	}
	h->pending      = false;
	h->pend_exposed = false;
	return PHASEROT_OK;
}

// The angle loop of PhaseRotate::thr_process (cli/phase-rotate.cc:409-428).
int
angle_schedule (phaserot* h, int ang_start, int ang_end, int ang_stride, std::vector<int>& idx, bool& raw)
{
	if (ang_stride < 1) {
		return PHASEROT_E_INVAL;
	}
	std::vector<char> seen ((size_t)h->MS, 0);
	idx.clear ();
	raw       = false;
	int angle = ang_start;
	while (angle <= ang_end) {
		if (angle == 0) {
			raw = true; // cli:413-414: raw input peak
		} else {
			const int a = ((angle % h->MS) + h->MS) % h->MS;
			if (!seen[(size_t)a]) {
				seen[(size_t)a] = 1;
				idx.push_back (a);
			}
		}
		angle += ang_stride;
		if (angle >= ang_end) {
			break;
		}
	}
	return PHASEROT_OK;
}

// bytes per sample of a host stream in PHASEROT_PCM_* format
size_t
pcm_bytes (int fmt)
{
	return fmt == PHASEROT_PCM_S16 ? 2 : fmt == PHASEROT_PCM_S24 ? 3 : 4;
}

// (cos, sin) of every angle of the schedule to d_cs, staged through a pinned buffer of the handle: no
// synchronisation (the caller has waited for the stream's previous pass)
int
upload_angle_table (phaserot* h, const std::vector<int>& idx)
{
	const size_t n  = std::max<size_t> (idx.size (), 1);
	int          rc = h->d_cs.ensure (sizeof (float2) * n);
	if (rc) return rc;
	rc = h->h_cs.ensure (sizeof (float2) * n);
	if (rc) return rc;
	float2* cs = (float2*)h->h_cs.p;
	for (size_t k = 0; k < idx.size (); ++k) cs[k] = make_float2 (h->lut_c[(size_t)idx[k]], h->lut_s[(size_t)idx[k]]);
	CK (cudaMemcpyAsync (h->d_cs.p, cs, sizeof (float2) * idx.size (), cudaMemcpyHostToDevice, h->stream));
	return PHASEROT_OK;
}

// (cos, sin) of a full-circle angle a: a + MS renders the negation of a, so it is the LUT pair of
// a mod MS, negated for odd half turns
float2
full_circle_cs (const phaserot* h, long long a)
{
	const long long q  = (a >= 0 ? a : a - h->MS + 1) / h->MS;
	const size_t    i  = (size_t)(a - q * h->MS);
	const float     sg = (q & 1) ? -1.f : 1.f;
	return make_float2 (sg * h->lut_c[i], sg * h->lut_s[i]);
}

// H2D of a host stream into d_inter (allocated by the caller) in chunks on the copy stream, integer PCM
// widened there; the compute stream waits for each chunk, and `landed (frames)` runs after every chunk
// but the last, so that the caller can start on the frames that have landed.
template <class Landed>
int
upload_chunks (phaserot* h, const void* src, int fmt, long long n_frames, Landed&& landed)
{
	int rc = PHASEROT_OK;
	const long long chunk_frames = std::max<long long> (4, ((8LL << 20) / h->C) & ~3LL); // ~32 MB of floats per chunk; a multiple of 4 frames keeps every chunk 4-byte aligned at 3 bytes per sample
	const size_t    bps          = pcm_bytes (fmt);
	const bool      widen        = fmt != PHASEROT_PCM_F32; // integer PCM: conversion pass on the copy stream
	cudaPointerAttributes at;
	const bool pinned = (cudaPointerGetAttributes (&at, src) == cudaSuccess) && (at.type == cudaMemoryTypeHost);
	cudaGetLastError ();
	if (!pinned) {
		for (int b = 0; b < 2; ++b) {
			rc = h->h_stage[b].ensure (bps * (size_t)std::min (chunk_frames, std::max<long long> (n_frames, 4)) * h->C); // short files: small staging (pinned allocation costs ~0.3 ms per MB)
			if (rc) return rc;
		}
	}
	if (widen) {
		// integer PCM: raw chunk -> device staging -> pcm_to_float_kernel on the copy
		// stream -> the float copy of the file; staging buffer b is reused two chunks
		// later on the same stream, i.e. after the kernel that read it
		for (int b = 0; b < 2; ++b) {
			rc = h->d_stage[b].ensure (bps * (size_t)std::min (chunk_frames, std::max<long long> (n_frames, 4)) * h->C);
			if (rc) return rc;
		}
	}
	// the previous pass may still be reading d_inter on the compute stream
	CK (cudaEventRecord (h->ev_done[0], h->stream));
	CK (cudaStreamWaitEvent (h->copy_stream, h->ev_done[0], 0));
	int       b  = 0;
	long long f0 = 0;
	bool      used[2] = { false, false };
	while (f0 < n_frames) {
		const long long nf    = std::min (chunk_frames, n_frames - f0);
		const size_t    bytes = bps * (size_t)nf * h->C;
		const void*     hsrc  = (const char*)src + bps * (size_t)f0 * h->C;
		if (!pinned) {
			if (used[b]) {
				CK (cudaEventSynchronize (h->ev_copy[b])); // staging buffer free again
			}
			memcpy (h->h_stage[b].p, hsrc, bytes);
			hsrc = h->h_stage[b].p;
		}
		float* d_chunk = (float*)h->d_inter.p + (size_t)f0 * h->C;
		if (widen) {
			CK (cudaMemcpyAsync (h->d_stage[b].p, hsrc, bytes, cudaMemcpyHostToDevice, h->copy_stream));
			const long long ns = nf * h->C;
			const unsigned  nb = (unsigned)((ns + 1023) / 1024);
			if (fmt == PHASEROT_PCM_S16) {
				pcm_to_float_kernel<int16_t><<<nb, 256, 0, h->copy_stream>>> ((const int16_t*)h->d_stage[b].p, d_chunk, ns);
			} else if (fmt == PHASEROT_PCM_S24) {
				pcm24_to_float_kernel<<<nb, 256, 0, h->copy_stream>>> ((const uint8_t*)h->d_stage[b].p, d_chunk, ns);
			} else {
				pcm_to_float_kernel<int32_t><<<nb, 256, 0, h->copy_stream>>> ((const int32_t*)h->d_stage[b].p, d_chunk, ns);
			}
			CK (cudaGetLastError ());
			++h->stats.kernel_launches;
		} else {
			CK (cudaMemcpyAsync (d_chunk, hsrc, bytes, cudaMemcpyHostToDevice, h->copy_stream));
		}
		CK (cudaEventRecord (h->ev_copy[b], h->copy_stream));
		CK (cudaStreamWaitEvent (h->stream, h->ev_copy[b], 0));
		h->stats.h2d_bytes += bytes;
		used[b] = true;
		f0 += nf;
		if (f0 < n_frames) {
			rc = landed (f0);
			if (rc) return rc;
		}
		b ^= 1;
	}
	return PHASEROT_OK;
}

// The float32 frames of a synchronous analysis pass on the device (*d_x): device input is read in place and
// leaves a pending device sweep alone; host input goes to d_inter, which may still be the source of the
// pending sweep's dense-mode repeat: that sweep is completed first.
int
land_input (phaserot* h, const void* src, bool dev_in, int fmt, long long n_frames, const float** d_x)
{
	if (dev_in) {
		*d_x = (const float*)src;
		return PHASEROT_OK;
	}
	int rc = finish_pending (h);
	if (rc) return rc;
	rc = h->d_inter.ensure (std::max<size_t> (sizeof (float) * (size_t)n_frames * h->C, 16));
	if (rc) return rc;
	rc = upload_chunks (h, src, fmt, n_frames, [] (long long) { return PHASEROT_OK; });
	if (rc) return rc;
	*d_x = (const float*)h->d_inter.p;
	return PHASEROT_OK;
}

// One analysis pass over a stream (see SweepJob and Pass).
int
sweep_core (phaserot* h, SweepJob job, Pass pass)
{
	const bool redo = pass == Pass::Continue;
	if (job.chn >= h->C) {
		return PHASEROT_E_INVAL;
	}
	int rc = redo ? PHASEROT_OK : finish_pending (h); // (the stream is then idle with respect to the previous pass)
	if (rc) return rc;

	std::vector<int> idx;
	bool             raw = false;
	rc                   = angle_schedule (h, job.ang_start, job.ang_end, job.ang_stride, idx, raw);
	if (rc) return rc;
	const int A  = (int)idx.size ();
	const int c0 = job.chn < 0 ? 0 : job.chn;
	const int c1 = job.chn < 0 ? h->C : job.chn + 1;

	rc = h->d_peaks.ensure (sizeof (unsigned) * ((size_t)std::max (A, 1) * h->C + (size_t)h->C + 1));
	if (rc) return rc;
	rc = upload_angle_table (h, idx);
	if (rc) return rc;
	h->pend_A = A; // d_raw() depends on it
	if (!redo) {
		CK (cudaMemsetAsync (h->d_peaks.p, 0, sizeof (unsigned) * ((size_t)std::max (A, 1) * h->C + (size_t)h->C + 1), h->stream));
	} else {
		CK (cudaMemsetAsync (d_overflow (h), 0, sizeof (unsigned), h->stream)); // the repeat starts with a clear flag
	}
	CK (cudaMemsetAsync (h->d_small.p, 0, kSmallBytes, h->stream));
	const bool no_prune = (h->cfg.flags & PHASEROT_FLAG_NO_PRUNE) != 0;
	const bool dense    = h->dense_mode || no_prune; // launches sized to the survivor list
	if (dense && !no_prune && A > 0) {
		// grid index -> slot of the swept angle set, for sweep_window_kernel
		rc = h->h_slot.ensure (sizeof (int) * (size_t)h->MS);
		if (rc) return rc;
		int* so = (int*)h->h_slot.p;
		std::fill (so, so + h->MS, -1);
		for (int k = 0; k < A; ++k) so[idx[(size_t)k]] = k;
		rc = h->d_slot.ensure (sizeof (int) * (size_t)h->MS);
		if (rc) return rc;
		rc = h->d_sec.ensure (sizeof (float) * (size_t)kSectors * h->C);
		if (rc) return rc;
		CK (cudaMemcpyAsync (h->d_slot.p, so, sizeof (int) * (size_t)h->MS, cudaMemcpyHostToDevice, h->stream));
	}

	const StreamGeom g      = stream_geom (h, job.n_frames, job.flush, job.first_block);
	const long long  nseg   = g.nseg;
	const float*     d_hist = nullptr;
	if (const float* hist = job.hist) {
		// frames [-L, 0) of the stream, read by the segments that reach before its start
		cudaPointerAttributes at;
		const bool on_device = cudaPointerGetAttributes (&at, hist) == cudaSuccess && at.type == cudaMemoryTypeDevice;
		cudaGetLastError ();
		if (on_device) {
			d_hist = hist; // read in place (the caller keeps it alive until the table is read back)
		} else {
			rc = h->d_hist.ensure (sizeof (float) * (size_t)h->L * h->C);
			if (rc) return rc;
			CK (cudaMemcpyAsync (h->d_hist.p, hist, sizeof (float) * (size_t)h->L * h->C, cudaMemcpyHostToDevice, h->stream));
			CK (cudaStreamSynchronize (h->stream));
			d_hist = (const float*)h->d_hist.p;
		}
	}

	// survivor list: one launch covers at most `segs_max` segments per channel
	const int       nchan      = c1 - c0;
	const int       OS         = h->OS;
	const ListPlan  lp         = plan_lists (h, nchan, nseg, job.on_device, dense);
	const long long segs_first = lp.segs_first, segs_max = lp.segs_max, cap = lp.cap, segs_cap = lp.segs_cap;
	h->list_stride           = cap;
	h->list_cap              = cap;
	rc                       = h->d_list.ensure ((size_t)h->list_stride * h->C * sizeof (float2));
	if (rc) return rc;
	if (dense && !no_prune && A > 0) {
		rc = h->d_wide.ensure ((size_t)h->list_stride * h->C * sizeof (float2));
		if (rc) return rc;
	}
	if (OS > 1) {
		h->tp_stride = (kTpCarry + segs_cap * h->V * 2 + 3) & ~3LL;
		rc           = h->d_tpH.ensure (sizeof (float) * (size_t)h->tp_stride * h->C);
		if (rc) return rc;
	}
	if (!job.on_device) {
		rc = h->d_inter.ensure (std::max<size_t> (sizeof (float) * (size_t)job.n_frames * h->C, 16));
		if (rc) return rc;
	}

	h->pend_idx = idx;
	h->pend_raw = raw;
	h->pend_c0  = c0;
	h->pend_c1  = c1;
	h->pend_A   = A;

	const float* d_x = job.on_device ? (const float*)job.src : (const float*)h->d_inter.p;
	ConvParams   p   = analysis_params (h, d_x, d_hist, job.n_frames, g, c0, nchan, (float2*)h->d_list.p, h->list_cap, d_count (h), d_overflow (h), d_thr2 (h),
	                                    d_raw (h));
	const int thr_mode = A == 0 ? 2 : (h->cfg.flags & PHASEROT_FLAG_NO_PRUNE) ? 0 : 1;
	if (OS > 1) {
		// true-peak: the radius filter sits in truepeak_kernel and reads thr2 from memory
		threshold_kernel<<<nchan, 32, 0, h->stream>>> ((const unsigned*)h->d_peaks.p, A, A, c0, d_thr2 (h), d_count (h), 1, A == 0 ? 2 : 0);
		CK (cudaGetLastError ());
		++h->stats.kernel_launches;
		p.thr_mode = -1;
	} else {
		// digital peak: the FFT kernel derives the radius from the running peaks in its
		// prologue and zeroes the counters of the list the previous sweep has consumed
		// (two counter sets, alternating by launch), so a steady-state round is two
		// launches: fftconv_kernel, sweep_kernel
		p.thr_mode     = thr_mode;
		p.peaks        = (const unsigned*)h->d_peaks.p;
		p.peaks_stride = A;
		p.A            = A;
		p.r2max        = d_r2max (h);
	}
	int parity = 0;

	long long       frames_ready = 0; // frames of `inter` that are valid on the device
	long long       seg_done     = 0;
	const long long wave     = std::max<long long> (1, (h->n_sm + nchan - 1) / nchan); // segments per channel in one wave
	bool            booted   = thr_mode != 1 || redo; // a repeat starts from the table the first attempt reached
	int             n_main   = 0; // contiguous launches so far

	// true-peak: Hilbert branch of the launch -> staging, carry of the last samples to the next launch
	TpParams tp {};
	if (OS > 1) {
		tp       = tp_params (h, p, g.t_end, (float*)h->d_tpH.p, h->tp_stride);
		tp.r2max = d_r2max (h);
	}

	// every angle over the survivors of one launch.  Normal mode: angles in lanes over the
	// (short) list.  Dense mode: sector thresholds, then one thread per point over the few
	// angles it can still raise (sweep_window_kernel); what that leaves goes angles-in-lanes.
	const float2*       lst    = (const float2*)h->d_list.p;
	unsigned*           table  = (unsigned*)h->d_peaks.p;
	unsigned long long* n_eval = d_stats (h) + 1;
	auto sweep_survivors = [&] (const unsigned* count, unsigned cap, bool boot) -> int {
		if (A == 0) return PHASEROT_OK;
		if (!dense || no_prune || (boot && !h->dense_mode)) {
			return launch_sweep (h, lst, h->list_stride, count, cap, boot, c0, nchan, A, table, n_eval);
		}
		if (boot) {
			// Bootstrap list of a dense handle (up to 1 M points per channel, 0.46 ms at every angle): the running
			// peaks are still zero and every window would be the whole grid, so the head of the list is swept at
			// every angle - and the whole list then goes through the windows like any other, against that table.
			static const unsigned kBootBrute = getenv ("PHASEROT_BOOT_BRUTE") ? (unsigned)atoi (getenv ("PHASEROT_BOOT_BRUTE")) : 128u << 10;
			const int          r          = launch_sweep (h, lst, h->list_stride, count, std::min (cap, kBootBrute), boot, c0, nchan, A, table, n_eval);
			if (r) return r;
		}
		CK (cudaMemsetAsync (d_wide_count (h), 0, sizeof (unsigned) * 64, h->stream));
		WinParams w;
		memset (&w, 0, sizeof (w));
		w.list         = (const float2*)h->d_list.p;
		w.list_stride  = h->list_stride;
		w.count        = count;
		w.cap          = cap;
		w.chan0        = c0;
		w.cs           = (const float2*)h->d_cs.p;
		w.slot_of      = (const int*)h->d_slot.p;
		w.MS           = h->MS;
		w.sec          = (const float*)h->d_sec.p;
		w.peaks        = (unsigned*)h->d_peaks.p;
		w.peaks_stride = A;
		w.wide         = (float2*)h->d_wide.p;
		w.wide_stride  = h->list_stride;
		w.wide_count   = d_wide_count (h);
		w.n_eval       = d_stats (h) + 1;
		w.n_listed     = d_stats (h);
		w.A            = A;
		// a run of consecutive grid indices (the usual full sweep): slot = index - first, no table
		w.slot_base = idx[0];
		for (int k = 1; k < A; ++k) {
			if (idx[(size_t)k] != idx[0] + k) {
				w.slot_base = -1;
				break;
			}
		}
		const size_t wsm = (size_t)A * (sizeof (float2) + sizeof (unsigned));
		w.smem_tables    = wsm <= 40 * 1024; // up to ~3400 angles (0.1 degree grid: 21 KB); finer grids read the tables through L1
		{
			ProfScope ps (h, 1);
			sector_thr_kernel<<<dim3 (kSectors, (unsigned)nchan), 64, 0, h->stream>>> ((const unsigned*)h->d_peaks.p, A, (const int*)h->d_slot.p, h->MS, c0, (float*)h->d_sec.p);
			static const int walk = getenv ("PHASEROT_WALK") ? atoi (getenv ("PHASEROT_WALK")) : 1;
			if (walk && (size_t)A * sizeof (float4) <= 44 * 1024 && w.slot_base >= 0 && A + 2 >= h->MS && A >= 64) { // (nearly) the whole grid: a window around the direction of the point, then walk outwards
				const dim3 wg ((unsigned)(h->n_sm * 8), (unsigned)nchan);
				static const double wrad = getenv ("PHASEROT_WALK_RAD") ? atof (getenv ("PHASEROT_WALK_RAD")) : 5e-3;
				const int  wh = (int)ceil (wrad * h->MS / M_PI); // half width of the first window: 5e-3 rad in grid angles (reaches points up to 7e-6 above the threshold)
				const size_t tsm = (size_t)A * sizeof (float4);
				static const int wsteps = getenv ("PHASEROT_WALK_STEPS") ? atoi (getenv ("PHASEROT_WALK_STEPS")) : 12;
				w.walk_steps     = wsteps;
				if (wh <= 1) sweep_walk_kernel<1><<<wg, 256, tsm, h->stream>>> (w);
				else if (wh <= 2) sweep_walk_kernel<2><<<wg, 256, tsm, h->stream>>> (w);
				else if (wh <= 3) sweep_walk_kernel<3><<<wg, 256, tsm, h->stream>>> (w);
				else if (wh <= 4) sweep_walk_kernel<4><<<wg, 256, tsm, h->stream>>> (w);
				else if (wh <= 6) sweep_walk_kernel<6><<<wg, 256, tsm, h->stream>>> (w);
				else sweep_walk_kernel<8><<<wg, 256, tsm, h->stream>>> (w);
			} else {
				sweep_window_kernel<<<dim3 ((unsigned)(h->n_sm * 8), (unsigned)nchan), 256, w.smem_tables ? wsm : 0, h->stream>>> (w);
			}
		}
		CK (cudaGetLastError ());
		h->stats.kernel_launches += 2;
		return launch_sweep (h, (const float2*)h->d_wide.p, h->list_stride, d_wide_count (h), cap, false, c0, nchan, A, table, n_eval);
	};

	// one conv launch + sweep of its survivors + new filter radius
	auto run_launch = [&] (long long s0, long long stride, long long n, bool boot = false) -> int {
		p.seg0       = s0;
		p.seg_stride = stride;
		p.nseg       = n;
		int r;
		if (OS > 1) {
			p.seg_jitter = boot && stride > 1;
			p.r2max      = boot ? d_r2max (h) : nullptr;
			r = launch_conv<EPI_HILBERT, SRC_INTER> (h, p);
			if (r) return r;
			tp.seg0       = s0;
			tp.seg_stride = stride;
			tp.seg_jitter = p.seg_jitter;
			tp.boot_beta  = boot ? kBootBeta : 0.f;
			tp.list_cap   = boot ? (unsigned)std::min<long long> (h->list_cap, kBootCap) : (unsigned)h->list_cap;
			tp.overflow   = boot ? d_overflow_ignored (h) : d_overflow (h);
			{
				ProfScope  ps (h, 6);
				const dim3 grid ((unsigned)(n * (tp.V2 / kTpTile)), (unsigned)nchan);
				truepeak_kernel<false><<<grid, 256, 0, h->stream>>> (tp);
				CK (cudaGetLastError ());
				++h->stats.kernel_launches;
			}
			if (stride == 1) {
				r = launch_tp_carry (h, (float*)h->d_tpH.p, h->tp_stride, c0, nchan, n * 2 * h->V);
				if (r) return r;
			}
		} else {
			p.count       = parity ? d_count_odd (h) : d_count (h);
			p.count_reset = parity ? d_count (h) : d_count_odd (h);
			p.boot_beta   = boot ? kBootBeta : 0.f;
			p.seg_jitter  = boot && stride > 1;
			// the bootstrap wave only has to raise the running peaks (any subset of its points is
			// valid, the contiguous passes visit the segments again): what does not fit kBootCap
			// points is dropped without flagging the pass
			p.list_cap    = boot ? (unsigned)std::min<long long> (h->list_cap, kBootCap) : (unsigned)h->list_cap;
			p.overflow    = boot ? d_overflow_ignored (h) : d_overflow (h);
			r = launch_conv<EPI_POINTS, SRC_INTER> (h, p);
			if (r) return r;
			r = sweep_survivors (p.count, p.list_cap, boot);
			if (r) return r;
			parity ^= 1;
			return PHASEROT_OK;
		}
		r = sweep_survivors (d_count (h), tp.list_cap, boot);
		if (r) return r;
		{
			ProfScope ps (h, 5);
			threshold_kernel<<<nchan, 256, 0, h->stream>>> ((const unsigned*)h->d_peaks.p, A, A, c0, d_thr2 (h), d_count (h), 1, thr_mode);
		}
		CK (cudaGetLastError ());
		++h->stats.kernel_launches;
		return PHASEROT_OK;
	};

	auto process_ready = [&] (bool final) -> int {
		// a segment reads frames below 2 (s + 1) V
		const long long seg_ready = final ? nseg : std::min (nseg, frames_ready / (2 * (long long)h->V));
		if (!booted && seg_ready >= 2 * wave) {
			// Bootstrap the filter radius from a sparse sample of the segments
			// available so far.  Digital peak: one wave spread over the range (with a
			// pseudo-random offset per segment: a regular grid once locked onto the
			// slow envelope of the programme and saw only its quiet phase), of
			// which only the strongest points (squared radius within kBootBeta of the
			// largest one the launch has seen) are swept - a few hundred well-spread
			// strong points already put every angle's running peak close to its
			// final value.  True-peak: the same wave, gated on the largest H^2 the
			// FFT kernel saw in it.  The main passes below visit these segments
			// again, which is harmless for a running maximum.
			const int r = run_launch (0, seg_ready / wave, wave, true);
			if (r) return r;
			booted = true;
		}
		while (pass != Pass::BootOnly && seg_done < seg_ready) {
			const long long want = !booted ? wave : next_launch_segs (n_main, seg_done, nseg, segs_first, segs_max, job.on_device && final);
			const long long n    = std::min (want, seg_ready - seg_done);
			if (!final && n < want && seg_ready < nseg) {
				break; // wait for more data to keep launches full
			}
			const int r = run_launch (seg_done, 1, n);
			if (r) return r;
			seg_done += n;
			booted = true;
			++n_main;
		}
		return PHASEROT_OK;
	};

	if (OS > 1) {
		rc = seed_tp_carry (h, p, (float*)h->d_tpH.p, h->tp_stride, 0, c0, nchan);
		if (rc) return rc;
	}
	if (job.on_device) {
		frames_ready = job.n_frames;
		rc           = process_ready (true);
		if (rc) return rc;
	} else {
		// H2D in chunks on the copy stream straight into the device copy of the
		// file; the compute stream starts on a chunk as soon as it has landed
		rc = upload_chunks (h, job.src, job.fmt, job.n_frames, [&] (long long f) {
			frames_ready = f;
			return process_ready (false);
		});
		if (rc) return rc;
		rc = process_ready (true);
		if (rc) return rc;
	}
	if (!redo) {
		h->pend_again   = 0;
		h->pend_exposed = false;
		h->pend_redone  = false;
		h->pend_points  = g.points (nchan, OS > 1 ? OS + 1 : 1);
		h->stats.points_total += h->pend_points;
		// the device-resident form of this pass, should it have to be repeated or resumed
		h->redo           = job;
		h->redo.src       = d_x;
		h->redo.on_device = true;
		h->redo.fmt       = PHASEROT_PCM_F32;
		h->redo.hist      = d_hist;
	}
	h->pending = true;
	return PHASEROT_OK;
}

// ---------------------------------------------------------------------------
// Per-section analysis: the rows of the sweep are (section, channel) pairs.
// ---------------------------------------------------------------------------

// sweep_kernel walks the rows with grid.z: at most 65535 (section, channel) rows per call,
// e.g. one hour of 48 kHz stereo in 0.11 s sections or of 8 channels in 0.44 s sections
constexpr long long kMaxSectionRows = 65535;

int
check_sections (phaserot* h, long long n_frames, long long S, int nchan, long long* n_sect)
{
	const long long align = (long long)phaserot_shard_align (h);
	if (n_frames <= 0 || S <= 0 || S % align) {
		snprintf (g_last_error, sizeof (g_last_error), "section length %lld is not a positive multiple of %lld frames", S, align);
		return PHASEROT_E_INVAL;
	}
	*n_sect = (n_frames + S - 1) / S;
	if (*n_sect * nchan > kMaxSectionRows) {
		snprintf (g_last_error, sizeof (g_last_error), "%lld sections x %d channels exceed the limit of %lld section rows", *n_sect, nchan, kMaxSectionRows);
		return PHASEROT_E_INVAL;
	}
	return PHASEROT_OK;
}

/*
 * One analysis pass over a whole stream (the arguments of phaserot_sweep) with a table per section of
 * S frames.  The FFT pass is the one of sweep_core - the same continuous input and segment grid - and
 * only the epilogue's destination follows the section (EPI_SECT_POINTS): every row has its own filter
 * radius, survivor list and table.  Normal mode only: a row whose list overflows is flagged, and its
 * section is repeated afterwards through sweep_core as a shard with history (which has dense mode).
 * Synchronous.
 */
int
sweep_sections_core (phaserot* h, const float* src, bool src_is_device, int fmt, long long n_frames, long long S, int ang_start, int ang_end,
                     int ang_stride, int chn)
{
	if (chn >= h->C) {
		return PHASEROT_E_INVAL;
	}
	if (h->OS > 1) {
		return PHASEROT_E_UNSUPPORTED;
	}
	const int c0    = chn < 0 ? 0 : chn;
	const int c1    = chn < 0 ? h->C : chn + 1;
	const int nchan = c1 - c0;
	long long n_sect;
	int       rc = check_sections (h, n_frames, S, nchan, &n_sect);
	if (rc) return rc;
	std::vector<int> idx;
	bool             raw = false;
	rc                   = angle_schedule (h, ang_start, ang_end, ang_stride, idx, raw);
	if (rc) return rc;
	rc = finish_pending (h); // a pending sweep of the handle's own table completes first
	if (rc) return rc;
	rc = load_kernels (h, KA_SECT_POINTS | KA_SECT_RENDER);
	if (rc) return rc;
	h->sect_n = 0;
	h->sect_redo_k.clear ();
	h->sect_redo.clear ();

	const int        A         = (int)idx.size ();
	const long long  R         = n_sect * nchan;
	const StreamGeom g         = stream_geom (h, n_frames, 1, true); // like phaserot_sweep
	const long long  nseg      = g.nseg;
	const long long  sps       = S / (2 * (long long)h->V); // segments per section
	const long long  last_segs = nseg - (n_sect - 1) * sps;

	// survivor lists, pooled: 1/32 of the points of a row (the largest one: the last section takes the remainder
	// and the flush block), at least 8 K points.  Rows only ever receive points of their own section, so a row's
	// list needs nothing like the 1 M floor of a whole channel.
	const long long cap = std::max<long long> (8192, 2 * (long long)h->V * std::max (sps, last_segs) / 32);
	rc = h->d_list.ensure ((size_t)(R * cap) * sizeof (float2));
	if (rc) return rc;
	const size_t sect_bytes = sizeof (unsigned) * (size_t)(R * std::max (A, 1) + R);
	const size_t aux_bytes  = sizeof (unsigned long long) + sizeof (unsigned) * 5 * (size_t)R;
	rc                      = h->d_sect.ensure (sect_bytes);
	if (rc) return rc;
	rc = h->d_sect_aux.ensure (aux_bytes);
	if (rc) return rc;
	unsigned*           table = (unsigned*)h->d_sect.p;
	unsigned*           rawpk = table + (size_t)R * A;
	unsigned long long* n_ev  = (unsigned long long*)h->d_sect_aux.p;
	float*              thr2  = (float*)(n_ev + 1);
	unsigned*           count = (unsigned*)(thr2 + R);
	unsigned*           ovf   = count + R;
	unsigned*           ovf_b = ovf + R;
	unsigned*           r2max = ovf_b + R;
	CK (cudaMemsetAsync (h->d_sect.p, 0, sect_bytes, h->stream));
	CK (cudaMemsetAsync (h->d_sect_aux.p, 0, aux_bytes, h->stream));
	rc = upload_angle_table (h, idx);
	if (rc) return rc;

	// the bootstrap wave samples every section, so the pass starts once the whole stream has landed
	const float* d_src;
	rc = land_input (h, src, src_is_device, fmt, n_frames, &d_src);
	if (rc) return rc;

	const bool no_prune = (h->cfg.flags & PHASEROT_FLAG_NO_PRUNE) != 0;
	const int  thr_mode = A == 0 ? 2 : no_prune ? 0 : 1;
	ConvParams p        = analysis_params (h, d_src, nullptr, n_frames, g, c0, nchan, (float2*)h->d_list.p, cap, count, ovf, thr2, rawpk);
	p.r2max             = r2max;
	p.sect_segs         = sps;
	p.n_sect            = (int)n_sect;

	// new radius of every row from its running peaks; zeroes the list counters
	auto thresholds = [&] () -> int {
		ProfScope ps (h, 5);
		threshold_kernel<<<(unsigned)R, 256, 0, h->stream>>> (table, A, A, 0, thr2, count, 1, thr_mode);
		CK (cudaGetLastError ());
		++h->stats.kernel_launches;
		return PHASEROT_OK;
	};

	if (thr_mode == 1) {
		// Bootstrap: a quarter of the segments of every section (at least one; more when there are fewer
		// sections than a wave has segments), gated like sweep_core's wave on the largest radius the row
		// has seen.  A whole-stream sweep refreshes its radius between launches; a row is usually done
		// within one contiguous launch, so its radius has to be close to final before it starts (one
		// segment per 10 s section left 40 % of the programme's samples on the lists).  Any subset is
		// valid: the contiguous passes visit these segments again.
		const long long wave = std::max<long long> (1, (h->n_sm + nchan - 1) / nchan);
		rc = thresholds ();
		if (rc) return rc;
		p.sect_boot  = (int)std::min<long long> (std::max ((wave + n_sect - 1) / n_sect, (sps + 3) / 4), sps);
		p.seg0       = 0;
		p.seg_stride = 2; // sparse: no stash reuse between consecutive segments of a CTA
		p.nseg       = n_sect * p.sect_boot;
		p.boot_beta  = kBootBeta;
		p.overflow   = ovf_b; // nobody reads it
		rc = launch_conv<EPI_SECT_POINTS, SRC_INTER> (h, p);
		if (rc) return rc;
		rc = launch_sweep (h, p.list, cap, count, (unsigned)cap, true, 0, (int)R, A, table, n_ev);
		if (rc) return rc;
	}
	// contiguous launches sized like sweep_core's device-resident ones
	p.sect_boot  = 0;
	p.seg_stride = 1;
	p.boot_beta  = 0.f;
	p.overflow   = ovf;
	const ListPlan lp       = plan_lists (h, nchan, nseg, true, false);
	long long      seg_done = 0;
	for (int n_main = 0; seg_done < nseg; ++n_main) {
		const long long n = std::min (next_launch_segs (n_main, seg_done, nseg, lp.segs_first, lp.segs_max, true), nseg - seg_done);
		rc = thresholds ();
		if (rc) return rc;
		p.seg0 = seg_done;
		p.nseg = n;
		rc = launch_conv<EPI_SECT_POINTS, SRC_INTER> (h, p);
		if (rc) return rc;
		rc = launch_sweep (h, p.list, cap, count, (unsigned)cap, false, 0, (int)R, A, table, n_ev); // a flagged row is redone: its full list is skipped
		if (rc) return rc;
		seg_done += n;
	}

	// flagged rows -> sections to repeat
	std::vector<unsigned> flags ((size_t)R);
	unsigned long long    evaluated = 0;
	CK (cudaMemcpyAsync (flags.data (), ovf, sizeof (unsigned) * (size_t)R, cudaMemcpyDeviceToHost, h->stream));
	CK (cudaMemcpyAsync (&evaluated, n_ev, sizeof (evaluated), cudaMemcpyDeviceToHost, h->stream));
	CK (cudaStreamSynchronize (h->stream));
	prof_resolve (h);
	h->stats.points_total += g.points (nchan, 1);
	h->stats.points_evaluated += evaluated;
	h->sect_n   = n_sect;
	h->sect_A   = A;
	h->sect_c0  = c0;
	h->sect_c1  = c1;
	h->sect_raw = raw;
	h->sect_idx = idx;
	for (long long k = 0; k < n_sect; ++k) {
		bool any = false;
		for (int ci = 0; ci < nchan; ++ci) any = any || flags[(size_t)(k * nchan + ci)] != 0;
		if (!any) continue;
		// The shard path with history, in dense mode from the start (its launches are sized to the list), on a
		// zeroed handle table; the handle's own table and mode are restored afterwards.
		const std::vector<float> keep  = h->table;
		const bool               dense = h->dense_mode;
		std::fill (h->table.begin (), h->table.end (), 0.f);
		h->dense_mode       = true;
		const long long f0  = k * S;
		const long long F   = std::min (S, n_frames - f0);
		rc = sweep_core (h, shard_job (d_src + (size_t)f0 * h->C, true, PHASEROT_PCM_F32, F, k ? d_src + (size_t)(f0 - h->L) * h->C : nullptr, k == 0, k == n_sect - 1,
		                               ang_start, ang_end, ang_stride, chn), Pass::Fresh);
		if (!rc) rc = finish_pending (h);
		if (!rc) {
			h->sect_redo_k.push_back (k);
			h->sect_redo.insert (h->sect_redo.end (), h->table.begin (), h->table.end ());
			++h->stats.dense_repeats;
		}
		h->table      = keep;
		h->dense_mode = dense;
		if (rc) {
			h->sect_n = 0;
			return rc;
		}
	}
	return PHASEROT_OK;
}

/*
 * Render with one angle per (section, channel): the fused CLI render of render_core (interleaved in,
 * interleaved out, t_end frames) with EPI_SECT_RENDER, which forms (ca, sa) per sample from the
 * [n_sect][C] angle table.  angles: host [n_sect][C], full circle.
 */
int
render_sections_core (phaserot* h, const float* d_src, long long n_frames, long long t_end, long long S, long long n_sect, const int* angles, float* d_dst)
{
	int rc = load_kernels (h, KA_SECT_POINTS | KA_SECT_RENDER);
	if (rc) return rc;
	const size_t        nrow = (size_t)(n_sect * h->C);
	std::vector<float2> cs (nrow);
	for (size_t r = 0; r < nrow; ++r) cs[r] = full_circle_cs (h, angles[r]);
	rc = h->d_sect_rt.ensure ((sizeof (float2) + sizeof (int)) * nrow);
	if (rc) return rc;
	float2* d_cs  = (float2*)h->d_sect_rt.p;
	int*    d_ang = (int*)(d_cs + nrow);
	CK (cudaMemcpyAsync (d_cs, cs.data (), sizeof (float2) * nrow, cudaMemcpyHostToDevice, h->stream));
	CK (cudaMemcpyAsync (d_ang, angles, sizeof (int) * nrow, cudaMemcpyHostToDevice, h->stream));
	ConvParams p;
	fill_conv_common (h, p);
	p.chan0      = 0;
	p.nchan      = h->C;
	p.seg0       = 0;
	p.m_end      = (t_end + 1) / 2;
	p.nseg       = (p.m_end + h->V - 1) / h->V;
	p.inter      = d_src;
	p.n_frames   = n_frames;
	p.C          = h->C;
	p.out_inter  = d_dst;
	p.out_frames = t_end;
	p.sect_segs  = S / (2 * (long long)h->V);
	p.n_sect     = (int)n_sect;
	p.sect_cs    = d_cs;
	p.sect_ang   = d_ang;
	p.ang_mp     = (float)(2.f * M_PI / h->S / -360.0); // build_lut()
	rc = launch_conv<EPI_SECT_RENDER, SRC_INTER> (h, p);
	if (rc) return rc;
	CK (cudaStreamSynchronize (h->stream)); // the host tables above are about to go
	return PHASEROT_OK;
}

// ---------------------------------------------------------------------------
// Integrated loudness of the rotated output (phaserot_loudness*, loudness.cuh)
// ---------------------------------------------------------------------------

// K-weighting at any rate, derived like libebur128 does; at 48 kHz these are the
// coefficients of BS.1770-4 Tables 1 and 2
KwCoef
kweight_coef (double fs)
{
	KwCoef       k {};
	double       K  = std::tan (M_PI * 1681.974450955533 / fs);
	const double Qs = 0.7071752369554196;
	const double Vh = std::pow (10.0, 3.999843853973347 / 20.0);
	const double Vb = std::pow (Vh, 0.4996667741545416);
	double       a0 = 1.0 + K / Qs + K * K;
	k.b[0][0]       = (Vh + Vb * K / Qs + K * K) / a0;
	k.b[0][1]       = 2.0 * (K * K - Vh) / a0;
	k.b[0][2]       = (Vh - Vb * K / Qs + K * K) / a0;
	k.a[0][0]       = 1.0;
	k.a[0][1]       = 2.0 * (K * K - 1.0) / a0;
	k.a[0][2]       = (1.0 - K / Qs + K * K) / a0;
	K               = std::tan (M_PI * 38.13547087602444 / fs);
	const double Qh = 0.5003270373238773;
	a0              = 1.0 + K / Qh + K * K;
	k.b[1][0]       = 1.0;
	k.b[1][1]       = -2.0;
	k.b[1][2]       = 1.0;
	k.a[1][0]       = 1.0;
	k.a[1][1]       = 2.0 * (K * K - 1.0) / a0;
	k.a[1][2]       = (1.0 - K / Qh + K * K) / a0;
	return k;
}

// P[m - 1] = A^(m N), m = 1 .. 32: A is the zero-input state transition of the K cascade (kw_step)
std::vector<double>
kweight_powers (const KwCoef& k, long long N)
{
	using M4 = std::vector<double>;
	auto mul = [] (const M4& a, const M4& b) {
		M4 r (16, 0.0);
		for (int i = 0; i < 4; ++i)
			for (int j = 0; j < 4; ++j)
				for (int q = 0; q < 4; ++q) r[4 * i + j] += a[4 * i + q] * b[4 * q + j];
		return r;
	};
	M4 A (16, 0.0);
	for (int j = 0; j < 4; ++j) { // column j = one zero-input step from unit state j
		double s[4] = { 0., 0., 0., 0. };
		s[j]            = 1.0;
		const double y1 = s[0];
		const double n0 = -k.a[0][1] * y1 + s[1], n1 = -k.a[0][2] * y1;
		const double y2 = k.b[1][0] * y1 + s[2];
		const double n2 = k.b[1][1] * y1 - k.a[1][1] * y2 + s[3], n3 = k.b[1][2] * y1 - k.a[1][2] * y2;
		A[0 + j] = n0, A[4 + j] = n1, A[8 + j] = n2, A[12 + j] = n3;
	}
	M4 AN (16, 0.0);
	for (int i = 0; i < 4; ++i) AN[5 * i] = 1.0;
	for (long long e = N; e; e >>= 1, A = mul (A, A)) {
		if (e & 1) AN = mul (AN, A);
	}
	std::vector<double> P;
	M4                  Am = AN;
	for (int m = 1; m <= 32; ++m, Am = mul (Am, AN)) P.insert (P.end (), Am.begin (), Am.end ());
	return P;
}

constexpr long long kKwChunk = 4096; // frames per thread of kweight_kernel

/*
 * phaserot_loudness over F frames of interleaved float32 audio on the device.
 *   weights : host [C] or null (1.0)      angles : host [n_sets][C], full circle
 */
int
loudness_core (phaserot* h, const float* d_x, long long F, double fs, const float* weights, const int* angles, int n_sets, double* lufs)
{
	const int       C     = h->C;
	const long long step  = (long long)std::floor (fs / 10.0 + 0.5); // 100 ms sub-block
	const long long n_sub = F / step;
	if (n_sub < 4) { // no complete 400 ms block
		std::fill (lufs, lufs + n_sets, -std::numeric_limits<double>::infinity ());
		return PHASEROT_OK;
	}
	int rc = load_kernels (h, KA_HILBERT); // phaserot_create() loads it for true-peak handles only
	if (rc) return rc;
	const long long Fu       = n_sub * step;                  // samples that lie in a sub-block
	const int       D        = h->L / 2;                      // latency of the render
	const long long T        = Fu + D;                        // K(x) frames the Hilbert branch of t < Fu reads
	const long long n_chunk  = (T + kKwChunk - 1) / kKwChunk;
	const int       nz       = (int)std::min (Fu, step);      // samples of the head correction
	const long long V2       = 2LL * h->V;                    // samples per FFT segment
	const long long nseg     = (T + V2 - 1) / V2;
	const long long segs     = std::min (nseg, std::max<long long> (1, (long long)h->n_sm * 16 / C)); // per FFT launch
	const long long h_stride = (kTpCarry + segs * V2 + 3) & ~3LL;
	const KwCoef    kc       = kweight_coef (fs);

	// fp64 work area
	const size_t n_sums = (size_t)n_sub * C * 3, n_zc = (size_t)C * nz, n_st = (size_t)n_chunk * C * 4;
	rc = h->d_kx.ensure (sizeof (float) * (size_t)T * C);
	if (rc) return rc;
	rc = h->d_lH.ensure (sizeof (float) * (size_t)h_stride * C);
	if (rc) return rc;
	rc = h->d_lwork.ensure (sizeof (double) * (n_sums + n_zc + n_st + 32 * 16 + C + (size_t)n_sets));
	if (rc) return rc;
	rc = h->d_lset.ensure (sizeof (float2) * (size_t)n_sets * C);
	if (rc) return rc;
	double*  d_sums = (double*)h->d_lwork.p;
	double*  d_zc   = d_sums + n_sums;
	KwState* d_st   = (KwState*)(d_zc + n_zc);
	double*  d_P    = d_zc + n_zc + n_st;
	double*  d_G    = d_P + 32 * 16;
	double*  d_lufs = d_G + C;
	float*   d_kx   = (float*)h->d_kx.p;
	float*   d_H    = (float*)h->d_lH.p;

	// rotations of every set, as phaserot_render_sections forms them
	std::vector<float2> cs ((size_t)n_sets * C);
	for (size_t r = 0; r < cs.size (); ++r) cs[r] = full_circle_cs (h, angles[r]);
	std::vector<double> G ((size_t)C, 1.0);
	if (weights) {
		for (int c = 0; c < C; ++c) G[(size_t)c] = weights[c];
	}
	const std::vector<double> P = kweight_powers (kc, kKwChunk);
	CK (cudaMemcpyAsync (h->d_lset.p, cs.data (), sizeof (float2) * cs.size (), cudaMemcpyHostToDevice, h->stream));
	CK (cudaMemcpyAsync (d_P, P.data (), sizeof (double) * P.size (), cudaMemcpyHostToDevice, h->stream));
	CK (cudaMemcpyAsync (d_G, G.data (), sizeof (double) * G.size (), cudaMemcpyHostToDevice, h->stream));
	CK (cudaMemsetAsync (d_sums, 0, sizeof (double) * n_sums, h->stream));

	ConvParams p;
	fill_conv_common (h, p);
	p.C           = C;
	p.chan0       = 0;
	p.nchan       = C;
	p.seg_stride  = 1;
	p.out         = (float2*)d_H;
	p.out_stride  = h_stride / 2;
	p.out_compact = 1;

	// head correction: the Hilbert branch of x itself over its first segment (2 V >= D samples)
	p.inter    = d_x;
	p.n_frames = F;
	p.m_end    = (T + 1) / 2;
	p.seg0     = 0;
	p.nseg     = 1;
	rc         = launch_conv<EPI_HILBERT, SRC_INTER> (h, p);
	if (rc) return rc;
	{
		ProfScope ps (h, 5);
		loudness_head_kernel<<<C, 32, 0, h->stream>>> (d_H, h_stride, D, kc, d_zc, nz);
	}
	CK (cudaGetLastError ());
	++h->stats.kernel_launches;

	// K(x) over [0, T): zero-state chunks, carry, re-run from the carried states
	{
		ProfScope      ps (h, 5);
		const unsigned nb = (unsigned)((n_chunk * C + 255) / 256);
		kweight_kernel<false><<<nb, 256, 0, h->stream>>> (d_x, F, T, C, kKwChunk, kc, d_st, nullptr);
		kweight_carry_kernel<<<C, 32, 0, h->stream>>> (d_st, n_chunk, C, d_P);
		kweight_kernel<true><<<nb, 256, 0, h->stream>>> (d_x, F, T, C, kKwChunk, kc, d_st, d_kx);
	}
	CK (cudaGetLastError ());
	h->stats.kernel_launches += 3;

	// Hilbert branch of K(x), one launch of segments at a time, each consumed by the sums
	p.inter    = d_kx;
	p.n_frames = T;
	for (long long s0 = 0; s0 < nseg; s0 += segs) {
		p.seg0 = s0;
		p.nseg = std::min (segs, nseg - s0);
		rc     = launch_conv<EPI_HILBERT, SRC_INTER> (h, p);
		if (rc) return rc;
		const long long u0 = s0 * V2, lo = std::max (0LL, u0 - D), hi = std::min (Fu, u0 + p.nseg * V2 - D);
		if (lo >= hi) continue;
		const long long j0 = lo / step, j1 = (hi - 1) / step;
		{
			ProfScope ps (h, 5);
			loudness_stats_kernel<<<dim3 ((unsigned)(j1 - j0 + 1), (unsigned)C), 256, 0, h->stream>>> (d_kx, C, d_H, h_stride, u0, D, step, j0, lo, hi, d_zc, nz,
			                                                                                           d_sums);
		}
		CK (cudaGetLastError ());
		++h->stats.kernel_launches;
	}

	{
		ProfScope ps (h, 5);
		loudness_gate_kernel<<<(unsigned)n_sets, 256, 0, h->stream>>> (d_sums, C, n_sub - 3, step, (const float2*)h->d_lset.p, d_G, d_lufs);
	}
	CK (cudaGetLastError ());
	++h->stats.kernel_launches;
	CK (cudaMemcpyAsync (lufs, d_lufs, sizeof (double) * (size_t)n_sets, cudaMemcpyDeviceToHost, h->stream));
	CK (cudaStreamSynchronize (h->stream));
	h->stats.d2h_bytes += sizeof (double) * (size_t)n_sets;
	prof_resolve (h);
	return PHASEROT_OK;
}

// Argument checks of the synchronous analysis entry points: the handle, the audio, its sample format and length,
// then the entry's own (`more`: the first of them that fails, or null).  A failed check sets "<entry>: <check>".
template <class More>
int
check_analysis (const phaserot* h, const void* src, int format, uint64_t n_frames, const char* entry, More&& more)
{
	if (!h) {
		return PHASEROT_E_INVAL;
	}
	if (h->plugin) {
		return PHASEROT_E_STATE;
	}
	const char* bad = nullptr;
	if (!src) bad = "NULL audio";
	else if (format < PHASEROT_PCM_F32 || format > PHASEROT_PCM_S24) bad = "unknown sample format";
	else if (n_frames == 0) bad = "n_frames is 0";
	else bad = more ();
	if (bad) {
		snprintf (g_last_error, sizeof (g_last_error), "%s: %s", entry, bad);
		return PHASEROT_E_INVAL;
	}
	return PHASEROT_OK;
}

int
loudness_entry (phaserot* h, const void* src, bool dev_in, int format, uint64_t n_frames, double fs, const float* weights, const int* angles, int n_sets,
                double* lufs)
{
	int rc = check_analysis (h, src, format, n_frames, "phaserot_loudness", [&] () -> const char* {
		if (!(fs >= 8000.0 && fs <= 768000.0)) return "sample_rate outside [8000, 768000]";
		if (n_sets < 1) return "n_sets < 1";
		if (!angles || !lufs) return "NULL angles or lufs";
		for (int c = 0; weights && c < h->C; ++c) {
			if (!std::isfinite (weights[c]) || weights[c] < 0.f) return "a channel weight is negative or not finite";
		}
		return nullptr;
	});
	if (rc) return rc;
	DevGuard     guard (h->dev);
	const float* d_x;
	rc = land_input (h, src, dev_in, format, (long long)n_frames, &d_x);
	if (rc) return rc;
	return loudness_core (h, d_x, (long long)n_frames, fs, weights, angles, n_sets, lufs);
}

/*
 * Render stream: y[t] = ca x[t - L/2] + sa H[t] for t in [0, t_end).
 *   d_dst_inter == nullptr   planar result left in d_out (float2 per two samples; plugin bulk path)
 *   d_dst_inter != nullptr   fused CLI render: the FFT kernel reads the interleaved frames in place
 *                            and writes interleaved frames [0, t_end) to d_dst_inter (device) - one
 *                            pass over the audio, 8 bytes per sample
 */
int
render_core (phaserot* h, const float* src, bool src_is_device, long long n_frames, long long t_end, const float* hist,
             const float2* chan_cs /*host [C]*/, const float2* ramp /*host [C][ramp_stride] or null*/, long long ramp_stride,
             const int* ramp_len /*host [C] or null*/, long long* m_end_out, float* d_dst_inter = nullptr)
{
	const long long m_end = (t_end + 1) / 2;
	long long       nseg  = (m_end + h->V - 1) / h->V;
	int             rc    = PHASEROT_OK;
	const float*    d_hist = nullptr;
	if (!d_dst_inter) {
		rc = ensure_planes (h, m_end, &nseg);
		if (rc) return rc;
		rc = init_front_pad (h, hist);
		if (rc) return rc;
		h->out_stride = (m_end + 3) & ~3LL;
		rc            = h->d_out.ensure (sizeof (float2) * (size_t)h->out_stride * h->C);
		if (rc) return rc;
	} else if (hist) {
		rc = h->d_hist.ensure (sizeof (float) * (size_t)h->L * h->C);
		if (rc) return rc;
		CK (cudaMemcpyAsync (h->d_hist.p, hist, sizeof (float) * (size_t)h->L * h->C, cudaMemcpyHostToDevice, h->stream));
		d_hist = (const float*)h->d_hist.p;
	}
	rc = h->d_chancs.ensure (sizeof (float2) * (size_t)h->C);
	if (rc) return rc;
	CK (cudaMemcpyAsync (h->d_chancs.p, chan_cs, sizeof (float2) * (size_t)h->C, cudaMemcpyHostToDevice, h->stream));
	if (ramp && ramp_len) {
		rc = h->d_ramp.ensure (sizeof (float2) * (size_t)ramp_stride * h->C);
		if (rc) return rc;
		CK (cudaMemcpyAsync (h->d_ramp.p, ramp, sizeof (float2) * (size_t)ramp_stride * h->C, cudaMemcpyHostToDevice, h->stream));
		CK (cudaMemcpyAsync (d_ramplen (h), ramp_len, sizeof (int) * (size_t)h->C, cudaMemcpyHostToDevice, h->stream));
	}
	CK (cudaStreamSynchronize (h->stream)); // small host arrays above may be stack buffers

	const float* d_src = src;
	if (!src_is_device) {
		const size_t bytes = sizeof (float) * (size_t)n_frames * h->C;
		rc                 = h->d_io.ensure (std::max<size_t> (bytes, 16));
		if (rc) return rc;
		if (bytes) {
			CK (cudaMemcpyAsync (h->d_io.p, src, bytes, cudaMemcpyHostToDevice, h->stream));
			h->stats.h2d_bytes += bytes;
		}
		d_src = (const float*)h->d_io.p;
	}
	if (!d_dst_inter) {
		rc = launch_deinterleave (h, d_src, 0, n_frames, 0, nseg * h->V);
		if (rc) return rc;
	}
	ConvParams p;
	fill_conv_common (h, p);
	p.chan0       = 0;
	p.nchan       = h->C;
	p.seg0        = 0;
	p.nseg        = nseg;
	p.m_end       = m_end;
	p.out         = (float2*)h->d_out.p;
	p.out_stride  = h->out_stride;
	p.cs          = (const float2*)h->d_chancs.p;
	p.ramp        = (ramp && ramp_len) ? (const float2*)h->d_ramp.p : nullptr;
	p.ramp_stride = ramp_stride;
	p.ramp_len    = (ramp && ramp_len) ? d_ramplen (h) : nullptr;
	if (d_dst_inter) {
		p.inter      = d_src;
		p.hist       = d_hist;
		p.n_frames   = n_frames;
		p.C          = h->C;
		p.out_inter  = d_dst_inter;
		p.out_frames = t_end;
		rc           = launch_conv<EPI_RENDER, SRC_INTER> (h, p);
	} else {
		rc = launch_conv<EPI_RENDER> (h, p);
	}
	if (rc) return rc;
	*m_end_out = m_end;
	return PHASEROT_OK;
}

int
launch_interleave (phaserot* h, long long m_count, long long m_first, float* d_dst, long long n_frames_out)
{
	if (m_count <= 0) {
		return PHASEROT_OK;
	}
	const int       nt = 256;
	const long long nb = (m_count + nt - 1) / nt;
	ProfScope       ps (h, 2);
	interleave_kernel<<<(unsigned)nb, nt, 0, h->stream>>> ((const float2*)h->d_out.p + m_first, h->out_stride, h->C, m_count, d_dst, n_frames_out);
	CK (cudaGetLastError ());
	++h->stats.kernel_launches;
	return PHASEROT_OK;
}

int
flush_analyze (phaserot* h)
{
	if (h->an_blocks == 0) {
		return PHASEROT_OK;
	}
	const long long frames = (long long)h->an_blocks * h->L;
	const SweepJob  job { h->an_buf.data (), false, PHASEROT_PCM_F32, frames, 0, h->an_first != 0, h->hist_valid ? h->hist.data () : nullptr,
                         h->an_start, h->an_end, h->an_stride, h->an_chn };
	const int rc = sweep_core (h, job, Pass::Fresh);
	if (rc) return rc;
	// keep the last block as history for a continued stream
	h->hist.assign (h->an_buf.end () - (size_t)h->L * h->C, h->an_buf.end ());
	h->hist_valid = true;
	h->an_buf.clear ();
	h->an_blocks = 0;
	h->an_first  = 0;
	return finish_pending (h);
}

/*
 * phaserot_overs over F frames of interleaved float32 audio on the device: the FFT pass of the sweep with a
 * fixed filter radius T^2 (1 - 1e-5) (a point whose radius is below T cannot be over T at any angle, up to the
 * margin threshold_kernel relies on), the survivors counted by overs_kernel, grid index 0 by overs_raw_kernel.
 * Launches and lists as a device-resident sweep (plan_lists, next_launch_segs); the counters of every launch
 * are kept, and a (launch, channel) whose list overflowed - low ceilings put most points on it - is re-run
 * afterwards in pieces the list holds in full.  Synchronous.  counts / excess: host [C][MS] (excess may be null).
 */
int
overs_core (phaserot* h, const float* d_x, long long F, float T, int ang_start, int ang_end, int ang_stride, int chn, uint64_t* counts, double* excess)
{
	std::vector<int> idx;
	bool             raw = false;
	int              rc  = angle_schedule (h, ang_start, ang_end, ang_stride, idx, raw);
	if (rc) return rc;
	const int        C        = h->C;
	const int        A        = (int)idx.size ();
	const int        c0       = chn < 0 ? 0 : chn;
	const int        c1       = chn < 0 ? C : chn + 1;
	const int        nchan    = c1 - c0;
	const int        OS       = h->OS;
	const int        G        = OS > 1 ? OS + 1 : 1;          // points per record
	const StreamGeom g        = stream_geom (h, F, 1, true); // like phaserot_sweep
	const long long  nseg     = g.nseg;
	const bool       no_prune = (h->cfg.flags & PHASEROT_FLAG_NO_PRUNE) != 0;
	const ListPlan   lp       = plan_lists (h, nchan, nseg, true, no_prune);
	const long long  n_lmax   = nseg / lp.segs_first + 3; // launches of the schedule (+ 1 counter set for the re-runs)

	// work area: u64 counts [C][A] | u64 excess [C][A] | u64 raw counts [C] | u64 raw excess [C] | u64 evaluated |
	// (ca, sa) [A] | thr2 [C] | raw peaks [C] (unused) | overflow word (unused) | list counters [n_lmax][C]
	const size_t n_tab = (size_t)C * A;
	const size_t n_u64 = 2 * n_tab + 2 * (size_t)C + 1;
	const size_t bytes = sizeof (unsigned long long) * n_u64 + sizeof (float2) * (size_t)std::max (A, 1) + sizeof (float) * (2 * (size_t)C + 1) +
	                     sizeof (unsigned) * (size_t)n_lmax * C;
	rc = h->d_ovw.ensure (bytes);
	if (rc) return rc;
	unsigned long long* d_cnt  = (unsigned long long*)h->d_ovw.p;
	unsigned long long* d_exc  = d_cnt + n_tab;
	unsigned long long* d_rcnt = d_exc + n_tab;
	unsigned long long* d_rexc = d_rcnt + C;
	unsigned long long* d_eval = d_rexc + C;
	float2*             d_cs   = (float2*)(d_eval + 1);
	float*              d_thr2 = (float*)(d_cs + std::max (A, 1));
	unsigned*           d_rawp = (unsigned*)(d_thr2 + C);
	unsigned*           d_ovf  = d_rawp + C;
	unsigned*           d_lcnt = d_ovf + 1;
	CK (cudaMemsetAsync (h->d_ovw.p, 0, bytes, h->stream));
	{
		std::vector<float2> cs ((size_t)A);
		for (int k = 0; k < A; ++k) cs[(size_t)k] = make_float2 (h->lut_c[(size_t)idx[(size_t)k]], h->lut_s[(size_t)idx[(size_t)k]]);
		// the margin of threshold_kernel; NO_PRUNE: radius 0, every examined point (true-peak: every sample's group) is listed
		const std::vector<float> thr2 ((size_t)C, no_prune ? 0.f : (T * T) * 0.99999f);
		CK (cudaMemcpyAsync (d_cs, cs.data (), sizeof (float2) * cs.size (), cudaMemcpyHostToDevice, h->stream));
		CK (cudaMemcpyAsync (d_thr2, thr2.data (), sizeof (float) * thr2.size (), cudaMemcpyHostToDevice, h->stream));
	}

	// grid index 0: the raw input (the interpolator reaches 11 frames past the last one)
	if (raw) {
		const long long f_end = std::min (F + (OS > 1 ? 11 : 0), g.t_end - h->L / 2);
		const long long nb    = std::min<long long> ((f_end + 255) / 256, (long long)h->n_sm * 8);
		ProfScope       ps (h, 5);
		overs_raw_kernel<<<dim3 ((unsigned)nb, (unsigned)nchan), 256, 0, h->stream>>> (d_x, F, C, c0, f_end, OS, T, d_rcnt, d_rexc);
		CK (cudaGetLastError ());
		++h->stats.kernel_launches;
	}

	std::vector<unsigned> lcnt;
	std::vector<long long> l_s0, l_n;
	if (A > 0) {
		rc = h->d_ovl.ensure (sizeof (float2) * (size_t)lp.cap * C);
		if (rc) return rc;
		const long long tp_stride = (kTpCarry + lp.segs_cap * 2 * h->V + 3) & ~3LL;
		if (OS > 1) {
			rc = h->d_ovH.ensure (sizeof (float) * (size_t)tp_stride * C);
			if (rc) return rc;
		}
		float*     H = (float*)h->d_ovH.p;
		ConvParams p = analysis_params (h, d_x, nullptr, F, g, c0, nchan, (float2*)h->d_ovl.p, lp.cap, nullptr, d_ovf, d_thr2, d_rawp);
		p.thr_mode   = -1;
		TpParams tp {};
		if (OS > 1) tp = tp_params (h, p, g.t_end, H, tp_stride);
		// segments [s0, s0 + n) of channels [ch0, ch0 + nch): FFT pass -> list (counters `cnt`) -> overs_kernel
		auto run_launch = [&] (long long s0, long long n, int ch0, int nch, unsigned* cnt) -> int {
			p.chan0 = ch0;
			p.nchan = nch;
			p.seg0  = s0;
			p.nseg  = n;
			p.count = cnt;
			int r;
			if (OS > 1) {
				r = launch_conv<EPI_HILBERT, SRC_INTER> (h, p);
				if (r) return r;
				tp.chan0 = ch0;
				tp.seg0  = s0;
				tp.count = cnt;
				{
					ProfScope ps (h, 6);
					truepeak_kernel<true><<<dim3 ((unsigned)(n * (tp.V2 / kTpTile)), (unsigned)nch), 256, 0, h->stream>>> (tp);
					CK (cudaGetLastError ());
					++h->stats.kernel_launches;
				}
				r = launch_tp_carry (h, H, tp_stride, ch0, nch, n * 2 * h->V);
				if (r) return r;
			} else {
				r = launch_conv<EPI_POINTS, SRC_INTER> (h, p);
				if (r) return r;
			}
			const float2*  lst = (const float2*)h->d_ovl.p;
			const unsigned cap = (unsigned)lp.cap;
			ProfScope      ps (h, 1);
			auto overs = [&] (auto G_) {
				dispatch_sweep (h, A, nch, [&] (auto R, dim3 grid, int nt) {
					overs_kernel<decltype (R)::value, decltype (G_)::value><<<grid, nt, 0, h->stream>>> (lst, lp.cap, cnt, cap, ch0, d_cs, A, T, d_cnt, d_exc, d_eval);
				});
			};
			if (G == 1) overs (std::integral_constant<int, 1> ());
			else if (G == 3) overs (std::integral_constant<int, 3> ());
			else overs (std::integral_constant<int, 5> ());
			CK (cudaGetLastError ());
			++h->stats.kernel_launches;
			return PHASEROT_OK;
		};

		// the launches of a device-resident sweep, each with its own list counters
		if (OS > 1) {
			rc = seed_tp_carry (h, p, H, tp_stride, 0, c0, nchan);
			if (rc) return rc;
		}
		long long seg_done = 0;
		for (int n_main = 0; seg_done < nseg; ++n_main) {
			const long long n = std::min (next_launch_segs (n_main, seg_done, nseg, lp.segs_first, lp.segs_max, true), nseg - seg_done);
			rc                = run_launch (seg_done, n, c0, nchan, d_lcnt + (size_t)n_main * C);
			if (rc) return rc;
			l_s0.push_back (seg_done);
			l_n.push_back (n);
			seg_done += n;
		}
		lcnt.resize (l_s0.size () * C);
		CK (cudaMemcpyAsync (lcnt.data (), d_lcnt, sizeof (unsigned) * lcnt.size (), cudaMemcpyDeviceToHost, h->stream));
		CK (cudaStreamSynchronize (h->stream));
		h->stats.d2h_bytes += sizeof (unsigned) * lcnt.size ();

		// overflowed (launch, channel): overs_kernel skipped it; re-run its segments in pieces that fit the list
		unsigned*       d_rcnt_l = d_lcnt + (size_t)(n_lmax - 1) * C;
		const long long fit      = std::max<long long> (1, lp.cap / lp.ppseg);
		for (size_t k = 0; k < l_s0.size (); ++k) {
			for (int c = c0; c < c1; ++c) {
				if (lcnt[k * C + c] <= (unsigned)lp.cap) continue;
				++h->stats.dense_repeats;
				for (long long s = l_s0[k]; s < l_s0[k] + l_n[k]; s += fit) {
					if (OS > 1) {
						rc = seed_tp_carry (h, p, H, tp_stride, s, c, 1);
						if (rc) return rc;
					}
					CK (cudaMemsetAsync (d_rcnt_l + c, 0, sizeof (unsigned), h->stream));
					rc = run_launch (s, std::min (fit, l_s0[k] + l_n[k] - s), c, 1, d_rcnt_l);
					if (rc) return rc;
				}
			}
		}
	}

	std::vector<unsigned long long> res (n_u64);
	CK (cudaMemcpyAsync (res.data (), d_cnt, sizeof (unsigned long long) * n_u64, cudaMemcpyDeviceToHost, h->stream));
	CK (cudaStreamSynchronize (h->stream));
	prof_resolve (h);
	h->stats.d2h_bytes += sizeof (unsigned long long) * n_u64;
	if (A > 0) {
		h->stats.points_total += g.points (nchan, G);
		h->stats.points_evaluated += res[n_u64 - 1];
	}

	const size_t MS = (size_t)h->MS;
	std::fill (counts, counts + (size_t)C * MS, (uint64_t)0);
	if (excess) std::fill (excess, excess + (size_t)C * MS, 0.0);
	const double ulp = std::ldexp (1.0, -32);
	for (int c = c0; c < c1; ++c) {
		for (int k = 0; k < A; ++k) {
			const size_t i = (size_t)c * A + k, o = (size_t)c * MS + idx[(size_t)k];
			counts[o]      = res[i];
			if (excess) excess[o] = (double)res[n_tab + i] * ulp;
		}
		// grid index 0: the raw input; should the schedule also wrap onto index 0, the entry with more overs
		// (peak[c][0] is the larger of the two peaks)
		if (raw && res[2 * n_tab + c] >= counts[(size_t)c * MS]) {
			counts[(size_t)c * MS] = res[2 * n_tab + c];
			if (excess) excess[(size_t)c * MS] = (double)res[2 * n_tab + C + c] * ulp;
		}
	}
	return PHASEROT_OK;
}

int
overs_entry (phaserot* h, const void* src, bool dev_in, int format, uint64_t n_frames, float ceiling, int ang_start, int ang_end, int ang_stride, int chn,
             uint64_t* counts, double* excess)
{
	int rc = check_analysis (h, src, format, n_frames, "phaserot_overs", [&] () -> const char* {
		if (!(ceiling > 0.f) || !std::isfinite (ceiling)) return "the ceiling is not a finite value > 0";
		if (!counts) return "NULL counts";
		if (ang_stride < 1) return "ang_stride < 1";
		if (chn >= h->C) return "chn is not a channel of the handle";
		return nullptr;
	});
	if (rc) return rc;
	DevGuard     guard (h->dev);
	const float* d_x;
	rc = land_input (h, src, dev_in, format, (long long)n_frames, &d_x);
	if (rc) return rc;
	return overs_core (h, d_x, (long long)n_frames, ceiling, ang_start, ang_end, ang_stride, chn, counts, excess);
}

/*
 * phaserot_nth_peaks over F frames of interleaved float32 audio on the device.  kth[c][a] starts at 0 and
 * follows the N-th value of the row; threshold_kernel turns it into the filter radius (min_a kth)^2 (1 - 1e-5)
 * of the FFT pass (a sample below it is at or below kth at every angle, and so cannot change a row), and
 * nth_kernel / nth_merge_kernel turn each launch's survivors into candidates and merge them.  Launches and lists
 * as a device-resident sweep, including its bootstrap wave, whose rows are a subset's: they only seed kth from
 * below and are cleared.  After every launch the host reads the list counters and bucket flags.  Every sample
 * enters a row exactly once: a channel whose buckets ran over had all of the launch's candidates dropped and
 * takes its list again in chunks of K records, which one bucket holds in full; a channel whose list overflowed
 * was skipped by nth_kernel, and its segments are re-run at the end in pieces the list holds.  Grid index 0:
 * exact radix selection over the raw input values above a lower bound from block maxima.  Synchronous.  out: host
 * [C][MS][N].
 */
constexpr int kMaxRank = 256; // largest n_rank of phaserot_nth_peaks: a row and 256 candidates fill one sort of kNthSort

int
nth_core (phaserot* h, const float* d_x, long long F, int N, int ang_start, int ang_end, int ang_stride, int chn, float* out)
{
	std::vector<int> idx;
	bool             raw = false;
	int              rc  = angle_schedule (h, ang_start, ang_end, ang_stride, idx, raw);
	if (rc) return rc;
	const int        C        = h->C;
	const int        A        = (int)idx.size ();
	const int        A1       = A + 1; // slot A: grid index 0 from the raw input
	const int        c0       = chn < 0 ? 0 : chn;
	const int        c1       = chn < 0 ? C : chn + 1;
	const int        nchan    = c1 - c0;
	const int        OS       = h->OS;
	const int        G        = OS > 1 ? OS + 1 : 1;          // points per record
	const StreamGeom g        = stream_geom (h, F, 1, true); // like phaserot_sweep
	const long long  nseg     = g.nseg;
	const bool       no_prune = (h->cfg.flags & PHASEROT_FLAG_NO_PRUNE) != 0;
	const ListPlan   lp       = plan_lists (h, nchan, nseg, true, no_prune);
	// candidate floats per slot: 8 K, fewer on grids so fine or wide that the buckets would pass 512 MB
	const unsigned K = (unsigned)std::min<long long> (8192, std::max<long long> (kNthSort, (128LL << 20) / ((long long)C * A1)));

	// work area: u64 evaluated | (ca, sa) [A] | rows [C][A1][N] | kth [C][A1] | bucket counters [C][A1] |
	// histograms [C][kNthDigits] | selection state [C][4] | list counters [C] | bucket flags [C] | thr2 [C] |
	// raw peaks [C] (unused) | r2max [C] | list overflow word (unused)
	const size_t n_slot = (size_t)C * A1;
	const size_t bytes  = sizeof (unsigned long long) + sizeof (float2) * (size_t)std::max (A, 1) + sizeof (float) * n_slot * N +
	                     sizeof (unsigned) * (2 * n_slot + (size_t)C * (kNthDigits + 4 + 5) + 1);
	rc = h->d_nthw.ensure (bytes);
	if (rc) return rc;
	rc = h->d_nthc.ensure (sizeof (float) * n_slot * K);
	if (rc) return rc;
	unsigned long long* d_eval  = (unsigned long long*)h->d_nthw.p;
	float2*             d_cs    = (float2*)(d_eval + 1);
	float*              d_rows  = (float*)(d_cs + std::max (A, 1));
	unsigned*           d_kth   = (unsigned*)(d_rows + n_slot * N);
	unsigned*           d_ccnt  = d_kth + n_slot;
	unsigned*           d_hist  = d_ccnt + n_slot;
	unsigned*           d_sel   = d_hist + (size_t)C * kNthDigits;
	unsigned*           d_lcnt  = d_sel + 4 * (size_t)C;
	unsigned*           d_covf  = d_lcnt + C;
	float*              d_thr2  = (float*)(d_covf + C);
	unsigned*           d_rawp  = (unsigned*)(d_thr2 + C);
	unsigned*           d_r2max = d_rawp + C;
	unsigned*           d_lovf  = d_r2max + C;
	float*              d_cand  = (float*)h->d_nthc.p;
	CK (cudaMemsetAsync (h->d_nthw.p, 0, bytes, h->stream));
	{
		std::vector<float2> cs ((size_t)A);
		for (int k = 0; k < A; ++k) cs[(size_t)k] = make_float2 (h->lut_c[(size_t)idx[(size_t)k]], h->lut_s[(size_t)idx[(size_t)k]]);
		std::vector<unsigned> sel ((size_t)4 * C, 0u); // the raw selection looks for rank N
		for (int c = 0; c < C; ++c) sel[(size_t)4 * c + 1] = (unsigned)N;
		CK (cudaMemcpyAsync (d_cs, cs.data (), sizeof (float2) * cs.size (), cudaMemcpyHostToDevice, h->stream));
		CK (cudaMemcpyAsync (d_sel, sel.data (), sizeof (unsigned) * sel.size (), cudaMemcpyHostToDevice, h->stream));
	}

	if (A > 0) {
		rc = h->d_ovl.ensure (sizeof (float2) * (size_t)lp.cap * C);
		if (rc) return rc;
		const long long tp_stride = (kTpCarry + lp.segs_cap * 2 * h->V + 3) & ~3LL;
		if (OS > 1) {
			rc = h->d_ovH.ensure (sizeof (float) * (size_t)tp_stride * C);
			if (rc) return rc;
		}
		float*         H   = (float*)h->d_ovH.p;
		const float2*  lst = (const float2*)h->d_ovl.p;
		const unsigned cap = (unsigned)lp.cap;
		ConvParams     p   = analysis_params (h, d_x, nullptr, F, g, c0, nchan, (float2*)h->d_ovl.p, lp.cap, d_lcnt, d_lovf, d_thr2, d_rawp);
		p.thr_mode         = -1;
		TpParams tp {};
		if (OS > 1) tp = tp_params (h, p, g.t_end, H, tp_stride);

		// records [r0, r0 + n_rec) of the lists of channels [ch0, ch0 + nch) (list capacity lcap) -> candidates -> rows
		auto candidates = [&] (int ch0, int nch, unsigned lcap, unsigned skip_above, unsigned r0, unsigned n_rec, bool boot) -> int {
			{
				ProfScope ps (h, 1);
				auto nth = [&] (auto G_) {
					dispatch_sweep (h, A, nch, [&] (auto R, dim3 grid, int nt) {
						nth_kernel<decltype (R)::value, decltype (G_)::value><<<grid, nt, 0, h->stream>>> (lst, lp.cap, d_lcnt, lcap, skip_above, r0, n_rec, ch0, d_cs, A, A1,
						                                                                                    d_kth, d_cand, d_ccnt, K, d_covf, d_eval);
					});
				};
				if (G == 1) nth (std::integral_constant<int, 1> ());
				else if (G == 3) nth (std::integral_constant<int, 3> ());
				else nth (std::integral_constant<int, 5> ());
				CK (cudaGetLastError ());
			}
			{
				ProfScope ps (h, 5);
				nth_merge_kernel<<<dim3 ((unsigned)A, (unsigned)nch), 256, 0, h->stream>>> (d_rows, d_kth, d_cand, d_ccnt, K, A1, 0, N, ch0, d_covf, boot ? 1 : 0);
				CK (cudaGetLastError ());
			}
			h->stats.kernel_launches += 2;
			return PHASEROT_OK;
		};

		// segments s0 + i stride, i < n, of channels [ch0, ch0 + nch): radius, FFT pass, candidates; then on the host
		// the bucket re-runs, and the channels whose list overflowed (not for the bootstrap, whose list may drop
		// points) to `overflowed`
		std::vector<unsigned> st ((size_t)2 * C);
		auto run_launch = [&] (long long s0, long long stride, long long n, int ch0, int nch, bool boot, std::vector<int>& overflowed) -> int {
			{
				ProfScope ps (h, 5);
				threshold_kernel<<<nch, 256, 0, h->stream>>> (d_kth, A1, A, ch0, d_thr2, d_lcnt, 1, no_prune ? 0 : 1);
				CK (cudaGetLastError ());
				++h->stats.kernel_launches;
			}
			p.chan0      = ch0;
			p.nchan      = nch;
			p.seg0       = s0;
			p.seg_stride = stride;
			p.nseg       = n;
			p.seg_jitter = boot && stride > 1;
			// the bootstrap wave: any subset of its samples is valid, what does not fit kBootCap points is dropped
			const unsigned lcap = boot ? (unsigned)std::min<long long> (lp.cap, kBootCap) : cap;
			int            r;
			if (OS > 1) {
				p.r2max = boot ? d_r2max : nullptr;
				r       = launch_conv<EPI_HILBERT, SRC_INTER> (h, p);
				if (r) return r;
				tp.chan0      = ch0;
				tp.seg0       = s0;
				tp.seg_stride = stride;
				tp.seg_jitter = p.seg_jitter;
				tp.boot_beta  = boot ? kBootBeta : 0.f;
				tp.r2max      = d_r2max;
				tp.list_cap   = lcap;
				{
					ProfScope ps (h, 6);
					truepeak_kernel<true><<<dim3 ((unsigned)(n * (tp.V2 / kTpTile)), (unsigned)nch), 256, 0, h->stream>>> (tp);
					CK (cudaGetLastError ());
					++h->stats.kernel_launches;
				}
				if (stride == 1) {
					r = launch_tp_carry (h, H, tp_stride, ch0, nch, n * 2 * h->V);
					if (r) return r;
				}
			} else {
				p.boot_beta = boot ? kBootBeta : 0.f;
				p.r2max     = d_r2max;
				p.list_cap  = lcap;
				r           = launch_conv<EPI_POINTS, SRC_INTER> (h, p);
				if (r) return r;
			}
			const unsigned skip_above = boot ? ~0u : cap;
			r                         = candidates (ch0, nch, lcap, skip_above, 0, ~0u, boot);
			if (r) return r;
			CK (cudaMemcpyAsync (st.data (), d_lcnt, sizeof (unsigned) * 2 * C, cudaMemcpyDeviceToHost, h->stream)); // list counters | bucket flags
			CK (cudaStreamSynchronize (h->stream));
			h->stats.d2h_bytes += sizeof (unsigned) * 2 * C;
			for (int c = ch0; c < ch0 + nch; ++c) {
				if (st[(size_t)c] > skip_above) {
					overflowed.push_back (c);
				} else if (st[(size_t)C + c]) {
					++h->stats.dense_repeats;
					CK (cudaMemsetAsync (d_covf + c, 0, sizeof (unsigned), h->stream));
					const unsigned n_rec = std::min (st[(size_t)c], lcap) / (unsigned)G;
					for (unsigned r0 = 0; r0 < n_rec; r0 += K) {
						r = candidates (c, 1, lcap, skip_above, r0, K, boot);
						if (r) return r;
					}
				}
			}
			return PHASEROT_OK;
		};

		std::vector<int> overflowed;
		const long long  wave = std::max<long long> (1, (h->n_sm + nchan - 1) / nchan); // segments per channel in one wave
		if (!no_prune && nseg >= 2 * wave) {
			// the sweep's bootstrap wave: kth from below, then empty rows
			rc = run_launch (0, nseg / wave, wave, c0, nchan, true, overflowed);
			if (rc) return rc;
			CK (cudaMemsetAsync (d_rows, 0, sizeof (float) * n_slot * N, h->stream));
		}
		if (OS > 1) {
			rc = seed_tp_carry (h, p, H, tp_stride, 0, c0, nchan);
			if (rc) return rc;
		}
		std::vector<long long> l_s0, l_n;
		std::vector<int>       l_k; // launch of each overflowed channel
		long long              seg_done = 0;
		for (int n_main = 0; seg_done < nseg; ++n_main) {
			const long long n = std::min (next_launch_segs (n_main, seg_done, nseg, lp.segs_first, lp.segs_max, true), nseg - seg_done);
			rc                = run_launch (seg_done, 1, n, c0, nchan, false, overflowed);
			if (rc) return rc;
			l_s0.push_back (seg_done);
			l_n.push_back (n);
			l_k.resize (overflowed.size (), n_main);
			seg_done += n;
		}
		// overflowed (launch, channel): re-run its segments in pieces that fit the list
		const long long fit = std::max<long long> (1, lp.cap / lp.ppseg);
		for (size_t i = 0; i < overflowed.size (); ++i) {
			const int c = overflowed[i], k = l_k[i];
			++h->stats.dense_repeats;
			for (long long s = l_s0[(size_t)k]; s < l_s0[(size_t)k] + l_n[(size_t)k]; s += fit) {
				if (OS > 1) {
					rc = seed_tp_carry (h, p, H, tp_stride, s, c, 1);
					if (rc) return rc;
				}
				std::vector<int> none;
				rc = run_launch (s, 1, std::min (fit, l_s0[(size_t)k] + l_n[(size_t)k] - s), c, 1, false, none);
				if (rc) return rc;
			}
		}
	}

	// grid index 0: radix selection over the raw input (the interpolator reaches 11 frames past the last one)
	static_assert (kMaxRank <= kNthSort, "the raw lower bound needs at least N block maxima (K >= kNthSort)");
	if (raw) {
		const long long f_end = std::min (F + (OS > 1 ? 11 : 0), g.t_end - h->L / 2);
		const dim3      grid ((unsigned)std::min<long long> ((f_end + 255) / 256, (long long)h->n_sm * 8), (unsigned)nchan);
		ProfScope       ps (h, 5);
		// the lower bound from kNthSort .. 4096 block maxima (at least N), then the rows cleared of them
		nth_raw_max_kernel<<<dim3 (std::min (K, 4096u), (unsigned)nchan), 256, 0, h->stream>>> (d_x, F, C, c0, f_end, OS, A1, A, d_cand, d_ccnt, K);
		nth_merge_kernel<<<dim3 (1, (unsigned)nchan), 256, 0, h->stream>>> (d_rows, d_kth, d_cand, d_ccnt, K, A1, A, N, c0, d_covf, 1);
		CK (cudaMemset2DAsync (d_rows + ((size_t)c0 * A1 + A) * N, sizeof (float) * A1 * N, 0, sizeof (float) * N, (size_t)nchan, h->stream));
		const int shift[3] = { 20, 10, 0 }, hi[3] = { 31, 20, 10 };
		for (int k = 0; k < 3; ++k) {
			nth_raw_hist_kernel<<<grid, 256, 0, h->stream>>> (d_x, F, C, c0, f_end, OS, shift[k], hi[k], d_sel, d_kth, A1, A, d_hist);
			nth_raw_pick_kernel<<<nchan, 256, 0, h->stream>>> (d_sel, d_hist, c0, shift[k], k == 2, N, A1, A, d_cand, d_ccnt, K);
		}
		nth_raw_collect_kernel<<<grid, 256, 0, h->stream>>> (d_x, F, C, c0, f_end, OS, d_sel, A1, A, d_cand, K);
		nth_merge_kernel<<<dim3 (1, (unsigned)nchan), 256, 0, h->stream>>> (d_rows, d_kth, d_cand, d_ccnt, K, A1, A, N, c0, d_covf, 0);
		CK (cudaGetLastError ());
		h->stats.kernel_launches += 10;
	}

	std::vector<float> rows (n_slot * N);
	unsigned long long n_eval = 0;
	CK (cudaMemcpyAsync (rows.data (), d_rows, sizeof (float) * rows.size (), cudaMemcpyDeviceToHost, h->stream));
	CK (cudaMemcpyAsync (&n_eval, d_eval, sizeof (n_eval), cudaMemcpyDeviceToHost, h->stream));
	CK (cudaStreamSynchronize (h->stream));
	prof_resolve (h);
	h->stats.d2h_bytes += sizeof (float) * rows.size () + sizeof (n_eval);
	if (A > 0) {
		h->stats.points_total += g.points (nchan, G);
		h->stats.points_evaluated += n_eval;
	}

	const size_t MS = (size_t)h->MS, n = (size_t)N;
	std::fill (out, out + (size_t)C * MS * n, 0.f);
	for (int c = c0; c < c1; ++c) {
		const float* rw = rows.data () + (size_t)c * A1 * n;
		float*       oc = out + (size_t)c * MS * n;
		for (int k = 0; k < A; ++k) std::copy (rw + (size_t)k * n, rw + (size_t)(k + 1) * n, oc + (size_t)idx[(size_t)k] * n);
		// grid index 0: the raw input; should the schedule also wrap onto index 0, the row with the larger rank-1
		// value (peak[c][0] is the larger of the two peaks; ties: the raw row)
		if (raw && rw[(size_t)A * n] >= oc[0]) std::copy (rw + (size_t)A * n, rw + (size_t)A1 * n, oc);
	}
	return PHASEROT_OK;
}

int
nth_entry (phaserot* h, const void* src, bool dev_in, int format, uint64_t n_frames, int n_rank, int ang_start, int ang_end, int ang_stride, int chn,
           float* out)
{
	int rc = check_analysis (h, src, format, n_frames, "phaserot_nth_peaks", [&] () -> const char* {
		if (n_rank < 1 || n_rank > kMaxRank) return "n_rank is not in 1 .. 256";
		if (!out) return "NULL out";
		if (ang_stride < 1) return "ang_stride < 1";
		if (chn >= h->C) return "chn is not a channel of the handle";
		return nullptr;
	});
	if (rc) return rc;
	DevGuard     guard (h->dev);
	const float* d_x;
	rc = land_input (h, src, dev_in, format, (long long)n_frames, &d_x);
	if (rc) return rc;
	return nth_core (h, d_x, (long long)n_frames, n_rank, ang_start, ang_end, ang_stride, chn, out);
}

// Argument checks of the sweep entry points: data may be null for an empty stream only, and every
// shard of a stream but the last is a whole number of blocks
int
check_sweep (const phaserot* h, const void* data, uint64_t n_frames, bool last = true)
{
	if (!h || (!data && n_frames)) {
		return PHASEROT_E_INVAL;
	}
	if (h->plugin) {
		return PHASEROT_E_STATE;
	}
	if (!last && ((long long)n_frames % h->L) != 0) {
		return PHASEROT_E_INVAL;
	}
	return PHASEROT_OK;
}

// pinned staging of one plugin call of n frames: window [C][wstride] | ramp prefix
// [C][pre_cap] | outputs [C][n] | per-CTA meter maxima [C][n_cta][2]
constexpr uint32_t kSmallCallMax = 16384;
inline size_t
plugin_io_bytes (const phaserot* h, uint32_t n)
{
	const size_t keep    = (size_t)h->firlen + h->P;
	const size_t wstride = (keep + n + 3) & ~(size_t)3;
	const size_t pre_cap = (size_t)h->P * 20;
	const size_t n_cta   = ((size_t)n + kStreamOut - 1) / kStreamOut;
	return sizeof (float) * wstride * h->C + sizeof (float2) * pre_cap * h->C + (n <= kSmallCallMax ? sizeof (float) * ((size_t)n + 2 * n_cta) * h->C : 0) + 64;
}

// src/phaserotate.c:122-133
inline void
plugin_sin_cos (float angle, float* s, float* c)
{
	static const float twopi = (float)(2 * M_PI);
	sincosf (angle * twopi, s, c);
}

/*
 * Angle handling of one completed partition (src/phaserotate.c:673-717):
 * fills coef[0..P) with the (ca, sa) used for each sample and updates the
 * channel's angle state.  Returns true when the partition was ramped.
 */
bool
plugin_partition_coef (phaserot* h, PluginChan& ch, float target, float2* coef)
{
	const uint32_t P = h->P;
	if (target != ch.angle) {
		const float interp_nm = 1.f / (float)P;    // src:296
		const float thresh    = (float)P * 1e-6f;  // src:295
		float       da        = target - ch.angle;
		if (fabs (da) > 0.5) { // wrap around at +/- 180 (src:676-683)
			if (da < 0) {
				da += 1.f;
			} else {
				da -= 1.f;
			}
		}
		da *= interp_nm;
		bool final = false;
		if (da > thresh) {
			da = thresh;
		} else if (da < -thresh) {
			da = -thresh;
		} else {
			final = true;
		}
		float angle = ch.angle;
		for (uint32_t i = 0; i < P; ++i) {
			float s, c;
			plugin_sin_cos (angle, &s, &c);
			coef[i] = make_float2 (c, s);
			angle += da;
		}
		if (final) {
			angle = target;
		}
		ch.angle = angle;
		if (angle == target) {
			plugin_sin_cos (angle, &ch.sa, &ch.ca);
		}
		return true;
	}
	for (uint32_t i = 0; i < P; ++i) {
		coef[i] = make_float2 (ch.ca, ch.sa);
	}
	return false;
}

} // namespace

// ===========================================================================
// C ABI
// ===========================================================================

extern "C" {

int
phaserot_abi_version (void)
{
	return PHASEROT_ABI_VERSION;
}

const char*
phaserot_strerror (int code)
{
	switch (code) {
		case PHASEROT_OK: return "ok";
		case PHASEROT_E_INVAL: return "invalid argument";
		case PHASEROT_E_NO_DEVICE: return "no usable sm_100 CUDA device (this backend has no CPU fallback)";
		case PHASEROT_E_CUDA: return "CUDA error";
		case PHASEROT_E_NOMEM: return "out of memory";
		case PHASEROT_E_UNSUPPORTED: return "configuration not supported by the device path";
		case PHASEROT_E_STATE: return "call not valid in this mode";
		case PHASEROT_E_AGAIN: return "a shard of the combined sweep overflowed its survivor list: the pass has been re-enqueued in dense mode, combine the pending tables again";
		default: return "unknown error";
	}
}

const char*
phaserot_last_error (void)
{
	return g_last_error;
}

int
phaserot_create (phaserot_t** out, const phaserot_cfg_t* cfg)
{
	if (!out) {
		return PHASEROT_E_INVAL;
	}
	*out = nullptr;
	if (!cfg || cfg->abi_version != PHASEROT_ABI_VERSION) {
		return PHASEROT_E_INVAL;
	}
	const bool plugin = cfg->mode == PHASEROT_MODE_PLUGIN;
	if (cfg->mode != PHASEROT_MODE_CLI && !plugin) {
		return PHASEROT_E_INVAL;
	}
	if (cfg->n_channels < 1 || cfg->n_channels > 64 || (plugin && cfg->n_channels > 2)) {
		return PHASEROT_E_INVAL;
	}
	int L = 0;
	uint32_t P = 0, firlen = 0;
	if (plugin) {
		if (!(cfg->sample_rate > 0)) {
			return PHASEROT_E_INVAL;
		}
		// src/phaserotate.c:278-297
		uint32_t fftlen;
		if (cfg->sample_rate < 64000) {
			fftlen = 512;
			firlen = 3072;
		} else if (cfg->sample_rate < 128000) {
			fftlen = 1024;
			firlen = 4096;
		} else {
			fftlen = 2048;
			firlen = 8192;
		}
		P = fftlen / 2;
		L = (int)firlen;
	} else {
		L = cfg->blksiz;
		// cli/phase-rotate.cc:749-755: power of two in [1024, 32768]
		if (L < 1024 || L > 32768 || (L & (L - 1))) {
			return PHASEROT_E_INVAL;
		}
	}
	const int S = cfg->subsample == 0 ? 2 : cfg->subsample;
	if (S < 1 || S > 1000) {
		return PHASEROT_E_INVAL;
	}
	const int OS = cfg->oversample <= 1 ? 1 : cfg->oversample;
	if (cfg->oversample < 0 || (OS != 1 && OS != 2 && OS != 4) || (OS > 1 && plugin)) {
		return PHASEROT_E_INVAL;
	}
	if (L / 2 > kM) {
		snprintf (g_last_error, sizeof (g_last_error), "FIR length %d needs %d half-taps; this build supports at most %d", L, L / 2, kM);
		return PHASEROT_E_UNSUPPORTED;
	}

	std::lock_guard<std::mutex> lk (g_create_lock);

	int ndev = 0;
	if (cudaGetDeviceCount (&ndev) != cudaSuccess || ndev < 1) {
		cudaGetLastError ();
		snprintf (g_last_error, sizeof (g_last_error), "no CUDA device");
		return PHASEROT_E_NO_DEVICE;
	}
	int dev = cfg->device;
	if (dev < 0) {
		if (cudaGetDevice (&dev) != cudaSuccess) {
			dev = 0;
		}
	}
	if (dev >= ndev) {
		return PHASEROT_E_INVAL;
	}
	cudaDeviceProp prop;
	if (cudaGetDeviceProperties (&prop, dev) != cudaSuccess) {
		cudaGetLastError ();
		return PHASEROT_E_NO_DEVICE;
	}
	if (prop.major != 10) {
		snprintf (g_last_error, sizeof (g_last_error), "device %d is sm_%d%d; this library contains sm_100a code only", dev, prop.major, prop.minor);
		return PHASEROT_E_NO_DEVICE;
	}

	phaserot* h = new (std::nothrow) phaserot ();
	if (!h) {
		return PHASEROT_E_NOMEM;
	}
	h->cfg    = *cfg;
	h->dev    = dev;
	h->n_sm   = prop.multiProcessorCount;
	h->C      = cfg->n_channels;
	h->L      = L;
	h->Lh     = L / 2;
	h->NP     = h->Lh > kM / 2 ? 2 : 1;
	h->Lp     = h->Lh / h->NP;
	h->V      = kM - h->Lp;
	h->padf   = (h->Lh + 3) & ~3;
	h->S      = S;
	h->MS     = 180 * S;
	h->OS     = OS;
	h->plugin = plugin;
	h->P      = P;
	h->firlen = firlen;
	h->firlat = firlen / 2;

	DevGuard guard (dev);
	int      rc = PHASEROT_OK;
	do {
		design_fir (L, plugin, h->taps);
		build_lut (S, h->lut_s, h->lut_c);
		h->table.assign ((size_t)h->C * h->MS, 0.f);
		cudaError_t e = cudaStreamCreateWithFlags (&h->own_stream, cudaStreamNonBlocking);
		if (e == cudaSuccess) e = cudaStreamCreateWithFlags (&h->copy_stream, cudaStreamNonBlocking);
		for (int b = 0; b < 2 && e == cudaSuccess; ++b) {
			e = cudaEventCreateWithFlags (&h->ev_copy[b], cudaEventDisableTiming);
			if (e == cudaSuccess) e = cudaEventCreateWithFlags (&h->ev_done[b], cudaEventDisableTiming);
		}
		if (e != cudaSuccess) {
			rc = cuda_fail (e, "stream/event creation", __LINE__);
			break;
		}
		h->stream = h->own_stream;
		rc        = set_device_attrs (dev, h->NP, plugin ? (KA_RENDER_PLANE | KA_FIR_STREAM) : (KA_RENDER_INTER | (OS > 1 ? KA_HILBERT : KA_POINTS)));
		if (rc) break;
		rc = h->d_small.ensure (kSmallBytes);
		if (rc) break;
		if (cudaMemset (h->d_small.p, 0, kSmallBytes) != cudaSuccess) {
			rc = PHASEROT_E_CUDA;
			break;
		}
		rc = upload_tables (h);
		if (rc) break;
		if (plugin) {
			h->pch.resize ((size_t)h->C);
			for (auto& ch : h->pch) {
				ch.last.assign (P, make_float2 (1.f, 0.f));
				plugin_sin_cos (0.f, &ch.sa, &ch.ca); // channel_init, src:147,159
				ch.last_const = make_float2 (ch.ca, ch.sa);
			}
			h->ptail.assign ((size_t)h->C * (firlen + P), 0.f);
			// everything a small call (n <= kSmallCallMax frames; LV2 hosts stay below
			// MAXPERIOD 8192, robtk/jackwrap.c:36) touches is allocated here, so that
			// run() neither allocates nor locks in steady state, whatever period the
			// host picks or changes to
			rc = h->h_io.ensure (plugin_io_bytes (h, kSmallCallMax));
			if (rc) break;
			rc = h->d_ring.ensure (sizeof (float) * (size_t)kRing * h->C);
			if (rc) break;
		} else {
			h->ap_hist.assign ((size_t)h->C * L, 0.f);
		}
	} while (0);
	if (rc) {
		phaserot_destroy (h);
		return rc;
	}
	*out = h;
	return PHASEROT_OK;
}

void
phaserot_destroy (phaserot_t* h)
{
	if (!h) {
		return;
	}
	std::lock_guard<std::mutex> lk (g_create_lock);
	DevGuard                    guard (h->dev);
	if (h->own_stream) cudaStreamSynchronize (h->own_stream);
	if (h->copy_stream) cudaStreamSynchronize (h->copy_stream);
	for (DevBuf* b : { &h->d_G, &h->d_G1, &h->d_scratch, &h->d_tw, &h->d_g, &h->d_plane, &h->d_out, &h->d_list, &h->d_stage[0], &h->d_stage[1], &h->d_io, &h->d_inter, &h->d_hist, &h->d_small,
	                   &h->d_cs, &h->d_peaks, &h->d_ramp, &h->d_chancs, &h->d_tpH, &h->d_ring, &h->d_slot, &h->d_sec, &h->d_wide,
	                   &h->d_sect, &h->d_sect_aux, &h->d_sect_rt, &h->d_kx, &h->d_lH, &h->d_lwork, &h->d_lset, &h->d_ovl, &h->d_ovH, &h->d_ovw,
	                   &h->d_nthw, &h->d_nthc }) {
		b->release ();
	}
	for (PinBuf* b : { &h->h_stage[0], &h->h_stage[1], &h->h_res, &h->h_io, &h->h_cs, &h->h_slot }) {
		b->release ();
	}
	for (int b = 0; b < 2; ++b) {
		if (h->ev_copy[b]) cudaEventDestroy (h->ev_copy[b]);
		if (h->ev_done[b]) cudaEventDestroy (h->ev_done[b]);
	}
	for (cudaEvent_t e : h->prof_ev) cudaEventDestroy (e);
	if (h->own_stream) cudaStreamDestroy (h->own_stream);
	if (h->copy_stream) cudaStreamDestroy (h->copy_stream);
	delete h;
}

int
phaserot_set_stream (phaserot_t* h, void* cuda_stream)
{
	if (!h) {
		return PHASEROT_E_INVAL;
	}
	DevGuard guard (h->dev);
	const int rc = finish_pending (h);
	if (rc) return rc;
	h->stream = cuda_stream ? (cudaStream_t)cuda_stream : h->own_stream;
	return PHASEROT_OK;
}

int
phaserot_reset (phaserot_t* h)
{
	if (!h) {
		return PHASEROT_E_INVAL;
	}
	DevGuard guard (h->dev);
	CK (cudaStreamSynchronize (h->stream));
	h->pending = false;
	std::fill (h->table.begin (), h->table.end (), 0.f);
	h->an_buf.clear ();
	h->an_blocks  = 0;
	h->an_first   = 0;
	h->hist_valid = false;
	std::fill (h->ap_hist.begin (), h->ap_hist.end (), 0.f);
	if (h->plugin) {
		// activate() clears buffers but keeps the angle state (src:169-177, 511-520)
		std::fill (h->ptail.begin (), h->ptail.end (), 0.f);
		h->ppos       = 0;
		h->ring_valid = false;
		for (auto& ch : h->pch) {
			ch.last_is_ramp = false;
			ch.last_const   = make_float2 (ch.ca, ch.sa);
		}
	}
	return PHASEROT_OK;
}

int
phaserot_sweep (phaserot_t* h, const float* interleaved, uint64_t n_frames, int ang_start, int ang_end, int ang_stride, int chn)
{
	int rc = check_sweep (h, interleaved, n_frames);
	if (rc) return rc;
	DevGuard guard (h->dev);
	rc = sweep_core (h, shard_job (interleaved, false, PHASEROT_PCM_F32, (long long)n_frames, nullptr, true, true, ang_start, ang_end, ang_stride, chn),
	                 Pass::Fresh);
	if (rc) return rc;
	return finish_pending (h);
}

int
phaserot_sweep_pcm (phaserot_t* h, const void* pcm, int format, uint64_t n_frames, int ang_start, int ang_end, int ang_stride, int chn)
{
	if (format != PHASEROT_PCM_S16 && format != PHASEROT_PCM_S32 && format != PHASEROT_PCM_S24) {
		return PHASEROT_E_INVAL;
	}
	int rc = check_sweep (h, pcm, n_frames);
	if (rc) return rc;
	DevGuard guard (h->dev);
	rc = sweep_core (h, shard_job (pcm, false, format, (long long)n_frames, nullptr, true, true, ang_start, ang_end, ang_stride, chn), Pass::Fresh);
	if (rc) return rc;
	return finish_pending (h);
}

int
phaserot_sweep_device (phaserot_t* h, const float* d_interleaved, uint64_t n_frames, int ang_start, int ang_end, int ang_stride, int chn)
{
	const int rc = check_sweep (h, d_interleaved, n_frames);
	if (rc) return rc;
	DevGuard guard (h->dev);
	return sweep_core (h, shard_job (d_interleaved, true, PHASEROT_PCM_F32, (long long)n_frames, nullptr, true, true, ang_start, ang_end, ang_stride, chn),
	                   Pass::Fresh);
}

int
phaserot_analyze (phaserot_t* h, const float* block, int ang_start, int ang_end, int ang_stride, int chn, int start)
{
	if (!h || !block) {
		return PHASEROT_E_INVAL;
	}
	if (h->plugin) {
		return PHASEROT_E_STATE;
	}
	DevGuard guard (h->dev);
	if (h->an_blocks && (ang_start != h->an_start || ang_end != h->an_end || ang_stride != h->an_stride || chn != h->an_chn)) {
		const int rc = flush_analyze (h);
		if (rc) return rc;
	}
	if (h->an_blocks == 0) {
		h->an_start  = ang_start;
		h->an_end    = ang_end;
		h->an_stride = ang_stride;
		h->an_chn    = chn;
		h->an_first  = start;
		if (start) {
			h->hist_valid = false;
		}
	}
	try {
		h->an_buf.insert (h->an_buf.end (), block, block + (size_t)h->L * h->C);
	} catch (...) {
		return PHASEROT_E_NOMEM;
	}
	++h->an_blocks;
	// bound the staging memory: flush every ~256 MB
	if (h->an_buf.size () * sizeof (float) >= (256u << 20)) {
		return flush_analyze (h);
	}
	return PHASEROT_OK;
}

int
phaserot_sync (phaserot_t* h)
{
	if (!h) {
		return PHASEROT_E_INVAL;
	}
	DevGuard guard (h->dev);
	int      rc = flush_analyze (h);
	if (rc) return rc;
	rc = finish_pending (h);
	if (rc) return rc;
	CK (cudaStreamSynchronize (h->stream));
	prof_resolve (h);
	return PHASEROT_OK;
}

int
phaserot_set_profiling (phaserot_t* h, int on)
{
	if (!h) {
		return PHASEROT_E_INVAL;
	}
	DevGuard guard (h->dev);
	CK (cudaStreamSynchronize (h->stream));
	prof_resolve (h);
	h->prof = on != 0;
	memset (&h->ktimes, 0, sizeof (h->ktimes));
	return PHASEROT_OK;
}

int
phaserot_get_kernel_times (phaserot_t* h, phaserot_ktimes_t* out)
{
	if (!h || !out) {
		return PHASEROT_E_INVAL;
	}
	DevGuard guard (h->dev);
	CK (cudaStreamSynchronize (h->stream));
	prof_resolve (h);
	*out = h->ktimes;
	return PHASEROT_OK;
}

int
phaserot_sweep_shard_device (phaserot_t* h, const float* d_interleaved, uint64_t n_frames, const float* hist, int first, int last,
                             int ang_start, int ang_end, int ang_stride, int chn)
{
	const int rc = check_sweep (h, d_interleaved, n_frames, last != 0);
	if (rc) return rc;
	DevGuard guard (h->dev);
	return sweep_core (h, shard_job (d_interleaved, true, PHASEROT_PCM_F32, (long long)n_frames, hist, first != 0, last != 0, ang_start, ang_end, ang_stride, chn),
	                   Pass::Fresh);
}

int
phaserot_sweep_shard_boot_device (phaserot_t* h, const float* d_interleaved, uint64_t n_frames, const float* hist, int first, int last,
                                  int ang_start, int ang_end, int ang_stride, int chn)
{
	const int rc = check_sweep (h, d_interleaved, n_frames, last != 0);
	if (rc) return rc;
	DevGuard guard (h->dev);
	return sweep_core (h, shard_job (d_interleaved, true, PHASEROT_PCM_F32, (long long)n_frames, hist, first != 0, last != 0, ang_start, ang_end, ang_stride, chn),
	                   Pass::BootOnly);
}

int
phaserot_sweep_shard_resume (phaserot_t* h)
{
	if (!h) {
		return PHASEROT_E_INVAL;
	}
	if (h->plugin || !h->pending) {
		return PHASEROT_E_STATE;
	}
	DevGuard guard (h->dev);
	return sweep_core (h, h->redo, Pass::Continue);
}

int
phaserot_sweep_shard (phaserot_t* h, const void* data, int format, uint64_t n_frames, const float* hist, int first, int last,
                      int ang_start, int ang_end, int ang_stride, int chn)
{
	if (format < PHASEROT_PCM_F32 || format > PHASEROT_PCM_S24) {
		return PHASEROT_E_INVAL;
	}
	const int rc = check_sweep (h, data, n_frames, last != 0);
	if (rc) return rc;
	DevGuard guard (h->dev);
	return sweep_core (h, shard_job (data, false, format, (long long)n_frames, hist, first != 0, last != 0, ang_start, ang_end, ang_stride, chn), Pass::Fresh);
}

int
phaserot_plugin_angle (phaserot_t* h, float* angle_turns)
{
	if (!h || !angle_turns) {
		return PHASEROT_E_INVAL;
	}
	if (!h->plugin) {
		return PHASEROT_E_STATE;
	}
	for (int c = 0; c < h->C; ++c) {
		angle_turns[c] = h->pch[(size_t)c].angle;
	}
	return PHASEROT_OK;
}

int
phaserot_pending_table (phaserot_t* h, float** d_table, int* n_channels, int* n_angles)
{
	if (!h || !d_table || !n_channels || !n_angles) {
		return PHASEROT_E_INVAL;
	}
	if (!h->pending) {
		return PHASEROT_E_STATE;
	}
	h->pend_exposed = true; // completion is now the caller's protocol, see the header
	*d_table    = (float*)h->d_peaks.p;
	*n_channels = h->C;
	*n_angles   = std::max (h->pend_A, 1);
	return PHASEROT_OK;
}

float
phaserot_peak (phaserot_t* h, int c, int a)
{
	if (!h || phaserot_sync (h) != PHASEROT_OK) {
		return NAN;
	}
	a = ((a % h->MS) + h->MS) % h->MS;
	if (c < 0 || c >= h->C) {
		// PhaseRotate::peak_all (cli:287-299)
		float p = 0;
		for (int k = 0; k < h->C; ++k) {
			p = std::max (p, h->table[(size_t)k * h->MS + a]);
		}
		return p;
	}
	return h->table[(size_t)c * h->MS + a];
}

int
phaserot_peaks (phaserot_t* h, float* out)
{
	if (!h || !out) {
		return PHASEROT_E_INVAL;
	}
	const int rc = phaserot_sync (h);
	if (rc) return rc;
	memcpy (out, h->table.data (), sizeof (float) * h->table.size ());
	return PHASEROT_OK;
}

int
phaserot_lut (phaserot_t* h, float* s, float* c)
{
	if (!h || !s || !c) {
		return PHASEROT_E_INVAL;
	}
	memcpy (s, h->lut_s.data (), sizeof (float) * (size_t)h->MS);
	memcpy (c, h->lut_c.data (), sizeof (float) * (size_t)h->MS);
	return PHASEROT_OK;
}

static int
angles_to_cs (phaserot* h, const int* angles, std::vector<float2>& cs)
{
	cs.resize ((size_t)h->C);
	for (int c = 0; c < h->C; ++c) {
		const int a   = ((angles[c] % h->MS) + h->MS) % h->MS; // cli:463
		cs[(size_t)c] = make_float2 (h->lut_c[(size_t)a], h->lut_s[(size_t)a]);
	}
	return PHASEROT_OK;
}

int
phaserot_apply (phaserot_t* h, float* buf, const int* angles)
{
	if (!h || !buf || !angles) {
		return PHASEROT_E_INVAL;
	}
	if (h->plugin) {
		return PHASEROT_E_STATE;
	}
	DevGuard            guard (h->dev);
	std::vector<float2> cs;
	angles_to_cs (h, angles, cs);
	long long m_end = 0;
	int       rc    = h->d_stage[0].ensure (sizeof (float) * (size_t)h->L * h->C);
	if (rc) return rc;
	rc = render_core (h, buf, false, h->L, h->L, h->ap_hist.data (), cs.data (), nullptr, 0, nullptr, &m_end, (float*)h->d_stage[0].p);
	if (rc) return rc;
	// remember the input block as history (cli:461) before it is overwritten
	memcpy (h->ap_hist.data (), buf, sizeof (float) * (size_t)h->L * h->C);
	CK (cudaMemcpyAsync (buf, h->d_stage[0].p, sizeof (float) * (size_t)h->L * h->C, cudaMemcpyDeviceToHost, h->stream));
	CK (cudaStreamSynchronize (h->stream));
	h->stats.d2h_bytes += sizeof (float) * (size_t)h->L * h->C;
	return PHASEROT_OK;
}

static int
render_bulk (phaserot* h, const float* src, bool dev_in, uint64_t n_frames, const int* angles, int flush_blocks, float* dst, bool dev_out)
{
	if (!h || (!src && n_frames) || !angles || !dst || flush_blocks < 0) {
		return PHASEROT_E_INVAL;
	}
	if (h->plugin) {
		return PHASEROT_E_STATE;
	}
	DevGuard            guard (h->dev);
	std::vector<float2> cs;
	angles_to_cs (h, angles, cs);
	const long long F     = (long long)n_frames;
	const long long B     = (F + h->L - 1) / h->L;
	const long long t_end = stream_geom (h, F, flush_blocks, false).t_end;
	if (t_end == 0) {
		return PHASEROT_OK;
	}
	long long    m_end = 0;
	const size_t bytes = sizeof (float) * (size_t)t_end * h->C;
	int          rc    = PHASEROT_OK;
	if (!dev_out) {
		// d_io holds the uploaded input; the staging buffer takes the output
		rc = h->d_stage[0].ensure (bytes);
		if (rc) return rc;
	}
	rc = render_core (h, src, dev_in, F, t_end, nullptr, cs.data (), nullptr, 0, nullptr, &m_end, dev_out ? dst : (float*)h->d_stage[0].p);
	if (rc) return rc;
	// stream state for a following apply(): the last block that went in
	std::fill (h->ap_hist.begin (), h->ap_hist.end (), 0.f);
	if (flush_blocks == 0 && B > 0 && !dev_in) {
		const long long f0 = (B - 1) * h->L;
		memcpy (h->ap_hist.data (), src + (size_t)f0 * h->C, sizeof (float) * (size_t)(F - f0) * h->C);
	} else if (flush_blocks == 0 && B > 0 && dev_in) {
		const long long f0 = (B - 1) * h->L;
		CK (cudaMemcpyAsync (h->ap_hist.data (), src + (size_t)f0 * h->C, sizeof (float) * (size_t)(F - f0) * h->C, cudaMemcpyDeviceToHost, h->stream));
		CK (cudaStreamSynchronize (h->stream));
	}
	if (dev_out) {
		return PHASEROT_OK;
	}
	CK (cudaMemcpyAsync (dst, h->d_stage[0].p, bytes, cudaMemcpyDeviceToHost, h->stream));
	CK (cudaStreamSynchronize (h->stream));
	h->stats.d2h_bytes += bytes;
	return PHASEROT_OK;
}

int
phaserot_render (phaserot_t* h, const float* interleaved, uint64_t n_frames, const int* angles, int flush_blocks, float* out)
{
	return render_bulk (h, interleaved, false, n_frames, angles, flush_blocks, out, false);
}

int
phaserot_render_device (phaserot_t* h, const float* d_interleaved, uint64_t n_frames, const int* angles, int flush_blocks, float* d_out)
{
	return render_bulk (h, d_interleaved, true, n_frames, angles, flush_blocks, d_out, true);
}

int
phaserot_sweep_sections (phaserot_t* h, const void* data, int format, uint64_t n_frames, uint64_t section_frames, int ang_start, int ang_end, int ang_stride,
                         int chn)
{
	if (format < PHASEROT_PCM_F32 || format > PHASEROT_PCM_S24) {
		return PHASEROT_E_INVAL;
	}
	const int rc = check_sweep (h, data, n_frames);
	if (rc) return rc;
	DevGuard guard (h->dev);
	return sweep_sections_core (h, (const float*)data, false, format, (long long)n_frames, (long long)section_frames, ang_start, ang_end, ang_stride, chn);
}

int
phaserot_sweep_sections_device (phaserot_t* h, const float* d_interleaved, uint64_t n_frames, uint64_t section_frames, int ang_start, int ang_end,
                                int ang_stride, int chn)
{
	const int rc = check_sweep (h, d_interleaved, n_frames);
	if (rc) return rc;
	DevGuard guard (h->dev);
	return sweep_sections_core (h, d_interleaved, true, PHASEROT_PCM_F32, (long long)n_frames, (long long)section_frames, ang_start, ang_end, ang_stride, chn);
}

int
phaserot_section_peaks (phaserot_t* h, int* n_sections, float* out)
{
	if (!h || !n_sections) {
		return PHASEROT_E_INVAL;
	}
	if (h->plugin) {
		return PHASEROT_E_STATE;
	}
	*n_sections = (int)h->sect_n;
	if (!out || h->sect_n == 0) {
		return PHASEROT_OK;
	}
	DevGuard            guard (h->dev);
	const int           A = h->sect_A, nchan = h->sect_c1 - h->sect_c0;
	const size_t        R = (size_t)h->sect_n * nchan;
	std::vector<float>  res (R * A + R);
	CK (cudaMemcpyAsync (res.data (), h->d_sect.p, sizeof (float) * res.size (), cudaMemcpyDeviceToHost, h->stream));
	CK (cudaStreamSynchronize (h->stream));
	h->stats.d2h_bytes += sizeof (float) * res.size ();
	const size_t per = (size_t)h->C * h->MS;
	std::fill (out, out + (size_t)h->sect_n * per, 0.f);
	for (size_t r = 0; r < R; ++r) {
		merge_row (out + (r / nchan) * per + (size_t)(h->sect_c0 + (int)(r % nchan)) * h->MS, res.data () + r * A, h->sect_idx,
		           h->sect_raw ? res.data () + R * A + r : nullptr);
	}
	for (size_t i = 0; i < h->sect_redo_k.size (); ++i) {
		memcpy (out + (size_t)h->sect_redo_k[i] * per, h->sect_redo.data () + i * per, sizeof (float) * per);
	}
	return PHASEROT_OK;
}

static int
render_sections_bulk (phaserot* h, const float* src, bool dev_in, uint64_t n_frames, uint64_t section_frames, const int* angles, int flush_blocks, float* dst,
                      bool dev_out)
{
	if (!h || (!src && n_frames) || !angles || !dst || flush_blocks < 0) {
		return PHASEROT_E_INVAL;
	}
	if (h->plugin) {
		return PHASEROT_E_STATE;
	}
	DevGuard        guard (h->dev);
	const long long F = (long long)n_frames;
	long long       n_sect;
	int             rc = check_sections (h, F, (long long)section_frames, h->C, &n_sect);
	if (rc) return rc;
	const long long t_end = stream_geom (h, F, flush_blocks, false).t_end;
	const size_t    bytes = sizeof (float) * (size_t)t_end * h->C;
	const float*    d_src = src;
	if (!dev_in) {
		const size_t in_bytes = sizeof (float) * (size_t)F * h->C;
		rc                    = h->d_io.ensure (in_bytes);
		if (rc) return rc;
		CK (cudaMemcpyAsync (h->d_io.p, src, in_bytes, cudaMemcpyHostToDevice, h->stream));
		h->stats.h2d_bytes += in_bytes;
		d_src = (const float*)h->d_io.p;
	}
	float* d_dst = dst;
	if (!dev_out) {
		rc = h->d_stage[0].ensure (bytes);
		if (rc) return rc;
		d_dst = (float*)h->d_stage[0].p;
	}
	rc = render_sections_core (h, d_src, F, t_end, (long long)section_frames, n_sect, angles, d_dst);
	if (rc) return rc;
	if (!dev_out) {
		CK (cudaMemcpyAsync (dst, d_dst, bytes, cudaMemcpyDeviceToHost, h->stream));
		CK (cudaStreamSynchronize (h->stream));
		h->stats.d2h_bytes += bytes;
	}
	return PHASEROT_OK;
}

int
phaserot_render_sections (phaserot_t* h, const float* interleaved, uint64_t n_frames, uint64_t section_frames, const int* angles, int flush_blocks, float* out)
{
	return render_sections_bulk (h, interleaved, false, n_frames, section_frames, angles, flush_blocks, out, false);
}

int
phaserot_render_sections_device (phaserot_t* h, const float* d_interleaved, uint64_t n_frames, uint64_t section_frames, const int* angles, int flush_blocks,
                                 float* d_out)
{
	return render_sections_bulk (h, d_interleaved, true, n_frames, section_frames, angles, flush_blocks, d_out, true);
}

int
phaserot_loudness (phaserot_t* h, const void* data, int format, uint64_t n_frames, double sample_rate, const float* weights, const int* angles, int n_sets,
                   double* lufs)
{
	return loudness_entry (h, data, false, format, n_frames, sample_rate, weights, angles, n_sets, lufs);
}

int
phaserot_loudness_device (phaserot_t* h, const float* d_interleaved, uint64_t n_frames, double sample_rate, const float* weights, const int* angles, int n_sets,
                          double* lufs)
{
	return loudness_entry (h, d_interleaved, true, PHASEROT_PCM_F32, n_frames, sample_rate, weights, angles, n_sets, lufs);
}

int
phaserot_overs (phaserot_t* h, const void* data, int format, uint64_t n_frames, float ceiling, int ang_start, int ang_end, int ang_stride, int chn,
                uint64_t* counts, double* excess)
{
	return overs_entry (h, data, false, format, n_frames, ceiling, ang_start, ang_end, ang_stride, chn, counts, excess);
}

int
phaserot_overs_device (phaserot_t* h, const float* d_interleaved, uint64_t n_frames, float ceiling, int ang_start, int ang_end, int ang_stride, int chn,
                       uint64_t* counts, double* excess)
{
	return overs_entry (h, d_interleaved, true, PHASEROT_PCM_F32, n_frames, ceiling, ang_start, ang_end, ang_stride, chn, counts, excess);
}

PHASEROT_API int
phaserot_nth_peaks (phaserot_t* h, const void* data, int format, uint64_t n_frames, int n_rank, int ang_start, int ang_end, int ang_stride, int chn,
                    float* out)
{
	return nth_entry (h, data, false, format, n_frames, n_rank, ang_start, ang_end, ang_stride, chn, out);
}

PHASEROT_API int
phaserot_nth_peaks_device (phaserot_t* h, const float* d_interleaved, uint64_t n_frames, int n_rank, int ang_start, int ang_end, int ang_stride, int chn,
                           float* out)
{
	return nth_entry (h, d_interleaved, true, PHASEROT_PCM_F32, n_frames, n_rank, ang_start, ang_end, ang_stride, chn, out);
}

uint32_t
phaserot_shard_align (const phaserot_t* h)
{
	if (!h || h->plugin) {
		return 0;
	}
	// one FFT segment yields 2 V samples; 2 V = 32768 - L is a multiple of L for every power-of-two L
	uint32_t a = 2u * (uint32_t)h->V;
	while (a % (uint32_t)h->L) {
		a += 2u * (uint32_t)h->V;
	}
	return a;
}

uint32_t
phaserot_latency (const phaserot_t* h)
{
	if (!h) {
		return 0;
	}
	return h->plugin ? h->P + h->firlat : (uint32_t)h->L / 2;
}

int
phaserot_process (phaserot_t* h, const float* const* in, float* const* out, uint32_t n_frames, const float* angle_deg)
{
	return phaserot_process_levels (h, in, out, n_frames, angle_deg, nullptr, nullptr);
}

int
phaserot_process_levels (phaserot_t* h, const float* const* in, float* const* out, uint32_t n_frames, const float* angle_deg,
                         float* level_in, float* level_out)
{
	if (!h || !in || !out || !angle_deg) {
		return PHASEROT_E_INVAL;
	}
	if (!h->plugin) {
		return PHASEROT_E_STATE;
	}
	const bool want_levels = level_in && level_out;
	if (n_frames == 0) {
		for (int c = 0; want_levels && c < h->C; ++c) level_in[c] = level_out[c] = 0.f;
		return PHASEROT_OK;
	}
	DevGuard       guard (h->dev);
	const uint32_t P = h->P, firlen = h->firlen, keep = firlen + P, n = n_frames;
	const int      C  = h->C;
	const uint64_t t0 = h->ppos;

	// Window per channel: W = [tail (keep) | new (n)]; output i in [0, n) is
	// Y[u], u = t0 - P + i, at W index firlen + i.
	const size_t wlen    = (size_t)keep + n;
	const size_t wstride = (wlen + 3) & ~(size_t)3;
	// Coefficient prefix per channel: what is left of the last completed
	// partition, then every partition that completes in this call while the
	// angle is still moving.  Everything after it uses the steady (ca, sa).
	const uint32_t first_np = (uint32_t)(t0 / P);                  // partition being filled at t0
	const uint32_t n_comp   = (uint32_t)((t0 + n) / P) - first_np; // partitions completing in this call
	const size_t   pre_cap  = (size_t)P * 20;                      // a full 180 degree ramp is <= 9 partitions (src:295)
	const bool     small    = n <= kSmallCallMax;
	const size_t   n_cta    = (n + kStreamOut - 1) / kStreamOut; // CTAs per channel of the small-call kernel
	int            rc       = h->h_io.ensure (plugin_io_bytes (h, n)); // no-op for small calls: sized in create()
	if (rc) return rc;
	float*  W    = (float*)h->h_io.p;
	float2* pre  = (float2*)(W + wstride * C);
	float*  yout = (float*)(pre + pre_cap * C);
	float*  lev  = yout + (size_t)n * C; // small calls: [C][n_cta][2] per-CTA (max |delayed input|, max |output|)

	float2 chan_cs[2];
	int    ramp_len[2] = { 0, 0 };
	for (int c = 0; c < C; ++c) {
		float* w = W + wstride * c;
		memcpy (w, h->ptail.data () + (size_t)c * keep, sizeof (float) * keep);
		memcpy (w + keep, in[c], sizeof (float) * n);

		PluginChan& ch = h->pch[(size_t)c];
		float target   = angle_deg[c] / -360.f; // src:564-571
		if (target < -.5f) target = -.5f;
		if (target > 0.5f) target = 0.5f;

		float2* pc       = pre + pre_cap * c;
		size_t  plen     = 0; // prefix entries written
		size_t  need_len = 0; // entries that differ from the steady coefficients
		// outputs start at u = t0 - P: before the stream (zero) while t0 < P,
		// otherwise inside the last completed partition
		const uint32_t off0 = (uint32_t)(t0 % P);
		if (t0 < P) {
			for (uint32_t i = off0; i < P; ++i) pc[plen++] = make_float2 (0.f, 0.f);
			need_len = plen;
		} else {
			for (uint32_t i = off0; i < P; ++i) pc[plen++] = ch.last_is_ramp ? ch.last[i] : ch.last_const;
			if (ch.last_is_ramp) need_len = plen;
		}
		for (uint32_t k = 0; k < n_comp; ++k) {
			if (target == ch.angle) {
				// steady from here on: every remaining partition uses (ca, sa)
				ch.last_is_ramp = false;
				ch.last_const   = make_float2 (ch.ca, ch.sa);
				break;
			}
			plugin_partition_coef (h, ch, target, ch.last.data ());
			ch.last_is_ramp = true;
			ch.last_const   = make_float2 (ch.ca, ch.sa);
			if (plen + P > pre_cap) {
				snprintf (g_last_error, sizeof (g_last_error), "angle ramp longer than %zu partitions", pre_cap / P);
				return PHASEROT_E_UNSUPPORTED;
			}
			memcpy (pc + plen, ch.last.data (), sizeof (float2) * P);
			plen += P;
			need_len = plen;
		}
		ramp_len[c] = (int)std::min<size_t> (need_len, (size_t)n);
		chan_cs[c]  = ch.last_const;
		// new tail = last `keep` samples of W
		memcpy (h->ptail.data () + (size_t)c * keep, w + wlen - keep, sizeof (float) * keep);
	}
	h->ppos += n;

	if (small && h->h_io.d) {
		// small call: one launch.  The history stays in a device ring; the kernel
		// reads the n new samples from mapped pinned memory and writes the n
		// outputs back to it.
		const int    nodd = h->Lh;
		const size_t smem = sizeof (float) * (3 * (size_t)nodd + kStreamOut + 128);
		rc = h->d_ring.ensure (sizeof (float) * (size_t)kRing * C);
		if (rc) return rc;
		if (!h->ring_valid) {
			// (re-)seed: W[c][0 .. keep) are stream positions [t0 - keep, t0)
			for (int c = 0; c < C; ++c) {
				float*       r   = (float*)h->d_ring.p + (size_t)c * kRing;
				const float* w   = W + wstride * c;
				uint64_t     i0  = t0 < keep ? keep - t0 : 0; // positions before the stream start are never read
				while (i0 < keep) {
					const uint64_t pos = (t0 - keep + i0) & (kRing - 1);
					const uint64_t cnt = std::min<uint64_t> (keep - i0, kRing - pos);
					CK (cudaMemcpyAsync (r + pos, w + i0, sizeof (float) * cnt, cudaMemcpyHostToDevice, h->stream));
					i0 += cnt;
				}
			}
			h->ring_valid = true;
		}
		const char*   dbase = (const char*)h->h_io.d;
		const float*  dW    = (const float*)dbase;
		const float2* dpre  = (const float2*)(dbase + ((const char*)pre - (const char*)h->h_io.p));
		float*        dy    = (float*)(dbase + ((const char*)yout - (const char*)h->h_io.p));
		float*        dlev  = want_levels ? (float*)(dbase + ((const char*)lev - (const char*)h->h_io.p)) : nullptr;
		FirCoef       fc;
		for (int c = 0; c < 2; ++c) {
			fc.cs[c]   = chan_cs[c < C ? c : 0];
			fc.rlen[c] = ramp_len[c < C ? c : 0];
		}
		const dim3 grid ((n + kStreamOut - 1) / kStreamOut, (unsigned)C);
		{
			ProfScope ps (h, 4);
			fir_stream_kernel<<<grid, 128, smem, h->stream>>> ((float*)h->d_ring.p, dW + keep, (int)wstride, (int)n, (long long)t0, (int)P,
			                                                    (const float*)h->d_g.p, nodd, (int)h->firlat, dpre, (int)pre_cap, fc, dy, dlev);
		}
		CK (cudaGetLastError ());
		++h->stats.kernel_launches;
		CK (cudaStreamSynchronize (h->stream));
		for (int c = 0; c < C; ++c) {
			memcpy (out[c], yout + (size_t)c * n, sizeof (float) * n);
			if (want_levels) {
				float li = 0.f, lo = 0.f;
				for (size_t b = 0; b < n_cta; ++b) { // 32 values per 1024-frame call
					li = std::fmax (li, lev[2 * ((size_t)c * n_cta + b)]);
					lo = std::fmax (lo, lev[2 * ((size_t)c * n_cta + b) + 1]);
				}
				level_in[c]  = li;
				level_out[c] = lo;
			}
		}
		h->stats.h2d_bytes += sizeof (float) * (size_t)n * C;
		h->stats.d2h_bytes += sizeof (float) * (size_t)n * C;
		return PHASEROT_OK;
	}
	h->ring_valid = false; // the bulk path does not maintain the ring

	// bulk call: FFT convolution over W (planar already: one "channel-major" upload)
	{
		const long long t_end = (long long)wlen; // outputs wanted: W indices [firlen, wlen)
		const long long m_end = (t_end + 1) / 2;
		long long       nseg  = 0;
		rc                    = ensure_planes (h, m_end, &nseg);
		if (rc) return rc;
		rc = init_front_pad (h, nullptr);
		if (rc) return rc;
		const long long n_fill = nseg * h->V;
		for (int c = 0; c < C; ++c) {
			float2* pl = (float2*)h->d_plane.p + (long long)c * h->plane_stride + h->padf;
			CK (cudaMemcpyAsync (pl, W + wstride * c, sizeof (float) * wlen, cudaMemcpyHostToDevice, h->stream));
			const long long have = (long long)(wlen / 2); // whole complex elements copied
			if (wlen & 1) {
				// odd tail sample: its partner must read as zero
				CK (cudaMemsetAsync ((float*)(pl + have) + 1, 0, sizeof (float), h->stream));
			}
			const long long from = (long long)((wlen + 1) / 2);
			if (n_fill > from) {
				CK (cudaMemsetAsync (pl + from, 0, sizeof (float2) * (size_t)(n_fill - from), h->stream));
			}
		}
		h->stats.h2d_bytes += sizeof (float) * wlen * C;
		h->out_stride = (m_end + 3) & ~3LL;
		rc            = h->d_out.ensure (sizeof (float2) * (size_t)h->out_stride * C);
		if (rc) return rc;
		rc = h->d_chancs.ensure (sizeof (float2) * (size_t)C);
		if (rc) return rc;
		// ramp table indexed by W sample index: prefix starts at W index firlen
		size_t rmax = 0;
		for (int c = 0; c < C; ++c) rmax = std::max (rmax, (size_t)ramp_len[c]);
		const long long rstride = (long long)((firlen + rmax + 3) & ~(size_t)3);
		std::vector<float2> ramp ((size_t)rstride * C, make_float2 (0.f, 0.f));
		std::vector<int>    rl ((size_t)C);
		for (int c = 0; c < C; ++c) {
			memcpy (ramp.data () + (size_t)rstride * c + firlen, pre + pre_cap * c, sizeof (float2) * (size_t)ramp_len[c]);
			rl[(size_t)c] = (int)firlen + ramp_len[c];
		}
		rc = h->d_ramp.ensure (sizeof (float2) * ramp.size ());
		if (rc) return rc;
		CK (cudaMemcpyAsync (h->d_ramp.p, ramp.data (), sizeof (float2) * ramp.size (), cudaMemcpyHostToDevice, h->stream));
		CK (cudaMemcpyAsync (d_ramplen (h), rl.data (), sizeof (int) * (size_t)C, cudaMemcpyHostToDevice, h->stream));
		CK (cudaMemcpyAsync (h->d_chancs.p, chan_cs, sizeof (float2) * (size_t)C, cudaMemcpyHostToDevice, h->stream));
		CK (cudaStreamSynchronize (h->stream));

		ConvParams p;
		fill_conv_common (h, p);
		p.chan0       = 0;
		p.nchan       = C;
		p.seg0        = 0;
		p.nseg        = nseg;
		p.m_end       = m_end;
		p.out         = (float2*)h->d_out.p;
		p.out_stride  = h->out_stride;
		p.cs          = (const float2*)h->d_chancs.p;
		p.ramp        = (const float2*)h->d_ramp.p;
		p.ramp_stride = rstride;
		p.ramp_len    = d_ramplen (h);
		rc            = launch_conv<EPI_RENDER> (h, p);
		if (rc) return rc;
		// outputs live at W sample indices [firlen, firlen + n): plain float view of d_out
		for (int c = 0; c < C; ++c) {
			const float* src = (const float*)((float2*)h->d_out.p + (long long)c * h->out_stride) + firlen;
			CK (cudaMemcpyAsync (out[c], src, sizeof (float) * n, cudaMemcpyDeviceToHost, h->stream));
		}
		unsigned levbits[4] = { 0, 0, 0, 0 };
		if (want_levels) {
			// level meters: the delayed input of output i is W index firlen - firlat + i (plane, float view)
			unsigned* dl = (unsigned*)d_thr2 (h); // [C][2] scratch in the small-state buffer (unused in plugin mode)
			CK (cudaMemsetAsync (dl, 0, sizeof (unsigned) * 2 * (size_t)C, h->stream));
			const float* xa = (const float*)((float2*)h->d_plane.p + h->padf) + (firlen - h->firlat);
			const float* ya = (const float*)h->d_out.p + firlen;
			const dim3   grid ((unsigned)std::min<size_t> (((size_t)n + 255) / 256, (size_t)h->n_sm * 4), (unsigned)C);
			absmax2_kernel<<<grid, 256, 0, h->stream>>> (xa, 2 * h->plane_stride, ya, 2 * h->out_stride, (long long)n, dl);
			CK (cudaGetLastError ());
			++h->stats.kernel_launches;
			CK (cudaMemcpyAsync (levbits, dl, sizeof (unsigned) * 2 * (size_t)C, cudaMemcpyDeviceToHost, h->stream));
		}
		CK (cudaStreamSynchronize (h->stream));
		for (int c = 0; want_levels && c < C; ++c) {
			memcpy (&level_in[c], &levbits[2 * c], sizeof (float));
			memcpy (&level_out[c], &levbits[2 * c + 1], sizeof (float));
		}
		h->stats.d2h_bytes += sizeof (float) * (size_t)n * C;
	}
	return PHASEROT_OK;
}

// ---------------------------------------------------------------------------
// device group: one stream, several GPUs of one process (sample-range shards)
// ---------------------------------------------------------------------------
} // extern "C"

struct phaserot_group {
	std::vector<phaserot*>   h;
	std::vector<cudaEvent_t> ev;   // "sweep of device i enqueued work is complete", recorded on h[i]->stream
	std::vector<char>        peer; // device 0 can read device i's memory directly
	DevBuf                   d_gather; // device 0: copies of the other tables when peer access is missing
};

namespace {

// float32 history in front of a shard from a host stream in any PHASEROT_PCM_* format
void
shard_history (const void* data, int fmt, long long f0, int L, int C, std::vector<float>& out)
{
	out.resize ((size_t)L * C);
	const size_t n = (size_t)L * C, i0 = (size_t)(f0 - L) * C;
	switch (fmt) {
		case PHASEROT_PCM_S16: {
			const int16_t* q = (const int16_t*)data + i0;
			for (size_t i = 0; i < n; ++i) out[i] = (float)q[i] * (1.f / 32768.f);
		} break;
		case PHASEROT_PCM_S32: {
			const int32_t* q = (const int32_t*)data + i0;
			for (size_t i = 0; i < n; ++i) out[i] = (float)q[i] * (1.f / 2147483648.f);
		} break;
		case PHASEROT_PCM_S24: {
			const uint8_t* q = (const uint8_t*)data + 3 * i0;
			for (size_t i = 0; i < n; ++i) {
				const int32_t v = (int32_t)(((uint32_t)q[3 * i] << 8) | ((uint32_t)q[3 * i + 1] << 16) | ((uint32_t)q[3 * i + 2] << 24));
				out[i]          = (float)v * (1.f / 2147483648.f);
			}
		} break;
		default: memcpy (out.data (), (const float*)data + i0, sizeof (float) * n); break;
	}
}

} // namespace

extern "C" {

int
phaserot_group_create (phaserot_group_t** out, const phaserot_cfg_t* cfg, const int* devices, int n_devices)
{
	if (!out) {
		return PHASEROT_E_INVAL;
	}
	*out = nullptr;
	if (!cfg || n_devices < 1 || n_devices > 16 || cfg->mode != PHASEROT_MODE_CLI) {
		return PHASEROT_E_INVAL;
	}
	phaserot_group* g = new (std::nothrow) phaserot_group ();
	if (!g) {
		return PHASEROT_E_NOMEM;
	}
	// PHASEROT_GROUP_DEVICES="0,0,1": device list override when the caller passes none
	// (lets a one-GPU box exercise `phase-rotate --gpus 2`: two handles on one device)
	std::vector<int> env_dev;
	if (!devices) {
		if (const char* e = getenv ("PHASEROT_GROUP_DEVICES")) {
			for (const char* q = e; *q;) {
				env_dev.push_back (atoi (q));
				while (*q && *q != ',') ++q;
				if (*q == ',') ++q;
			}
			if ((int)env_dev.size () >= n_devices) {
				devices = env_dev.data ();
			}
		}
	}
	int rc = PHASEROT_OK;
	for (int i = 0; i < n_devices && rc == PHASEROT_OK; ++i) {
		phaserot_cfg_t c = *cfg;
		c.device         = devices ? devices[i] : i;
		phaserot*      h = nullptr;
		rc               = phaserot_create (&h, &c);
		if (rc == PHASEROT_OK) {
			g->h.push_back (h);
			DevGuard    guard (h->dev);
			cudaEvent_t e = nullptr;
			if (cudaEventCreateWithFlags (&e, cudaEventDisableTiming) != cudaSuccess) {
				rc = PHASEROT_E_CUDA;
			}
			g->ev.push_back (e);
		}
	}
	if (rc == PHASEROT_OK) {
		// peer access from the first device to the others (NVLink / NVSwitch on a B200 box)
		g->peer.assign (g->h.size (), 0);
		DevGuard guard (g->h[0]->dev);
		for (size_t i = 1; i < g->h.size (); ++i) {
			int can = 0;
			if (g->h[i]->dev == g->h[0]->dev) {
				g->peer[i] = 1;
			} else if (cudaDeviceCanAccessPeer (&can, g->h[0]->dev, g->h[i]->dev) == cudaSuccess && can) {
				const cudaError_t e = cudaDeviceEnablePeerAccess (g->h[i]->dev, 0);
				if (e == cudaSuccess || e == cudaErrorPeerAccessAlreadyEnabled) {
					g->peer[i] = 1;
				}
				cudaGetLastError ();
			}
		}
	}
	if (rc != PHASEROT_OK) {
		phaserot_group_destroy (g);
		return rc;
	}
	*out = g;
	return PHASEROT_OK;
}

void
phaserot_group_destroy (phaserot_group_t* g)
{
	if (!g) {
		return;
	}
	for (size_t i = 0; i < g->h.size (); ++i) {
		if (i < g->ev.size () && g->ev[i]) {
			DevGuard guard (g->h[i]->dev);
			cudaEventDestroy (g->ev[i]);
		}
	}
	if (!g->h.empty ()) {
		DevGuard guard (g->h[0]->dev);
		g->d_gather.release ();
	}
	for (phaserot* h : g->h) {
		phaserot_destroy (h);
	}
	delete g;
}

int
phaserot_group_size (const phaserot_group_t* g)
{
	return g ? (int)g->h.size () : 0;
}

phaserot_t*
phaserot_group_handle (phaserot_group_t* g, int i)
{
	return (g && i >= 0 && (size_t)i < g->h.size ()) ? g->h[(size_t)i] : nullptr;
}

int
phaserot_group_reset (phaserot_group_t* g)
{
	if (!g) {
		return PHASEROT_E_INVAL;
	}
	for (phaserot* h : g->h) {
		const int rc = phaserot_reset (h);
		if (rc) return rc;
	}
	return PHASEROT_OK;
}

int
phaserot_group_sweep (phaserot_group_t* g, const void* data, int format, uint64_t n_frames, int ang_start, int ang_end, int ang_stride, int chn)
{
	if (!g || (!data && n_frames) || format < PHASEROT_PCM_F32 || format > PHASEROT_PCM_S24) {
		return PHASEROT_E_INVAL;
	}
	phaserot*       h0    = g->h[0];
	const int       n     = (int)g->h.size ();
	const long long F     = (long long)n_frames;
	const long long align = (long long)phaserot_shard_align (h0);
	// equal shards cut on the FFT segment grid; short files use fewer devices
	long long per = (F + n - 1) / n;
	per           = std::max (align, (per + align - 1) / align * align);
	const int used = (int)std::max<long long> (1, std::min<long long> (n, (F + per - 1) / per));

	std::vector<int>         rcs ((size_t)used, PHASEROT_OK);
	std::vector<std::string> errs ((size_t)used);
	auto shard = [&] (int i) {
		phaserot*       h   = g->h[(size_t)i];
		const long long f0  = (long long)i * per;
		const long long nf  = std::max<long long> (0, std::min (per, F - f0));
		const bool      lst = i == used - 1;
		std::vector<float> hist;
		if (i > 0) {
			shard_history (data, format, f0, h->L, h->C, hist);
		}
		DevGuard guard (h->dev);
		int      rc = sweep_core (h, shard_job ((const char*)data + pcm_bytes (format) * (size_t)f0 * h->C, false, format, nf, i > 0 ? hist.data () : nullptr,
		                                        i == 0, lst, ang_start, ang_end, ang_stride, chn), Pass::Fresh);
		if (rc == PHASEROT_OK) {
			rc = complete_pending (h); // a shard whose survivor list overflowed is repeated in dense mode before the tables are combined
		}
		if (rc == PHASEROT_OK && cudaEventRecord (g->ev[(size_t)i], h->stream) != cudaSuccess) {
			rc = PHASEROT_E_CUDA;
		}
		rcs[(size_t)i]  = rc;
		errs[(size_t)i] = g_last_error; // thread-local in the worker
	};
	// one host thread per device: the chunked uploads of all shards are in flight together
	std::vector<std::thread> th;
	for (int i = 1; i < used; ++i) th.emplace_back (shard, i);
	shard (0);
	for (auto& t : th) t.join ();
	for (int i = 0; i < used; ++i) {
		if (rcs[(size_t)i]) {
			snprintf (g_last_error, sizeof (g_last_error), "device %d: %s", g->h[(size_t)i]->dev, errs[(size_t)i].c_str ());
			return rcs[(size_t)i];
		}
	}
	// handles that got no shard keep an empty table
	if (used > 1) {
		DevGuard     guard (h0->dev);
		const size_t cnt = (size_t)std::max (h0->pend_A, 1) * h0->C + (size_t)h0->C + 1; // maxima, raw peaks, overflow flag (clear: every shard was completed above)
		PeerTabs     pt;
		pt.n = 0;
		size_t n_copy = 0;
		for (int i = 1; i < used; ++i) n_copy += g->peer[(size_t)i] ? 0 : 1;
		if (n_copy) {
			const int rc = g->d_gather.ensure (sizeof (unsigned) * cnt * n_copy);
			if (rc) return rc;
		}
		size_t slot = 0;
		for (int i = 1; i < used; ++i) {
			phaserot* h = g->h[(size_t)i];
			CK (cudaStreamWaitEvent (h0->stream, g->ev[(size_t)i], 0));
			if (g->peer[(size_t)i]) {
				pt.p[pt.n++] = (const unsigned*)h->d_peaks.p;
			} else {
				unsigned* dst = (unsigned*)g->d_gather.p + cnt * slot++;
				CK (cudaMemcpyPeerAsync (dst, h0->dev, h->d_peaks.p, h->dev, sizeof (unsigned) * cnt, h0->stream));
				pt.p[pt.n++] = dst;
			}
		}
		{
			ProfScope ps (h0, 5);
			peer_max_kernel<<<(unsigned)((cnt + 255) / 256), 256, 0, h0->stream>>> ((unsigned*)h0->d_peaks.p, pt, (long long)cnt);
		}
		CK (cudaGetLastError ());
		++h0->stats.kernel_launches;
	}
	int rc = finish_pending (h0);
	if (rc) return rc;
	for (int i = 1; i < used; ++i) {
		// the other devices' tables have been consumed on device 0 (finish_pending waited for it)
		phaserot* h = g->h[(size_t)i];
		DevGuard  guard (h->dev);
		CK (cudaStreamSynchronize (h->stream));
		prof_resolve (h);
		h->pending = false;
	}
	return PHASEROT_OK;
}

int
phaserot_group_peaks (phaserot_group_t* g, float* out)
{
	if (!g || !out) {
		return PHASEROT_E_INVAL;
	}
	return phaserot_peaks (g->h[0], out);
}

void*
phaserot_alloc_host (uint64_t bytes)
{
	void* p = nullptr;
	if (cudaHostAlloc (&p, bytes ? bytes : 1, cudaHostAllocPortable) != cudaSuccess) { // page-locked for every device (device groups)
		cudaGetLastError ();
		return nullptr;
	}
	return p;
}

void
phaserot_free_host (void* p)
{
	if (p) {
		cudaFreeHost (p);
	}
}

int
phaserot_get_stats (phaserot_t* h, phaserot_stats_t* out)
{
	if (!h || !out) {
		return PHASEROT_E_INVAL;
	}
	*out = h->stats;
	return PHASEROT_OK;
}

int
phaserot_reset_stats (phaserot_t* h)
{
	if (!h) {
		return PHASEROT_E_INVAL;
	}
	memset (&h->stats, 0, sizeof (h->stats));
	return PHASEROT_OK;
}

} // extern "C"
