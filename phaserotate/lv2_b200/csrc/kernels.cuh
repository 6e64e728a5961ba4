// Device code of libphaserot_cuda (sm_100a).
//
// K0 deinterleave_kernel   interleaved frames -> planar "complex" planes
// K1 fftconv_kernel        Hilbert FIR as overlap-save FFT convolution in shared
//                          memory, with fused epilogues:
//                            EPI_POINTS  analytic pair (x_d, h) -> exact radius
//                                        filter -> compacted survivor list
//                            EPI_RENDER  y = ca * x_d + sa * h  (K4)
//                            EPI_HILBERT h only (tests / diagnostics)
// K3 sweep_kernel          every angle over a survivor list, angles in lanes,
//                          running max in registers, one atomicMax per angle/CTA
//    threshold_kernel      min over angles of the running peaks -> next filter radius
//    fir_stream_kernel     small-call plugin path: direct-form FIR + rotate, history in a device ring
//    truepeak_kernel       oversampled true-peak front end of the sweep
//
// Data layout.  A channel's samples x[0..F) are viewed as complex numbers
// z[n] = x[2n] + i x[2n+1] ("plane", float2, with a zero front pad).  The
// reference FIR (cli/phase-rotate.cc:144-161, src/phaserotate.c:374-391) has
// non-zero taps only at odd k, so with g[j] = fir[2j+1]
//     w = z (*) g        (complex sequence, real taps, Lh = L/2 taps)
//     H[2m+1] = Re w[m],  H[2m] = Im w[m-1],
// i.e. one complex FFT convolution of half the length yields the Hilbert branch
// of two real samples per point with no real/complex split step.  The delayed
// direct branch x_d[t] = x[t - L/2] is z[m - Lh/2] (cli:220, src:665-671).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include "fft16k.cuh"
#include "tmem_stash.cuh"

namespace prk {

constexpr int kXchFloats = 16 * 32;                                   // Im of lane 31's outputs, per warp
constexpr int kRedThr    = 24;                                       // slot of the launch's squared filter radius
constexpr int kRedFloats = 32;                                       // block reductions (filter radius, bootstrap gate)
constexpr int kTidOff    = kXchFloats + 4 + kRedFloats;               // lane ids [32] | warp bases [16], see opaque_tid()
// 133456 bytes: with the 1 KB the system reserves per CTA this stays inside the
// 132 KB shared-memory carve-out, which leaves 124 KB of L1 to the twiddle
// tables (measured: every carve-out step up costs 1.5 - 6 % of the kernel)
constexpr int kSmemBytes = kM * (int)sizeof (float2) + (kTidOff + 48) * (int)sizeof (float);
static_assert (kSmemBytes + 1024 <= 132 * 1024, "fftconv_kernel must fit the 132 KB carve-out");

// EPI_SECT_*: the same epilogues with rows by section (phaserot_sweep_sections, phaserot_render_sections):
// the row of a segment is section * nchan + channel, see ConvParams::sect_segs
enum { EPI_POINTS = 0, EPI_RENDER = 1, EPI_HILBERT = 2, EPI_SECT_POINTS = 3, EPI_SECT_RENDER = 4 };
__host__ __device__ constexpr bool epi_points (int e) { return e == EPI_POINTS || e == EPI_SECT_POINTS; }
__host__ __device__ constexpr bool epi_render (int e) { return e == EPI_RENDER || e == EPI_SECT_RENDER; }
__host__ __device__ constexpr bool epi_sect (int e) { return e == EPI_SECT_POINTS || e == EPI_SECT_RENDER; }

enum { SRC_PLANE = 0, SRC_INTER = 1 };

struct ConvParams {
	const float2* plane;        // SRC_PLANE: [n_chan][plane_stride], element (padf + n) = z[n]
	long long     plane_stride;
	int           padf;
	const float*  inter;        // SRC_INTER: interleaved frames [n_frames][C], frame 0 = stream position 0
	const float*  hist;         // SRC_INTER: interleaved frames [-2 Lh, 0) preceding the stream, or nullptr (silence)
	long long     n_frames;     // SRC_INTER: frames present in `inter`
	int           C;            // SRC_INTER: channels per frame
	const float2* G;            // [kM] filter spectrum / kM in MID-pass order (fft16k_tables.h)
	const float2* tw1;          // [10][512]  W_M^(e a), a = 1..7 | W_M^(8 e b), b = 1..3
	const float2* tw2;          // [15][32]   W_512^(j q2), j = 1..15
	int           Lh;           // overlap of consecutive segments = half taps of one partition (multiple of 512)
	int           V;            // valid complex outputs per segment = kM - Lh
	int           dl;           // delay of the direct branch in complex points = (all half taps) / 2
	int           hist_frames;  // SRC_INTER: frames in `hist` (= FIR length)
	const float2* G1;           // two partitions: spectrum of the second half of the taps (same order as G)
	float4*       scratch;      // two partitions: [gridDim.x][kM / 2] spectrum of the previous segment, per CTA
	int           chan0;        // first channel of this launch
	long long     seg0;         // first segment
	long long     seg_stride;   // segment index step (1 = contiguous; > 1 = sparse bootstrap sample)
	int           seg_jitter;   // sparse sample: pseudo-random offset in [0, seg_stride) per segment, so that the
	                            // sample cannot lock onto a periodic envelope of the programme
	long long     nseg;         // segments per channel in this launch
	int           nchan;
	long long     m_end;        // outputs exist for complex index m < m_end
	long long     m_skip;       // m <  m_skip : not examined            (first-block rule, cli:418-419)
	long long     m_zero;       // m <  m_zero : direct branch forced to 0
	// EPI_POINTS
	float2*       list;         // [n_chan][list_stride]
	long long     list_stride;
	unsigned*     count;        // [n_chan]
	unsigned      list_cap;     // points that fit a channel's list; survivors beyond it are dropped and *overflow is set
	unsigned*     overflow;     // [1] the pass is incomplete: the host repeats it in dense mode (launches sized to the list)
	const float*  thr2;         // [n_chan] squared filter radius (thr_mode < 0: written by threshold_kernel)
	unsigned*     rawpeak;      // [n_chan] bits of max |x|
	// EPI_POINTS, thr_mode >= 0: the filter radius is derived inside the kernel from the
	// running peaks (what threshold_kernel computes), 0 keep every point, 1 prune, 2 drop every point
	int             thr_mode;
	const unsigned* peaks;      // [n_chan][peaks_stride] float bits of the running per-angle maxima
	int             peaks_stride, A;
	unsigned*       count_reset; // [n_chan] counters of the previous launch's list (already swept): zeroed here
	// bootstrap launch: additionally gate on boot_beta * (largest squared radius seen so far
	// in this launch, r2max[c]) - only the strongest points of the sampled segments are kept
	float           boot_beta;
	unsigned*       r2max;      // [n_chan] float bits
	// EPI_RENDER / EPI_HILBERT
	float2*       out;          // [n_chan][out_stride], element m
	long long     out_stride;
	const float2* cs;           // [n_chan] (ca, sa) steady state
	const float2* ramp;         // [n_chan][ramp_stride] per-sample (ca, sa) for t < ramp_len[c]
	long long     ramp_stride;
	const int*    ramp_len;     // [n_chan] (in samples, even) or nullptr
	float*        out_inter;    // EPI_RENDER: interleaved destination [out_frames][C] instead of `out` (fused CLI render)
	long long     out_frames;
	int           out_compact;  // EPI_HILBERT: segment j of the launch writes its V outputs at out[8 + j V ..) (true-peak staging)
	int           prefetch;     // > 0: L2 prefetch distance in segments (experiments; 0 = off, the default)
	// EPI_SECT_*: segment seg lies in section min (seg / sect_segs, n_sect - 1) (sections start on segment
	// boundaries; the last one takes the remainder); thr2, list, count, overflow, rawpeak and r2max are
	// indexed by row = section * nchan + (channel - chan0) instead of by channel
	long long     sect_segs;
	int           n_sect;
	int           sect_boot;    // EPI_SECT_POINTS bootstrap launch: segment si of the launch samples section si / sect_boot
	const float2* sect_cs;      // EPI_SECT_RENDER: [n_sect][C] steady-state (ca, sa)
	const int*    sect_ang;     // EPI_SECT_RENDER: [n_sect][C] angles in grid steps; the first hist_frames samples of a
	                            // section k > 0 ramp linearly from the angle of section k - 1
	float         ang_mp;       // EPI_SECT_RENDER: radians per grid step (the SinCosLut constant)
};

// Segment input loaders: z[n0 + idx] for the first forward pass and the direct
// branch of the epilogue.  `thread (e)` binds the per-thread part of the address
// once; the returned object is then indexed with compile-time offsets (512 k),
// which become immediate offsets of the load instructions.
// The input is streamed: every byte is used once per CTA, so it bypasses L1
// (no_allocate) and leaves the cache to the twiddle tables, which every segment
// reads again.
__device__ __forceinline__ float2 ldg_stream (const float2* p)
{
	float2 v;
	asm volatile ("ld.global.nc.L1::no_allocate.v2.f32 {%0, %1}, [%2];" : "=f"(v.x), "=f"(v.y) : "l"(p));
	return v;
}
__device__ __forceinline__ float4 ldg_stream (const float4* p)
{
	float4 v;
	asm volatile ("ld.global.nc.L1::no_allocate.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p));
	return v;
}
struct PlaneLoader { // planar float2 stream
	const float2* src;
	struct T {
		const float2* p;
		__device__ __forceinline__ float2 operator() (int off) const { return ldg_stream (p + off); }
	};
	__device__ __forceinline__ T thread (int e) const { return T { src + e }; }
};
typedef PlaneLoader Inter1Loader; // mono: the interleaved stream is the plane
struct Inter2Loader { // stereo: one 16 byte load = frames 2n, 2n+1 of both channels
	const float4* src;
	int           chan;
	struct T {
		const float4* p;
		int           chan;
		__device__ __forceinline__ float2 operator() (int off) const
		{
			const float4 v = ldg_stream (p + off);
			return chan ? make_float2 (v.y, v.w) : make_float2 (v.x, v.z);
		}
	};
	__device__ __forceinline__ T thread (int e) const { return T { src + e, chan }; }
};
struct InterNLoader { // any channel count, two scalar loads
	const float* src; // &inter[(2 n0) * C + c]
	int          C;
	struct T {
		const float* p;
		int          C;
		__device__ __forceinline__ float2 operator() (int off) const
		{
			const float* a = p + (long long)(2 * off) * C;
			return make_float2 (__ldg (a), __ldg (a + C));
		}
	};
	__device__ __forceinline__ T thread (int e) const { return T { src + (long long)(2 * e) * C, C }; }
};
struct EdgeLoader { // segments that touch the stream start (history / silence) or its end (zero padding)
	const float* inter;
	const float* hist;
	long long    n_frames, f0; // f0 = frame index of idx 0 (= 2 n0)
	int          C, c, L;      // L = frames of history available
	__device__ __forceinline__ float at (long long f) const
	{
		if (f >= 0) return f < n_frames ? __ldg (inter + f * C + c) : 0.f;
		return (hist && f >= -(long long)L) ? __ldg (hist + (L + f) * C + c) : 0.f;
	}
	struct T {
		const EdgeLoader* l;
		int               e;
		__device__ __forceinline__ float2 operator() (int off) const
		{
			const long long f = l->f0 + 2 * (long long)(e + off);
			return make_float2 (l->at (f), l->at (f + 1));
		}
	};
	__device__ __forceinline__ T thread (int e) const { return T { this, e }; }
};

__device__ __forceinline__ unsigned lanemask_lt ()
{
	unsigned m;
	asm ("mov.u32 %0, %%lanemask_lt;" : "=r"(m));
	return m;
}

// ---------------------------------------------------------------------------
// K1: FFT convolution with fused epilogue.  Persistent: one CTA per SM walks
// (channel, segment) pairs.
// ---------------------------------------------------------------------------
// warp-aggregated append of up to two points per lane to the survivor list
struct ListDst {
	float2*   lst;
	unsigned* cnt;
	unsigned  cap;
	unsigned* ovf;
};
__device__ __forceinline__ void append_points (const ListDst& d, bool k0, float2 p0, bool k1, float2 p1, unsigned lt, int lane)
{
	const unsigned b0 = __ballot_sync (0xffffffffu, k0);
	const unsigned b1 = __ballot_sync (0xffffffffu, k1);
	if (b0 | b1) {
		const int n0   = __popc (b0);
		unsigned  base = 0;
		if (lane == 0) {
			base = atomicAdd (d.cnt, (unsigned)(n0 + __popc (b1)));
			if (base + (unsigned)(n0 + __popc (b1)) > d.cap) *d.ovf = 0x3f800000u; // rare: the pass is repeated in dense mode (bits of 1.0f: the flag is a table element)
		}
		base = __shfl_sync (0xffffffffu, base, 0);
		const unsigned i0 = base + __popc (b0 & lt), i1 = base + n0 + __popc (b1 & lt);
		if (k0 && i0 < d.cap) d.lst[i0] = p0;
		if (k1 && i1 < d.cap) d.lst[i1] = p1;
	}
}

// The same for the eight samples a lane holds of one block of four strides: ONE reservation per warp
// and block.  On material where most samples survive (dense mode) the list counter is the
// bottleneck of the kernel: same-address atomics retire at ~1 per ns.
__device__ __forceinline__ void append_points4 (const ListDst& d, const bool (&k0)[4], const float2 (&p0)[4], const bool (&k1)[4], const float2 (&p1)[4], unsigned lt, int lane)
{
	unsigned b[8];
	int      n = 0;
#pragma unroll
	for (int kk = 0; kk < 4; ++kk) {
		b[2 * kk]     = __ballot_sync (0xffffffffu, k0[kk]);
		b[2 * kk + 1] = __ballot_sync (0xffffffffu, k1[kk]);
		n += __popc (b[2 * kk]) + __popc (b[2 * kk + 1]);
	}
	unsigned base = 0;
	if (lane == 0) {
		base = atomicAdd (d.cnt, (unsigned)n);
		if (base + (unsigned)n > d.cap) *d.ovf = 0x3f800000u;
	}
	base = __shfl_sync (0xffffffffu, base, 0);
#pragma unroll
	for (int kk = 0; kk < 4; ++kk) {
		const unsigned i0 = base + __popc (b[2 * kk] & lt);
		base += __popc (b[2 * kk]);
		const unsigned i1 = base + __popc (b[2 * kk + 1] & lt);
		base += __popc (b[2 * kk + 1]);
		if (k0[kk] && i0 < d.cap) d.lst[i0] = p0[kk];
		if (k1[kk] && i1 < d.cap) d.lst[i1] = p1[kk];
	}
}

// Epilogue state shared by the loader-specific instantiations.
struct EpiCtx {
	int       c, i_hi, i_skip, i_zero;
	long long mbase, obase; // complex stream index / output index of local index 0
	float     rawmax;
	int       row;          // EPI_SECT_*: row of the segment
	long long t_sect;       // EPI_SECT_RENDER: first output sample of the segment's section
};

// (ca, sa) of sample j of the ramp into the section of row `row` (EPI_SECT_RENDER):
// phi = a[k-1] + (a[k] - a[k-1]) (j + 1) / L grid steps
__device__ __forceinline__ float2 sect_ramp_cs (const ConvParams& p, int row, long long j)
{
	const int   a0  = p.sect_ang[row - p.nchan], a1 = p.sect_ang[row];
	const float phi = (float)a0 + (float)(a1 - a0) * (float)(j + 1) / (float)p.hist_frames;
	float       s, c;
	sincosf (phi * p.ang_mp, &s, &c);
	return make_float2 (c, s);
}

// Epilogue straight from the registers of the last inverse pass: thread e holds
// the outputs w[k] of local index i = e + 512 k; valid ones have i in [Lh, i_hi),
// complex index m = mbase + i.
//   H[2m] = Im w[m-1], H[2m+1] = Re w[m];  direct branch x_d pair = z[m - Lh/2] = ld (i - Lh/2).
// Im w[i-1] comes from the neighbouring lane (shuffle), for lane 0 from the
// previous warp through `xch` (written by every lane 31 before the barrier).
struct TmemStash {
	uint32_t tb;
	__device__ __forceinline__ void operator() (int k, float2 a, float2 b, float2 c, float2 d) const { tmem_st4 (tb + 2 * k, a, b, c, d); }
};

// Filter spectrum of the thread's two MID rows, parked in TMEM columns
// kTmemGCol .. kTmemGCol + 63 by fftconv_kernel before the first segment.
struct GTmem {
	uint32_t tb;
	uint32_t r[32];
	__device__ __forceinline__ void issue (int h) { tmem_ld16_issue (tb + kTmemGCol + 32 * h, r); }
	__device__ __forceinline__ void get (float4 (&g)[8])
	{
		tmem_wait_ld16 (r);
#pragma unroll
		for (int c = 0; c < 8; ++c) {
			g[c] = make_float4 (__uint_as_float (r[4 * c]), __uint_as_float (r[4 * c + 1]), __uint_as_float (r[4 * c + 2]), __uint_as_float (r[4 * c + 3]));
		}
	}
};

// Overlap-save reuse: a CTA walks consecutive segments of one channel, so the
// first Lh points of a segment are the last Lh of the previous one - still in
// the TMEM stash (input k of the previous segment sits in columns 2k, 2k + 1).
// `rows` = Lh / 512 when the previous segment is the stream predecessor, else 0;
// `shift` = V / 512.
struct TmemReuse {
	uint32_t tb;
	int      rows, shift;
	__device__ __forceinline__ bool operator() (int k, float2 (&v)[4]) const
	{
		if (k >= rows) return false;
		tmem_ld4 (tb + 2 * (k + shift), v);
		return true;
	}
};

// The stash serves the epilogue when the delay Lh/2 is a multiple of 2048 points:
// output block kb .. kb + 3 then needs the aligned input block kb - Lh/1024 of
// the same thread (Lh = 4096 and 8192, i.e. the CLI block sizes 8192 and 16384).
__device__ __forceinline__ bool stash_usable (int dl) { return (dl & 2047) == 0; }

// The direct-branch inputs of outputs k .. k + 3: from the TMEM stash when the
// delay Lh/2 is a whole number of 512-point strides (then they are inputs
// k - Lh/1024 .. of the same thread), else re-read through the loader.
template <class Loader>
__device__ __forceinline__ void load_direct (float2 (&zd)[4], const bool (&ok)[4], int tid, int kb, int dl, uint32_t tb, const Loader& ld)
{
	if (stash_usable (dl)) {
		tmem_ld4 (tb + 2 * (kb - (dl >> 9)), zd);
	} else {
		const auto lt = ld.thread (tid - dl);
#pragma unroll
		for (int kk = 0; kk < 4; ++kk) zd[kk] = ok[kk] ? lt (512 * (kb + kk)) : make_float2 (0.f, 0.f);
	}
}

// Bounds-checked walk over the outputs of a segment (segments at the stream edges,
// delays that are not a multiple of the stash stride, and the bootstrap pre-pass):
// f (p0, p1, in, ok, zd) per output pair i = tid + 512 k, where p0 / p1 are the
// analytic pairs of samples 2m and 2m + 1, `ok` = the pair exists, `in` = it is
// also examined (first-block rule), zd = the raw direct-branch inputs.
template <class Loader, class F>
__device__ __forceinline__ void walk_pairs_checked (const float2 (&w)[32], const float* xch, uint32_t tb, const ConvParams& p, int tid, int lane, const EpiCtx& cx, const Loader& ld, F&& f)
{
	const int dl    = p.dl;
	const int warp  = tid >> 5;
	const int xbase = warp ? (warp - 1) * 32 : 15 * 32 - 1;
#pragma unroll 1
	for (int kb = 0; kb < 32; kb += 4) {
		if (512 * (kb + 4) <= p.Lh) continue; // whole block in the overlap region (uniform)
		float2 zd[4];
		bool   ok[4];
#pragma unroll
		for (int kk = 0; kk < 4; ++kk) {
			const int i = tid + 512 * (kb + kk);
			ok[kk]      = i >= p.Lh && i < cx.i_hi;
		}
		load_direct (zd, ok, tid, kb, dl, tb, ld);
#pragma unroll
		for (int kk = 0; kk < 4; ++kk) {
			const int k  = kb + kk;
			const int i  = tid + 512 * k;
			float     wy = w[0].y, wx = w[0].x;
#pragma unroll
			for (int kq = 1; kq < 32; ++kq) { // rare path: select instead of unrolling the block loop
				if (kq == k) {
					wy = w[kq].y;
					wx = w[kq].x;
				}
			}
			float pv = __shfl_up_sync (0xffffffffu, wy, 1);
			if (lane == 0) pv = xch[xbase + k];
			const float2 z = i < cx.i_zero ? make_float2 (0.f, 0.f) : zd[kk];
			f (make_float2 (z.x, pv), make_float2 (z.y, wx), ok[kk] && i >= cx.i_skip, ok[kk], zd[kk]);
		}
	}
}

template <int EPI, class Loader>
__device__ __forceinline__ void epilogue (const float2 (&w)[32], float* xch, uint32_t tb, const ConvParams& p, int tid, int lane, EpiCtx& cx, const Loader& ld)
{
	const int dl    = p.dl;
	const int warp  = tid >> 5;
	const int xbase = warp ? (warp - 1) * 32 : 15 * 32 - 1;
	if (epi_points (EPI)) {
		// (sections: the radius, list and flags of the segment's row)
		const int      row    = epi_sect (EPI) ? cx.row : cx.c;
		float          thr2   = epi_sect (EPI) ? __ldg (p.thr2 + row) : xch[kXchFloats + 4 + kRedThr]; // parked in shared memory by the kernel prologue
		const ListDst  dst    = { p.list + (long long)row * p.list_stride, p.count + row, p.list_cap, epi_sect (EPI) ? p.overflow + row : p.overflow };
		const unsigned lt     = lanemask_lt ();
		float          rawmax = cx.rawmax;
		if (p.boot_beta > 0.f) {
			// Bootstrap launch (uniform branch): largest squared radius of this segment,
			// merged with what the other CTAs of the launch have published so far; only
			// points within boot_beta of it are kept.  Any subset is valid here - the
			// bootstrap only has to raise the running peaks, the contiguous passes
			// visit every segment again.
			float r2m = 0.f;
			walk_pairs_checked (w, xch, tb, p, tid, lane, cx, ld, [&] (float2 p0, float2 p1, bool in, bool, float2) {
				if (in) r2m = fmaxf (r2m, fmaxf (fmaf (p0.x, p0.x, p0.y * p0.y), fmaf (p1.x, p1.x, p1.y * p1.y)));
			});
			for (int o = 16; o; o >>= 1) r2m = fmaxf (r2m, __shfl_xor_sync (0xffffffffu, r2m, o));
			float* red = xch + kXchFloats + 4;
			if (lane == 0) red[warp] = r2m;
			__syncthreads ();
			if (tid == 0) {
				float m = red[0];
				for (int i = 1; i < kConvThreads / 32; ++i) m = fmaxf (m, red[i]);
				const unsigned old = atomicMax (p.r2max + row, __float_as_uint (m));
				red[kConvThreads / 32] = fmaxf (m, __uint_as_float (old));
			}
			__syncthreads ();
			thr2 = fmaxf (thr2, p.boot_beta * red[kConvThreads / 32]);
		}
		// interior segment whose valid region starts on a block of four strides:
		// no bounds logic, the direct branch comes from the TMEM stash
		const bool interior = cx.i_hi == kM && cx.i_skip == p.Lh && cx.i_zero == p.Lh && stash_usable (dl);
		if (interior) {
			const int dk = dl >> 9;
#pragma unroll
			for (int kb = 8; kb < 32; kb += 4) { // Lh >= 4096
				if (512 * kb < p.Lh) continue;
				float2 zd[4];
				tmem_ld4 (tb + 2 * (kb - dk), zd);
				float pv[4];
				bool  k0[4], k1[4], any = false;
#pragma unroll
				for (int kk = 0; kk < 4; ++kk) {
					const int k = kb + kk;
					pv[kk]      = __shfl_up_sync (0xffffffffu, w[k].y, 1);
					if (lane == 0) pv[kk] = xch[xbase + k];
					rawmax = fmaxf (rawmax, fmaxf (fabsf (zd[kk].x), fabsf (zd[kk].y)));
					k0[kk] = fmaf (zd[kk].x, zd[kk].x, pv[kk] * pv[kk]) >= thr2;
					k1[kk] = fmaf (zd[kk].y, zd[kk].y, w[k].x * w[k].x) >= thr2;
					any    = any || k0[kk] || k1[kk];
				}
				if (__any_sync (0xffffffffu, any)) { // one vote per eight samples; survivors are a fraction of a percent
					float2 q0[4], q1[4];
#pragma unroll
					for (int kk = 0; kk < 4; ++kk) {
						q0[kk] = make_float2 (zd[kk].x, pv[kk]);
						q1[kk] = make_float2 (zd[kk].y, w[kb + kk].x);
					}
					append_points4 (dst, k0, q0, k1, q1, lt, lane);
				}
			}
		} else {
			walk_pairs_checked (w, xch, tb, p, tid, lane, cx, ld, [&] (float2 p0, float2 p1, bool in, bool ok, float2 zd) {
				if (ok) rawmax = fmaxf (rawmax, fmaxf (fabsf (zd.x), fabsf (zd.y)));
				const bool k0 = in && fmaf (p0.x, p0.x, p0.y * p0.y) >= thr2;
				const bool k1 = in && fmaf (p1.x, p1.x, p1.y * p1.y) >= thr2;
				if (__any_sync (0xffffffffu, k0 || k1)) append_points (dst, k0, p0, k1, p1, lt, lane);
			});
		}
		cx.rawmax = rawmax;
	} else {
		float2*      outc = p.out + (cx.obase + (long long)cx.c * p.out_stride);
		const float2 cs   = (EPI == EPI_RENDER) ? p.cs[cx.c] : (EPI == EPI_SECT_RENDER) ? p.sect_cs[cx.row] : make_float2 (0.f, 1.f);
		const int    rlen = (EPI == EPI_RENDER && p.ramp_len) ? p.ramp_len[cx.c] : 0;
#pragma unroll
		for (int kb = 0; kb < 32; kb += 4) {
			if (512 * (kb + 4) <= p.Lh) continue; // whole block in the overlap region (uniform)
			float2 zd[4];
			bool   ok[4];
#pragma unroll
			for (int kk = 0; kk < 4; ++kk) {
				const int i = tid + 512 * (kb + kk);
				ok[kk]      = i >= p.Lh && i < cx.i_hi;
				zd[kk]      = make_float2 (0.f, 0.f);
			}
			if (epi_render (EPI)) load_direct (zd, ok, tid, kb, dl, tb, ld);
#pragma unroll
			for (int kk = 0; kk < 4; ++kk) {
				const int k  = kb + kk;
				const int i  = tid + 512 * k;
				float     pv = __shfl_up_sync (0xffffffffu, w[k].y, 1);
				if (lane == 0) pv = xch[xbase + k];
				if (ok[kk]) {
					float2          y  = make_float2 (pv, w[k].x);
					const long long t0 = 2 * (cx.mbase + i);
					if (EPI == EPI_HILBERT) cx.rawmax = fmaxf (cx.rawmax, fmaxf (fabsf (pv), fabsf (w[k].x))); // bootstrap gate of the true-peak sweep
					if (epi_render (EPI)) {
						float2 cs0 = cs, cs1 = cs;
						if (EPI == EPI_SECT_RENDER && cx.t_sect > 0 && t0 - cx.t_sect < p.hist_frames) { // ramp (rare: sincosf per sample)
							cs0 = sect_ramp_cs (p, cx.row, t0 - cx.t_sect);
							if (t0 + 1 - cx.t_sect < p.hist_frames) cs1 = sect_ramp_cs (p, cx.row, t0 + 1 - cx.t_sect);
						}
						if (t0 < rlen) {
							const float2* r = p.ramp + (long long)cx.c * p.ramp_stride + t0;
							cs0             = r[0];
							if (t0 + 1 < rlen) cs1 = r[1];
						}
						// mul, mul, add like the reference (cli:223, src:700,715)
						y.x = __fadd_rn (__fmul_rn (cs0.x, zd[kk].x), __fmul_rn (cs0.y, pv));
						y.y = __fadd_rn (__fmul_rn (cs1.x, zd[kk].y), __fmul_rn (cs1.y, w[k].x));
					}
					if (epi_render (EPI) && p.out_inter) {
						// straight into the interleaved frames (plain stores: the CTAs of the
						// other channels fill the rest of each sector side by side, L2 merges them)
						float* o = p.out_inter + t0 * p.C + cx.c;
						if (t0 < p.out_frames) o[0] = y.x;
						if (t0 + 1 < p.out_frames) o[p.C] = y.y;
					} else {
						__stcs (outc + i, y);
					}
				}
			}
		}
	}
}

// The thread index, re-assembled from two small tables in shared memory
// (volatile) at the start of every pass.  Neither nvcc nor ptxas can see through
// it, so everything a pass derives from the thread index (addresses, twiddle
// and filter loads) is recomputed inside the pass instead of being hoisted out
// of the persistent loop and kept alive - i.e. spilled to local memory - across
// the other passes, each of which needs the whole register file.
__device__ __forceinline__ int opaque_tid (const float* xch, int tid)
{
	const volatile int* tb = reinterpret_cast<const volatile int*> (xch + kTidOff);
	return tb[tid & 31] + tb[32 + (tid >> 5)];
}

// One segment: five passes, four shared-memory round trips, epilogue from registers.
template <int EPI, int NP, class Loader>
__device__ __forceinline__ void run_segment (float2* sm, float* xch, uint32_t tb, const ConvParams& p, int tid, int lane, EpiCtx& cx, const Loader ld, int reuse_rows = 0)
{
	if (EPI != EPI_HILBERT && stash_usable (p.dl)) {
		p1_forward (sm, p.tw1, opaque_tid (xch, tid), ld, TmemStash { tb }, TmemReuse { tb, reuse_rows, p.V >> 9 });
		tmem_wait_st ();
	} else {
		p1_forward (sm, p.tw1, opaque_tid (xch, tid), ld);
	}
	__syncthreads ();
	// the three middle passes of a block pair stay inside one warp (see p2_block())
	p2_pass<-1> (sm, opaque_tid (xch, tid));
	__syncwarp ();
	if (NP == 2) {
		const int t = opaque_tid (xch, tid);
		mid_pass<MID_CONV2> (sm, GTmem { tb }, p.tw2, t, p.scratch + (size_t)blockIdx.x * (kM / 2) + t, reinterpret_cast<const float4*> (p.G),
		                     reinterpret_cast<const float4*> (p.G1));
	} else {
		mid_pass (sm, GTmem { tb }, p.tw2, opaque_tid (xch, tid));
	}
	__syncwarp ();
	p2_pass<+1> (sm, opaque_tid (xch, tid));
	__syncthreads ();
	float2 w[32];
	p1_inverse (sm, p.tw1, opaque_tid (xch, tid), w);
	if (lane == 31) {
		float* x = xch + (tid >> 5) * 32;
#pragma unroll
		for (int k = 0; k < 32; ++k) x[k] = w[k].y;
	}
	__syncthreads (); // xch visible; every warp is done reading sm, the next segment may overwrite it
	epilogue<EPI> (w, xch, tb, p, tid, lane, cx, ld);
}

// Two partitions: forward transform of the segment before the first one of a run,
// left in the CTA's scratch (see mid_pass()).
template <class Loader>
__device__ __noinline__ void spectrum_only (float2* sm, const float* xch, const float2* tw1, const float2* tw2, float4* scr, int tid, const Loader ld)
{
	p1_forward (sm, tw1, opaque_tid (xch, tid), ld);
	__syncthreads ();
	p2_pass<-1> (sm, opaque_tid (xch, tid));
	__syncwarp ();
	const int t = opaque_tid (xch, tid);
	mid_pass<MID_SPECTRUM> (sm, GTable { nullptr, 0, 0 }, tw2, t, scr + t);
	__syncthreads (); // every warp is done reading sm
}

// ---------------------------------------------------------------------------
// K1: FFT convolution with fused epilogue.  Persistent: one CTA per SM walks
// (segment, channel) pairs, channel fastest, so that the CTAs working on the
// channels of one stretch of interleaved input run at the same time and share
// it through L2.  NP = number of tap partitions (2 only for FIR length 32768).
// ---------------------------------------------------------------------------
__device__ __forceinline__ void flush_rawmax (unsigned* dst, float r, int lane)
{
	for (int o = 16; o; o >>= 1) r = fmaxf (r, __shfl_xor_sync (0xffffffffu, r, o));
	if (lane == 0) atomicMax (dst, __float_as_uint (r));
}

// Bootstrap wave of a sections sweep: segment si of the launch samples section k = si / sect_boot; the
// sect_boot samples of a section are spread over it, each at a pseudo-random offset inside its share.
__device__ __forceinline__ long long sect_boot_seg (const ConvParams& p, int si)
{
	const long long k    = si / p.sect_boot, j = si % p.sect_boot;
	const long long nall = (p.m_end + p.V - 1) / p.V;
	const long long n    = k == p.n_sect - 1 ? nall - k * p.sect_segs : p.sect_segs; // the last section takes the remainder
	const long long w    = max (1LL, n / p.sect_boot);
	return k * p.sect_segs + min (n - 1, j * n / p.sect_boot + (long long)(((unsigned)si * 2654435761u >> 8) % (unsigned)w));
}

template <int EPI, int SRC, int NP>
__global__ void __launch_bounds__ (kConvThreads, 1) fftconv_kernel (const ConvParams p)
{
	extern __shared__ __align__ (16) float2 sm[];
	float*    xch  = reinterpret_cast<float*> (sm + kM);
	const int tid  = threadIdx.x;
	if (tid < 32) reinterpret_cast<int*> (xch + kTidOff)[tid] = tid;                  // see opaque_tid(); made visible by the
	else if (tid < 48) reinterpret_cast<int*> (xch + kTidOff)[tid] = 32 * (tid - 32); // barrier in tmem_alloc_all()
	const uint32_t tmem = tmem_alloc_all (reinterpret_cast<uint32_t*> (xch + kXchFloats), tid);
	const uint32_t tb   = tmem_thread_base (tmem, tid);
	const int lane = tid & 31;
	EpiCtx cx;
	cx.rawmax = 0.f;
	if (EPI == EPI_POINTS) {
		// filter radius of this launch: thr2 = (min_a peaks[c][a])^2 (1 - 1e-5), see
		// threshold_kernel; parked in shared memory for the epilogues
		const int cc  = p.chan0 + (int)blockIdx.x % p.nchan;
		float*    red = xch + kXchFloats + 4;
		float     t2  = 0.f;
		if (p.thr_mode < 0) {
			t2 = p.thr2[cc];
		} else if (p.thr_mode == 2) {
			t2 = __int_as_float (0x7f800000);
		} else if (p.thr_mode == 1) {
			float m = __int_as_float (0x7f800000);
			for (int a = tid; a < p.A; a += kConvThreads) m = fminf (m, __uint_as_float (p.peaks[(long long)cc * p.peaks_stride + a]));
			for (int o = 16; o; o >>= 1) m = fminf (m, __shfl_xor_sync (0xffffffffu, m, o));
			if (lane == 0) red[tid >> 5] = m;
			__syncthreads ();
			m = red[0];
			for (int i = 1; i < kConvThreads / 32; ++i) m = fminf (m, red[i]);
			t2 = (m * m) * 0.99999f;
		}
		if (tid == 0) {
			red[kRedThr] = t2;
			if (p.count_reset) {
				for (int i = 0; i < p.nchan; ++i) p.count_reset[p.chan0 + i] = 0; // every CTA writes the same zeros
			}
		}
		// visible to every thread after the barriers of the first segment
	}
	{
		// this thread's share of the filter spectrum -> TMEM (rows tid and tid + 512 of MID)
		const float4* G4 = reinterpret_cast<const float4*> (p.G);
#pragma unroll
		for (int h = 0; h < 2; ++h) {
#pragma unroll
			for (int c = 0; c < 8; c += 2) {
				const float4 a = __ldg (G4 + c * 1024 + tid + 512 * h), b = __ldg (G4 + (c + 1) * 1024 + tid + 512 * h);
				tmem_st4 (tb + kTmemGCol + 32 * h + 4 * c, make_float2 (a.x, a.y), make_float2 (a.z, a.w), make_float2 (b.x, b.y), make_float2 (b.z, b.w));
			}
		}
		tmem_wait_st ();
	}

	// CTA b owns channel b % nchan and, among the CTAs of that channel, a
	// contiguous run of the launch's segments: consecutive segments share Lh
	// points, which stay in the TMEM stash (TmemReuse), and the CTAs of the
	// channels of one stretch of interleaved input run side by side and share it
	// through L2.
	const int ci = (int)blockIdx.x % p.nchan, jb = (int)blockIdx.x / p.nchan;
	const int nb = ((int)gridDim.x - ci + p.nchan - 1) / p.nchan; // CTAs of this channel
	const int run = ((int)p.nseg + nb - 1) / nb;
	const int s_begin = jb * run, s_end = min ((int)p.nseg, s_begin + run);
	const int c = p.chan0 + ci;
	bool prev_inside = false;
	cx.row = -1;
	for (int si = s_begin; si < s_end; ++si) {

		long long seg = p.seg0 + si * p.seg_stride + (p.seg_jitter ? (long long)(((unsigned)si * 2654435761u >> 8) % (unsigned)p.seg_stride) : 0);
		if (EPI == EPI_SECT_POINTS && p.sect_boot) seg = sect_boot_seg (p, si);
		if (epi_sect (EPI)) {
			const long long k   = min (seg / p.sect_segs, (long long)p.n_sect - 1);
			const int       row = (int)k * p.nchan + ci;
			if (EPI == EPI_SECT_POINTS && row != cx.row && cx.row >= 0) {
				// a run crossing a section boundary: the raw peak so far belongs to the previous row
				flush_rawmax (p.rawpeak + cx.row, cx.rawmax, lane);
				cx.rawmax = 0.f;
			}
			cx.row    = row;
			cx.t_sect = k * p.sect_segs * 2 * p.V;
		}
		const long long n0  = seg * p.V - p.Lh; // complex stream index of local index 0
		if (NP == 2 && (si == s_begin || p.seg_stride != 1)) {
			// the scratch does not hold the spectrum of segment seg - 1 yet
			if (SRC == SRC_PLANE) {
				spectrum_only (sm, xch, p.tw1, p.tw2, p.scratch + (size_t)blockIdx.x * (kM / 2), tid, PlaneLoader { p.plane + (long long)c * p.plane_stride + p.padf + n0 - p.V });
			} else {
				spectrum_only (sm, xch, p.tw1, p.tw2, p.scratch + (size_t)blockIdx.x * (kM / 2), tid, EdgeLoader { p.inter, p.hist, p.n_frames, 2 * (n0 - p.V), p.C, c, p.hist_frames });
			}
		}
		// (No L2 prefetch of the next segment by default: a cp.async.bulk.prefetch.L2 of the stretch one
		// segment ahead made the long launches read 1.26x their bytes from HBM - the lines were
		// fetched, evicted and fetched again - and was 1 % slower than plain loads; r02 traffic probe.
		// p.prefetch = d > 0 prefetches the new part of segment si + d instead, for experiments.)
		if (p.prefetch > 0 && SRC == SRC_INTER && p.seg_stride == 1 && si + p.prefetch < s_end && lane == 0 && ci == 0) {
			const long long nn0    = n0 + (long long)p.prefetch * p.V + p.Lh;
			const long long nbytes = (nn0 >= 0 && 2 * (nn0 + p.V) <= p.n_frames) ? (long long)p.V * 2 * p.C * (long long)sizeof (float) : 0;
			if (nbytes > 0) {
				const unsigned piece = (unsigned)(nbytes >> 4) & ~15u;
				const char*    a     = reinterpret_cast<const char*> (reinterpret_cast<uintptr_t> (p.inter + 2 * nn0 * p.C) & ~(uintptr_t)15) + (size_t)(tid >> 5) * piece;
				asm volatile ("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(a), "r"(piece) : "memory");
			}
		}

		// local bounds of the output regions (clamped to the segment)
		cx.c     = c;
		cx.mbase = n0;
		cx.obase = p.out_compact ? (long long)si * p.V - p.Lh + 8 : n0;
		{
			const long long hi = p.m_end - n0, sk = p.m_skip - n0, ze = p.m_zero - n0;
			cx.i_hi   = hi >= kM ? kM : (hi <= p.Lh ? p.Lh : (int)hi);
			cx.i_skip = sk <= p.Lh ? p.Lh : (sk >= kM ? kM : (int)sk);
			cx.i_zero = ze <= p.Lh ? p.Lh : (ze >= kM ? kM : (int)ze);
		}

		if (SRC == SRC_PLANE) {
			run_segment<EPI, NP> (sm, xch, tb, p, tid, lane, cx, PlaneLoader { p.plane + (long long)c * p.plane_stride + p.padf + n0 });
		} else {
			const bool inside = n0 >= 0 && 2 * (n0 + kM) <= p.n_frames;
			const int  reuse  = (inside && prev_inside && p.seg_stride == 1) ? (p.Lh >> 9) : 0;
			prev_inside       = inside;
			if (!inside) {
				run_segment<EPI, NP> (sm, xch, tb, p, tid, lane, cx, EdgeLoader { p.inter, p.hist, p.n_frames, 2 * n0, p.C, c, p.hist_frames });
			} else if (p.C == 2 && (reinterpret_cast<uintptr_t> (p.inter) & 15) == 0) {
				run_segment<EPI, NP> (sm, xch, tb, p, tid, lane, cx, Inter2Loader { reinterpret_cast<const float4*> (p.inter) + n0, c }, reuse);
			} else if (p.C == 1 && (reinterpret_cast<uintptr_t> (p.inter) & 7) == 0) {
				run_segment<EPI, NP> (sm, xch, tb, p, tid, lane, cx, Inter1Loader { reinterpret_cast<const float2*> (p.inter) + n0 }, reuse);
			} else {
				run_segment<EPI, NP> (sm, xch, tb, p, tid, lane, cx, InterNLoader { p.inter + 2 * n0 * p.C + c, p.C }, reuse);
			}
		}
	}

	if (EPI == EPI_POINTS && s_begin < s_end) {
		float r = cx.rawmax;
		for (int o = 16; o; o >>= 1) r = fmaxf (r, __shfl_xor_sync (0xffffffffu, r, o));
		if (lane == 0) atomicMax (p.rawpeak + c, __float_as_uint (r));
	}
	if (EPI == EPI_SECT_POINTS && s_begin < s_end) flush_rawmax (p.rawpeak + cx.row, cx.rawmax, lane);
	if (EPI == EPI_HILBERT && p.r2max && s_begin < s_end) {
		// largest H^2 of the launch: truepeak_kernel gates its bootstrap wave on it
		float r = cx.rawmax;
		for (int o = 16; o; o >>= 1) r = fmaxf (r, __shfl_xor_sync (0xffffffffu, r, o));
		if (lane == 0) atomicMax (p.r2max + c, __float_as_uint (r * r));
	}
	tmem_free_all (tmem, tid);
}

// ---------------------------------------------------------------------------
// K0: interleaved frames -> planes.  One thread per complex element n of a
// chunk: frames 2n and 2n+1 of every channel.  Frames >= n_frames read as 0.
// ---------------------------------------------------------------------------
__global__ void deinterleave_kernel (const float* __restrict__ in, long long frame0, long long n_frames_total,
                                     long long n_first, long long n_count, int C,
                                     float2* __restrict__ plane, long long plane_stride, int padf)
{
	const long long n = n_first + (long long)blockIdx.x * blockDim.x + threadIdx.x;
	if (n >= n_first + n_count) return;
	const long long f0 = 2 * n, f1 = 2 * n + 1;
	// `in` points at frame `frame0` of the stream
	const float* a = in + (f0 - frame0) * C;
	if (C == 2 && f1 < n_frames_total) {
		const float4 v = *reinterpret_cast<const float4*> (a);
		plane[padf + n]                = make_float2 (v.x, v.z);
		plane[plane_stride + padf + n] = make_float2 (v.y, v.w);
		return;
	}
	for (int c = 0; c < C; ++c) {
		const float x0 = f0 < n_frames_total ? a[c] : 0.f;
		const float x1 = f1 < n_frames_total ? a[C + c] : 0.f;
		plane[(long long)c * plane_stride + padf + n] = make_float2 (x0, x1);
	}
}

// Integer PCM -> float on the device, the conversion libsndfile applies in
// sf_readf_float (what the reference reads with, cli/phase-rotate.cc:573):
// 16-bit sample / 2^15; 32-bit container (24-bit samples left-justified, as
// sf_readf_int delivers them) / 2^31.  Both are exact scalings of an exactly
// (16/24-bit) or correctly rounded (32-bit) converted integer, i.e. bit-identical
// to the host conversion.  The file then crosses PCIe at 2 (or 4) bytes per
// sample and is widened at HBM speed.  n = samples (frames * channels).
template <class I>
__global__ void __launch_bounds__ (256) pcm_to_float_kernel (const I* __restrict__ in, float* __restrict__ out, long long n)
{
	constexpr float   scale = sizeof (I) == 2 ? 1.f / 32768.f : 1.f / 2147483648.f;
	const long long   i4    = ((long long)blockIdx.x * blockDim.x + threadIdx.x) * 4;
	if (i4 + 3 < n && (reinterpret_cast<uintptr_t> (in + i4) & (4 * sizeof (I) - 1)) == 0 && (reinterpret_cast<uintptr_t> (out + i4) & 15) == 0) {
		I v[4];
		if (sizeof (I) == 2) {
			*reinterpret_cast<uint2*> (v) = __ldcs (reinterpret_cast<const uint2*> (in + i4));
		} else {
			*reinterpret_cast<uint4*> (v) = __ldcs (reinterpret_cast<const uint4*> (in + i4));
		}
		*reinterpret_cast<float4*> (out + i4) = make_float4 ((float)v[0] * scale, (float)v[1] * scale, (float)v[2] * scale, (float)v[3] * scale);
		return;
	}
	for (long long i = i4; i < n && i < i4 + 4; ++i) out[i] = (float)in[i] * scale;
}

// packed 24-bit little-endian PCM (3 bytes per sample, as in the file's data chunk) -> float:
// the sample left-justified in 32 bits times 2^-31 = sample / 2^23, what sf_readf_float returns.
// `in` is 4-byte aligned; a thread converts 4 samples = 12 bytes = three aligned words.
__global__ void __launch_bounds__ (256) pcm24_to_float_kernel (const uint8_t* __restrict__ in, float* __restrict__ out, long long n)
{
	constexpr float scale = 1.f / 2147483648.f;
	const long long i4    = ((long long)blockIdx.x * blockDim.x + threadIdx.x) * 4;
	if (i4 + 3 < n && (reinterpret_cast<uintptr_t> (out + i4) & 15) == 0) {
		const uint32_t* w = reinterpret_cast<const uint32_t*> (in + 3 * i4);
		const uint32_t  a = __ldcs (w), b = __ldcs (w + 1), c = __ldcs (w + 2);
		const int       s0 = (int)(a << 8);
		const int       s1 = (int)(((a >> 24) << 8) | (b << 16));
		const int       s2 = (int)(((b >> 16) << 8) | (c << 24));
		const int       s3 = (int)(c & 0xffffff00u);
		*reinterpret_cast<float4*> (out + i4) = make_float4 ((float)s0 * scale, (float)s1 * scale, (float)s2 * scale, (float)s3 * scale);
		return;
	}
	for (long long i = i4; i < n && i < i4 + 4; ++i) {
		const uint8_t* q = in + 3 * i;
		const int      v = (int)(((uint32_t)q[0] << 8) | ((uint32_t)q[1] << 16) | ((uint32_t)q[2] << 24));
		out[i]           = (float)v * scale;
	}
}

// Combine the tables of a device group on its first device: dst[i] = max (dst[i], src_k[i]) over the
// other devices' tables, read in place through NVLink peer memory (or from a gathered copy when peer
// access is not available).  The values are bit patterns of non-negative floats: unsigned order = float order.
struct PeerTabs {
	const unsigned* p[15];
	int             n;
};
__global__ void __launch_bounds__ (256) peer_max_kernel (unsigned* __restrict__ dst, const PeerTabs src, long long n)
{
	const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
	if (i >= n) return;
	unsigned v = dst[i];
	for (int k = 0; k < src.n; ++k) v = max (v, src.p[k][i]);
	dst[i] = v;
}

// planes of float2 (two consecutive samples) -> interleaved frames
__global__ void interleave_kernel (const float2* __restrict__ plane, long long plane_stride, int C,
                                   long long n_count, float* __restrict__ out, long long n_frames_out)
{
	const long long n = (long long)blockIdx.x * blockDim.x + threadIdx.x;
	if (n >= n_count) return;
	const long long f0 = 2 * n, f1 = f0 + 1;
	if (C == 2 && f1 < n_frames_out) {
		const float2 l = plane[n], r = plane[plane_stride + n];
		*reinterpret_cast<float4*> (out + f0 * 2) = make_float4 (l.x, r.x, l.y, r.y);
		return;
	}
	for (int c = 0; c < C; ++c) {
		const float2 v = plane[(long long)c * plane_stride + n];
		if (f0 < n_frames_out) out[f0 * C + c] = v.x;
		if (f1 < n_frames_out) out[f1 * C + c] = v.y;
	}
}

// ---------------------------------------------------------------------------
// K3: sweep.  Thread t of a CTA owns angles a = agrp + t + blockDim * r, r < R:
// (ca, sa) and the running max stay in registers; the survivor points are
// broadcast from shared memory.  Replaces calc_rotated_peak (cli:98-121) and
// dsp_compute_peak (cli/dsp_peak_calc.h): max_i |ca x_d[i] + sa h[i]|.
// grid = (point tiles, angle groups, channels).
// ---------------------------------------------------------------------------
constexpr int kSweepTile = 256; // points per tile

template <int R>
__global__ void __launch_bounds__ (256) sweep_kernel (const float2* __restrict__ list, long long list_stride,
                                                       const unsigned* __restrict__ count, unsigned cap, int skip_overflowed, int chan0,
                                                       const float2* __restrict__ cs, int A,
                                                       unsigned* __restrict__ peaks, int peaks_stride,
                                                       unsigned long long* __restrict__ n_eval)
{
	__shared__ __align__ (16) float2 tile[kSweepTile];
	const int       c    = chan0 + blockIdx.z;
	if (skip_overflowed && count[c] > cap) return;  // the pass is flagged and will be repeated in dense mode: do not brute-force a full list first
	const unsigned  n    = min (count[c], cap); // (bootstrap wave: the counter may run past its small capacity, the excess was dropped)
	// Short lists (the usual case: a few hundred survivors per launch) are cut into small tiles so that
	// many CTAs share them: one CTA walking a 256-point tile alone is a 10 us serial chain.
	const unsigned tile_pts = min ((unsigned)kSweepTile, max (32u, ((n + gridDim.x - 1) / gridDim.x + 1) & ~1u));
	if (blockIdx.x * tile_pts >= n) return; // nothing for this CTA
	const float2*   pts  = list + (long long)c * list_stride;
	const int       a0   = blockIdx.y * (blockDim.x * R) + threadIdx.x;

	float ca[R], sa[R], pk[R];
#pragma unroll
	for (int r = 0; r < R; ++r) {
		const int a = a0 + r * blockDim.x;
		const float2 v = a < A ? cs[a] : make_float2 (0.f, 0.f);
		ca[r] = v.x;
		sa[r] = v.y;
		pk[r] = 0.f;
	}

	for (unsigned base = blockIdx.x * tile_pts; base < n; base += gridDim.x * tile_pts) {
		const unsigned cnt = min (tile_pts, n - base);
		__syncthreads ();
		for (unsigned i = threadIdx.x; i < tile_pts; i += blockDim.x) {
			tile[i] = i < cnt ? pts[base + i] : make_float2 (0.f, 0.f);
		}
		__syncthreads ();
		const float4* t4 = reinterpret_cast<const float4*> (tile);
		const unsigned n2 = (cnt + 1) >> 1;
#pragma unroll 4
		for (unsigned i = 0; i < n2; ++i) {
			const float4 q = t4[i]; // two points: (x0, h0, x1, h1), broadcast
#pragma unroll
			for (int r = 0; r < R; ++r) {
				const float y0 = fmaf (ca[r], q.x, sa[r] * q.y);
				const float y1 = fmaf (ca[r], q.z, sa[r] * q.w);
				pk[r]          = fmaxf (pk[r], fmaxf (fabsf (y0), fabsf (y1)));
			}
		}
		if (n_eval && blockIdx.y == 0 && threadIdx.x == 0) atomicAdd (n_eval, (unsigned long long)cnt);
	}

#pragma unroll
	for (int r = 0; r < R; ++r) {
		const int a = a0 + r * blockDim.x;
		if (a < A && pk[r] > 0.f) atomicMax (peaks + (long long)c * peaks_stride + a, __float_as_uint (pk[r]));
	}
}

// thr2[c] = (min_a peaks[c][a])^2 * (1 - 1e-5): a point whose radius is below
// that cannot raise any angle's running maximum (|ca x + sa h| <= sqrt(x^2+h^2)
// up to a few ulp), so dropping it leaves every peak bit-identical.
// mode 0: keep every point (thr2 = 0); 1: prune; 2: drop every point (no angle wanted)
__global__ void threshold_kernel (const unsigned* __restrict__ peaks, int peaks_stride, int A, int chan0,
                                  float* __restrict__ thr2, unsigned* __restrict__ count, int reset_count, int mode)
{
	const int c = chan0 + blockIdx.x;
	if (mode != 1) {
		if (threadIdx.x == 0) {
			thr2[c] = mode == 0 ? 0.f : __int_as_float (0x7f800000);
			if (reset_count) count[c] = 0;
		}
		return;
	}
	float     m = __int_as_float (0x7f800000);
	for (int a = threadIdx.x; a < A; a += blockDim.x) {
		m = fminf (m, __uint_as_float (peaks[(long long)c * peaks_stride + a]));
	}
	__shared__ float red[32];
	for (int o = 16; o; o >>= 1) m = fminf (m, __shfl_xor_sync (0xffffffffu, m, o));
	if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = m;
	__syncthreads ();
	if (threadIdx.x < 32) {
		m = threadIdx.x < (blockDim.x >> 5) ? red[threadIdx.x] : __int_as_float (0x7f800000);
		for (int o = 16; o; o >>= 1) m = fminf (m, __shfl_xor_sync (0xffffffffu, m, o));
		if (threadIdx.x == 0) {
			thr2[c] = (m * m) * 0.99999f;
			if (reset_count) count[c] = 0;
		}
	}
}

// ---------------------------------------------------------------------------
// Dense mode (long survivor lists: few-tone or constant-envelope material, where
// most samples lie on or near the hull of the point set {(x_d, H)} and the
// global radius filter keeps them).  A point p = r (cos phi, sin phi) gives
//     y_j = ca_j x + sa_j h = r cos (alpha_j - phi),   alpha_j = -j * step (grid index j)
// so it can raise the running peak of grid angle j only if
//     r |cos (alpha_j - phi)| >= T_j   (T_j <= peak[j], any earlier value of it).
// The grid is cut into kSectors sectors of equal width; sector_thr_kernel takes
// T_s = min over the swept angles of sector s of the running peaks, and
// sweep_window_kernel (one thread per point) visits only the sectors within
// reach of the global threshold, tests the sector bound
//     r cos (dist (phi, sector s)) >= T_s
// and evaluates only the angles of a passing sector with |alpha_j - phi| <=
// acos (T_s / r) - with the SAME fp32 expression as sweep_kernel, so the table is
// bit-identical to brute force.  Interior points (most of a two-tone signal's
// survivors) cost a few sector tests, points of a constant-envelope signal a
// handful of angles instead of all of them.  Points that still need more than
// kWideEvals evaluations go to a second list for sweep_kernel (angles in lanes).
// All margins err towards evaluating: 4e-6 relative on T / r (the fp32
// evaluation of y and r is good to ~3e-7), 6e-5 rad + one grid step on every
// angular bound (the fast atan2 is good to 2e-5 rad, the LUT's own rounding to 2e-6 rad).
// ---------------------------------------------------------------------------
constexpr int kSectors   = 60;  // divides 180 * S for every S
constexpr int kWideEvals = 768;

// sec[c][s] = min over slots k with grid index in sector s of peaks[c][k]  (+inf: nothing swept there)
__global__ void __launch_bounds__ (64) sector_thr_kernel (const unsigned* __restrict__ peaks, int peaks_stride, const int* __restrict__ slot_of, int MS, int chan0,
                                                          float* __restrict__ sec)
{
	const int c = chan0 + blockIdx.y, s = blockIdx.x, G = MS / kSectors;
	float     m = __int_as_float (0x7f800000);
	for (int j = s * G + threadIdx.x; j < (s + 1) * G; j += blockDim.x) {
		const int k = slot_of[j];
		if (k >= 0) m = fminf (m, __uint_as_float (peaks[(long long)c * peaks_stride + k]));
	}
	__shared__ float red[2];
	for (int o = 16; o; o >>= 1) m = fminf (m, __shfl_xor_sync (0xffffffffu, m, o));
	if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = m;
	__syncthreads ();
	if (threadIdx.x == 0) sec[c * kSectors + s] = fminf (red[0], red[1]);
}

struct WinParams {
	const float2*   list;
	long long       list_stride;
	const unsigned* count;
	unsigned        cap;
	int             chan0;
	const float2*   cs;       // [A] (ca, sa) per slot
	const int*      slot_of;  // [MS] grid index -> slot, -1 = not swept
	int             MS;
	const float*    sec;      // [C][kSectors]
	unsigned*       peaks;
	int             peaks_stride;
	float2*         wide;     // [C][wide_stride] points left to sweep_kernel
	long long       wide_stride;
	unsigned*       wide_count; // [C]
	unsigned long long* n_eval; // statistics: point-angle evaluations / A
	unsigned long long* n_listed; // statistics: points on the lists of this sweep
	int             slot_base; // >= 0: the swept set is a run of consecutive grid indices, slot = grid index - slot_base (no table)
	int             smem_tables; // 1: (ca, sa) and a snapshot of the running peaks sit in shared memory (A * 12 bytes)
	int             walk_steps;  // sweep_walk_kernel: evaluations beyond the first window before a point goes to the wide list
	int             A;
};

// acos (q) <= sqrt (2 u) (1 + 0.12 u), u = 1 - q in [0, 1]  (series sqrt(2u)(1 + u/12 + 3u^2/160 + ...); 1.584 >= pi/2 at u = 1)
__device__ __forceinline__ float acos_upper (float q)
{
	const float u = fmaxf (1.f - q, 1e-30f);
	return (2.f * u) * rsqrtf (2.f * u) * fmaf (0.12f, u, 1.00001f); // sqrt via MUFU.RSQ (2 ulp), rounded up by the factor
}

// atan2 to 2e-5 rad (polynomial of Abramowitz & Stegun 4.4.49 on [0, 1], 1e-5; approximate division): the window
// bounds carry 4e-5 rad of slack for it
__device__ __forceinline__ float atan2_fast (float y, float x)
{
	const float ax = fabsf (x), ay = fabsf (y);
	const float mx = fmaxf (ax, ay), mn = fminf (ax, ay);
	const float z  = __fdividef (mn, fmaxf (mx, 1e-30f));
	const float z2 = z * z;
	float       p  = fmaf (-0.0117212f, z2, 0.05265332f);
	p              = fmaf (p, z2, -0.11643287f);
	p              = fmaf (p, z2, 0.19354346f);
	p              = fmaf (p, z2, -0.33262347f);
	p              = fmaf (p, z2, 0.99997726f);
	float a        = z * p;
	if (ay > ax) a = 1.57079632679f - a;
	if (x < 0.f) a = 3.14159265359f - a;
	return y < 0.f ? -a : a;
}

__global__ void __launch_bounds__ (256) sweep_window_kernel (const WinParams p)
{
	const int      c = p.chan0 + blockIdx.y;
	const unsigned n = min (p.count[c], p.cap);
	const float    step = 3.14159265358979f / (float)p.MS, inv_step = (float)p.MS / 3.14159265358979f;
	const int      G = p.MS / kSectors;
	const float    inv_G = 1.f / (float)G;
	const float*   sec = p.sec + c * kSectors;
	unsigned*      pk  = p.peaks + (long long)c * p.peaks_stride;
	// The per-angle tables are hit at a different entry by every lane (neighbouring list entries are
	// neighbouring samples, whose directions differ by the signal's phase advance): from L1 that is one
	// 128-byte line per lane and load; from shared memory it is a bank conflict of degree ~3.
	extern __shared__ __align__ (16) unsigned char win_sm[];
	float2*   s_cs = reinterpret_cast<float2*> (win_sm);
	unsigned* s_pk = reinterpret_cast<unsigned*> (s_cs + p.A);
	if (p.smem_tables) {
		for (int k = threadIdx.x; k < p.A; k += blockDim.x) {
			s_cs[k] = p.cs[k];
			s_pk[k] = pk[k];
		}
	}
	// global threshold = the smallest sector threshold (every running peak is at least that)
	__shared__ float tg_s;
	if (threadIdx.x < 32) {
		float m = fminf (sec[threadIdx.x], threadIdx.x + 32 < kSectors ? sec[threadIdx.x + 32] : __int_as_float (0x7f800000));
		for (int o = 16; o; o >>= 1) m = fminf (m, __shfl_xor_sync (0xffffffffu, m, o));
		if (threadIdx.x == 0) tg_s = m;
	}
	__syncthreads ();
	const float tg = tg_s * (1.f - 4e-6f);
	if (!(tg < __int_as_float (0x7f800000))) return; // no angle swept
	if (blockIdx.x == 0 && threadIdx.x == 0 && p.n_listed) atomicAdd (p.n_listed, (unsigned long long)n);
	unsigned long long evals = 0;
	for (unsigned i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
		const float2 q  = p.list[(long long)c * p.list_stride + i];
		const float  r2 = fmaf (q.x, q.x, q.y * q.y);
		if (!(r2 > 0.f)) continue;
		const float ri = rsqrtf (r2) * (1.f - 1e-6f); // a lower bound of 1 / r: thresholds over r come out low, windows wide
		// fractional grid index of the direction of the point: alpha = phi (mod pi)  <=>  j = -phi / step (mod MS)
		const float jc = -atan2_fast (q.y, q.x) * inv_step;
		// reach of the global threshold in grid steps
		const float rg = (acos_upper (tg * ri) + 6e-5f) * inv_step + 1.f;
		bool        wide = !(2.f * rg + 2.f < (float)p.MS); // (nearly) the whole grid
		int         done = 0;
		if (!wide) {
			const int s_lo = __float2int_rd ((jc - rg) * inv_G), s_hi = __float2int_rd ((jc + rg) * inv_G);
			int       sm   = s_lo % kSectors;
			if (sm < 0) sm += kSectors;
			for (int su = s_lo; su <= s_hi && !wide; ++su, sm = sm + 1 == kSectors ? 0 : sm + 1) {
				const float qs = sec[sm] * (1.f - 4e-6f) * ri; // T_s / r
				if (!(qs <= 1.f)) continue;                    // nothing swept in the sector, or its threshold is above r
				// angular half width within which the point can still reach the sector's threshold
				const float rs = (acos_upper (qs) + 6e-5f) * inv_step + 1.f;
				const int   j0 = max (su * G, __float2int_ru (jc - rs)), j1 = min (su * G + G - 1, __float2int_rd (jc + rs));
				if (j1 < j0) continue;                         // the sector lies outside that window
				done += j1 - j0 + 1;
				if (done > kWideEvals) {
					wide = true; // what has been evaluated stays valid (a running maximum); the point is redone whole
					break;
				}
				int jj = j0 % p.MS;
				if (jj < 0) jj += p.MS;
				for (int j = j0; j <= j1; ++j) {
					int k = jj - p.slot_base;
					if (p.slot_base < 0) k = p.slot_of[jj];
					else if (k >= p.A) k = -1;
					if (++jj == p.MS) jj = 0;
					if (k < 0) continue;
					const float2   w  = p.smem_tables ? s_cs[k] : p.cs[k];
					const unsigned yb = __float_as_uint (fabsf (fmaf (w.x, q.x, w.y * q.y))); // sweep_kernel's expression
					if (p.smem_tables) {
						if (yb > s_pk[k]) { // the snapshot only lags behind the table: a stale value costs an atomic, never a maximum
							atomicMax (s_pk + k, yb);
							atomicMax (pk + k, yb);
						}
					} else if (yb > pk[k]) {
						atomicMax (pk + k, yb);
					}
				}
			}
			evals += (unsigned long long)done;
		}
		if (wide) {
			const unsigned at = atomicAdd (p.wide_count + c, 1u);
			p.wide[(long long)c * p.wide_stride + at] = q; // the wide list has the capacity of the list itself
		}
	}
	if (p.n_eval) {
		for (int o = 16; o; o >>= 1) evals += __shfl_xor_sync (0xffffffffu, evals, o);
		if ((threadIdx.x & 31) == 0 && evals) atomicAdd (p.n_eval, (evals + (unsigned long long)p.A - 1) / (unsigned long long)p.A);
	}
}

// The same sweep when the swept set is the whole grid, or all of it but an angle or two (the CLI's sweep leaves
// out angle 0; slot = grid index - slot_base), without a single acos: |y_j| = r |cos (alpha_j - phi)| falls
// monotonically with the distance of j from the direction of the point, out to 90 degrees on either side.  Every
// thread of a warp evaluates the 2 WH + 1 grid angles around the one nearest to phi (sweep_kernel's fp32
// expression, compared with the running peak); if both ends of that window lie below the global threshold (the
// smallest sector threshold) no angle farther out can be raised and the point is done.  Otherwise the thread
// walks outwards from the window, in both directions; the walk
//   * stops for good when |y_j| falls below the global threshold;
//   * jumps to the near edge of the next sector when |y_j| falls below the threshold of the sector j lies in:
//     no angle farther out IN THAT SECTOR can be raised;
//   * gives the point to the wide list (sweep_kernel, every angle) after a dozen steps.
// A point of a constant-envelope signal costs one atan2 and the first window; points well above the smallest
// threshold (interior points of a few-tone signal while the table is young) are cheaper at every angle, angles in
// lanes, than step by step in one lane.  Margins: 4e-6 relative on every threshold and 2e-6 (|x| + |h|) >= 2e-6 r
// absolute on every comparison (the fp32 evaluation of y is good to ~3e-7 r, so a value farther out can exceed
// the one that stopped the walk by at most 6e-7 r); window and walk start beyond the nearest grid angle on either
// side, and the nearest grid angle is found to 2e-5 rad (the atan2 polynomial) + one rounding - far less than
// half a step for every grid whose table fits shared memory (the condition for this kernel; finer grids keep
// sweep_window_kernel).
// MUFU.RCP / one instruction
__device__ __forceinline__ float rcp_approx (float x)
{
	float r;
	asm ("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
	return r;
}

template <int WH> // half width of the window every point starts with, in grid angles
__global__ void __launch_bounds__ (256) sweep_walk_kernel (const WinParams p)
{
	// A step of the walk costs a warp ~45 issue slots for one lane's benefit - 40 ps of the whole GPU - while
	// sweep_kernel does a point at every angle in 200 ps: beyond half a dozen steps either side the wide list is
	// the cheaper place, and a bounded walk also means no thread holds its CTA for 768 serial evaluations (which
	// made launches with a few far-out points take 150-240 us for 10 us of work; ncu launch list, two tones).
	const int      kWalkEvals = 2 * WH + 1 + p.walk_steps; // a dozen by default
	const int      c = p.chan0 + blockIdx.y;
	const unsigned n = min (p.count[c], p.cap);
	const int      MS = p.MS, G = MS / kSectors;
	const float    inv_step = (float)MS / 3.14159265358979f, inv_G = 1.f / (float)G;
	unsigned*      pk = p.peaks + (long long)c * p.peaks_stride;
	// (ca, sa, snapshot of the running peak, -) per angle in shared memory, one LDS.128 per evaluation.  The
	// snapshot only lags behind the table, so a stale value costs an atomic, never a maximum.
	extern __shared__ __align__ (16) unsigned char win_sm[];
	float4* s_tab = reinterpret_cast<float4*> (win_sm);
	for (int k = threadIdx.x; k < p.A; k += blockDim.x) {
		const float2 w = p.cs[k];
		s_tab[k]       = make_float4 (w.x, w.y, __uint_as_float (pk[k]), 0.f);
	}
	__shared__ float s_sec[kSectors + 4];
	if (threadIdx.x < kSectors) s_sec[threadIdx.x] = p.sec[c * kSectors + threadIdx.x] * (1.f - 4e-6f);
	__syncthreads ();
	if (threadIdx.x < 32) {
		float m = fminf (s_sec[threadIdx.x], threadIdx.x + 32 < kSectors ? s_sec[threadIdx.x + 32] : __int_as_float (0x7f800000));
		for (int o = 16; o; o >>= 1) m = fminf (m, __shfl_xor_sync (0xffffffffu, m, o));
		if (threadIdx.x == 0) s_sec[kSectors] = m;
	}
	__syncthreads ();
	const float tg = s_sec[kSectors];
	if (!(tg < __int_as_float (0x7f800000))) return;
	if (blockIdx.x == 0 && threadIdx.x == 0 && p.n_listed) atomicAdd (p.n_listed, (unsigned long long)n);
	auto eval = [&] (const float2& q, int k) -> float {
		const float4 w = s_tab[k];
		const float  y = fabsf (fmaf (w.x, q.x, w.y * q.y)); // sweep_kernel's expression
		if (y > w.z) {                                        // (peaks are never negative and never NaN: the same order as their bit patterns)
			atomicMax (reinterpret_cast<unsigned*> (&s_tab[k].z), __float_as_uint (y));
			atomicMax (pk + k, __float_as_uint (y));
		}
		return y;
	};
	unsigned       evals  = 0;
	const unsigned stride = gridDim.x * blockDim.x;
	// whole warps per trip, reconverged at the top: a thread that leaves the rare walk below late must not
	// drag its warp through the next point's window once more on its own
	const float2*  lst    = p.list + (long long)c * p.list_stride;
	const unsigned first  = blockIdx.x * blockDim.x + (threadIdx.x & ~31u);
	float2         qn     = first + (threadIdx.x & 31u) < n ? lst[first + (threadIdx.x & 31u)] : make_float2 (0.f, 0.f);
	for (unsigned base = first; base < n; base += stride) {
		__syncwarp ();
		const unsigned i = base + (threadIdx.x & 31u);
		const float2   q = qn;
		qn               = i + stride < n ? lst[i + stride] : make_float2 (0.f, 0.f); // the next trip's point: its latency hides behind this one
		const float    ax = fabsf (q.x), ay = fabsf (q.y);
		const float    tgs = fmaf (-2e-6f, ax + ay, tg); // global threshold less the slack of a comparison (2e-6 r at least)
		// nearest grid angle: alpha = phi (mod pi)  <=>  j = -phi / step (mod MS); atan2 as in atan2_fast()
		const float mx = fmaxf (ax, ay), mn = fminf (ax, ay);
		const float z  = mn * rcp_approx (fmaxf (mx, 1e-30f));
		const float z2 = z * z;
		float       pl = fmaf (-0.0117212f, z2, 0.05265332f);
		pl             = fmaf (pl, z2, -0.11643287f);
		pl             = fmaf (pl, z2, 0.19354346f);
		pl             = fmaf (pl, z2, -0.33262347f);
		pl             = fmaf (pl, z2, 0.99997726f);
		float a        = z * pl;
		if (ay > ax) a = 1.57079632679f - a;
		if (q.x < 0.f) a = 3.14159265359f - a;
		if (q.y >= 0.f) a = -a; // -phi
		int j0 = __float2int_rn (a * inv_step);
		if (j0 < 0) j0 += MS;
		if (j0 >= MS) j0 -= MS;
		// A window of 2 WH + 1 angles around j0 first, the same for every thread of the warp (no branch but the
		// rare atomic): for a point of a constant-envelope signal - r a few 1e-6 above the threshold - both ends
		// of it already lie below the global threshold and that is all there is.  (Near the ends of the table the
		// window is pushed inside - any evaluation is a valid one - and both walks start at distance 1.)
		const int k0 = j0 - p.slot_base;
		const int kc = min (max (k0, WH), p.A - 1 - WH);
		float     yl = 0.f, yr = 0.f;
#pragma unroll
		for (int t = -WH; t <= WH; ++t) {
			const float y = eval (q, kc + t);
			if (t == -WH) yl = y;
			if (t == WH) yr = y;
		}
		int  done = 2 * WH + 1;
		bool wide = false;
		if (mx > 0.f && (kc != k0 || yl >= tgs || yr >= tgs)) { // rare
#pragma unroll 1
			for (int dir = 0; dir < 2; ++dir) {
				const int room = dir ? (MS - 1) / 2 : MS / 2; // angles ahead out to 90 degrees
				int       t    = kc != k0 ? 1 : ((dir ? yl : yr) >= tgs ? WH + 1 : MS);
				while (t <= room) {
					int j = dir ? j0 - t : j0 + t; // distance t from j0
					if (j < 0) j += MS;
					if (j >= MS) j -= MS;
					const int k = j - p.slot_base;
					const int s = __float2int_rd (((float)j + 0.5f) * inv_G); // sector of j
					float     y = __int_as_float (0x7f800000); // not swept (the CLI leaves out angle 0): nothing to evaluate, nothing learnt
					if (k >= 0 && k < p.A) y = eval (q, k);
					++done;
					if (!(y >= tgs)) break;
					// within reach of the sector's threshold: next angle; else on to the near edge of the next sector
					t += (y >= s_sec[s] - (tg - tgs)) ? 1 : (dir ? j - s * G + 1 : (s + 1) * G - j);
					if (done > kWalkEvals) break;
				}
				if (done > kWalkEvals) {
					wide = true; // what has been evaluated stays valid (a running maximum); the point is redone whole
					break;
				}
			}
		}
		evals += i < n ? (unsigned)done : 0u;
		if (wide) {
			const unsigned at = atomicAdd (p.wide_count + c, 1u);
			p.wide[(long long)c * p.wide_stride + at] = q; // the wide list has the capacity of the list itself
		}
	}
	if (p.n_eval) {
		unsigned long long e = evals;
		for (int o = 16; o; o >>= 1) e += __shfl_xor_sync (0xffffffffu, e, o);
		if ((threadIdx.x & 31) == 0 && e) atomicAdd (p.n_eval, (e + (unsigned long long)p.A - 1) / (unsigned long long)p.A);
	}
}

// (ca, sa) of the plugin's small-call path: output i of channel c uses
// pre[c][i] for i < rlen[c] (angle ramp, src:673-709) and cs[c] after that.
struct FirCoef {
	float2 cs[2];
	int    rlen[2];
};
// ---------------------------------------------------------------------------
// Small-call plugin path, streaming form: the input history of every channel
// lives in a device ring (kRing floats, index = stream position & (kRing - 1)),
// a run() call only ships its n new samples (mapped pinned memory, read once)
// and gets n outputs back (written straight to mapped pinned memory).  One
// launch per run().  CTA = 32 outputs x 4 tap quarters; output u in
// [u0, u0 + n), u0 = t0 - parsiz:
//   Y[u] = ca_u * x[u - firlat] + sa_u * sum_j g[j] x[u - 1 - 2j]      (src:629-717)
// Every CTA also appends its 32 new samples to the ring; they are read by later
// calls only (positions >= t0 are never read from the ring in this launch, and
// n + firlen + parsiz <= kRing keeps them clear of the history being read).
// ---------------------------------------------------------------------------
constexpr int kRing      = 32768;
constexpr int kStreamOut = 32;

__global__ void __launch_bounds__ (128) fir_stream_kernel (float* __restrict__ ring, const float* __restrict__ xin, int xin_stride, int n,
                                                            long long t0, int parsiz, const float* __restrict__ g, int nodd, int firlat,
                                                            const float2* __restrict__ pre, int pre_stride, FirCoef fc, float* __restrict__ yout,
                                                            float* __restrict__ lev)
{
	extern __shared__ float sh[]; // g[nodd] | window[2 nodd + 32] | partial[4][32]
	const int c  = blockIdx.y;
	const int o0 = blockIdx.x * kStreamOut;
	const int nb = min (kStreamOut, n - o0);
	float*    sg = sh;
	float*    sx = sh + nodd;
	float*    sp = sx + 2 * nodd + kStreamOut;
	float*       rc = ring + (long long)c * kRing;
	const float* xc = xin + (long long)c * xin_stride;
	for (int j = threadIdx.x; j < nodd; j += blockDim.x) sg[j] = __ldg (g + j);
	// window: stream positions w0 .. w0 + 2 nodd + nb - 1, w0 = u_lo - 2 nodd, u_lo = t0 - parsiz + o0
	const long long w0 = t0 - parsiz + o0 - 2 * nodd;
	for (int i = threadIdx.x; i < 2 * nodd + nb; i += blockDim.x) {
		const long long t = w0 + i;
		sx[i]             = t < 0 ? 0.f : (t < t0 ? rc[t & (kRing - 1)] : xc[t - t0]);
	}
	if ((int)threadIdx.x < nb) rc[(t0 + o0 + threadIdx.x) & (kRing - 1)] = xc[o0 + threadIdx.x];
	__syncthreads ();
	const int o = threadIdx.x & 31, q = threadIdx.x >> 5;
	{
		// x[u - 1 - 2j] = sx[2 nodd + o - 1 - 2j]
		const int    nq = nodd >> 2; // nodd is a multiple of 4 (1536 / 2048 / 4096)
		const float* xp = sx + 2 * nodd + o - 1 - 2 * q * nq;
		const float* gp = sg + q * nq;
		float        a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
#pragma unroll 4
		for (int j = 0; j < nq; j += 4) {
			a0 = fmaf (gp[j], xp[-2 * j], a0);
			a1 = fmaf (gp[j + 1], xp[-2 * j - 2], a1);
			a2 = fmaf (gp[j + 2], xp[-2 * j - 4], a2);
			a3 = fmaf (gp[j + 3], xp[-2 * j - 6], a3);
		}
		sp[q * 32 + o] = (a0 + a1) + (a2 + a3);
	}
	__syncthreads ();
	if (q == 0) { // warp 0
		float ax = 0.f, ay = 0.f;
		if (o < nb) {
			const float  hv = (sp[o] + sp[32 + o]) + (sp[64 + o] + sp[96 + o]);
			const float  xd = sx[2 * nodd + o - firlat];
			const float2 cs = (o0 + o) < fc.rlen[c] ? pre[(long long)c * pre_stride + o0 + o] : fc.cs[c];
			const float  y  = __fadd_rn (__fmul_rn (cs.x, xd), __fmul_rn (cs.y, hv));
			yout[(long long)c * n + o0 + o] = y;
			ax = fabsf (xd);
			ay = fabsf (y);
		}
		if (lev) {
			// level meters of the plugin (src:573-609, 727-739): max |delayed input| and
			// max |output| of this CTA's 32 samples; the host takes the max over the
			// CTAs of the call.  fmaxf drops NaNs like the host meter did.
			for (int s = 16; s; s >>= 1) {
				ax = fmaxf (ax, __shfl_xor_sync (0xffffffffu, ax, s));
				ay = fmaxf (ay, __shfl_xor_sync (0xffffffffu, ay, s));
			}
			if (o == 0) {
				float* l = lev + 2 * ((long long)c * gridDim.x + blockIdx.x);
				l[0]     = ax;
				l[1]     = ay;
			}
		}
	}
}

// max |a[i]| and max |b[i]|, i < n, per channel (blockIdx.y) -> lev[c][0], lev[c][1]
// (float bits, atomicMax; values >= 0).  Bulk plugin calls: a = delayed input, b = output.
__global__ void __launch_bounds__ (256) absmax2_kernel (const float* __restrict__ a, long long a_stride, const float* __restrict__ b, long long b_stride,
                                                         long long n, unsigned* __restrict__ lev)
{
	const int    c  = blockIdx.y;
	const float* pa = a + (long long)c * a_stride;
	const float* pb = b + (long long)c * b_stride;
	float        ma = 0.f, mb = 0.f;
	for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
		ma = fmaxf (ma, fabsf (pa[i]));
		mb = fmaxf (mb, fabsf (pb[i]));
	}
	for (int s = 16; s; s >>= 1) {
		ma = fmaxf (ma, __shfl_xor_sync (0xffffffffu, ma, s));
		mb = fmaxf (mb, __shfl_xor_sync (0xffffffffu, mb, s));
	}
	if ((threadIdx.x & 31) == 0) {
		atomicMax (lev + 2 * c, __float_as_uint (ma));
		atomicMax (lev + 2 * c + 1, __float_as_uint (mb));
	}
}

// ---------------------------------------------------------------------------
// Oversampled true-peak front end of the sweep (cfg.oversample = 2 or 4; not a
// reference feature, definition in include/phaserot_cuda.h).  The FFT kernel
// leaves the Hilbert branch H of one launch in `H` (EPI_HILBERT, compact
// layout: 16 floats of carry from the previous launch, then 2 V samples per
// segment); this kernel forms the pairs p[t] = (x_d[t], H[t]), interpolates
// both components with the BS.1770-4 Annex 2 polyphase FIR
//     p^[t, ph] = sum_{k < 12} c[ph][k] p[t - k]
// and sends p[t] and every p^[t, ph] through the same exact radius filter and
// survivor list as the digital sweep, so sweep_kernel and threshold_kernel are
// shared.  grid = (tiles of 1024 samples, channels), 256 threads x 4 samples.
// ---------------------------------------------------------------------------
constexpr int kTpTile  = 1024;
constexpr int kTpHalo  = 12; // 11 past samples are needed; 12 keeps the 16-byte alignment of a thread's window
constexpr int kTpCarry = 16; // floats kept in front of H from the previous launch

// ITU-R BS.1770-4 Annex 2, table "filter coefficients" (all multiples of 2^-13: exact in fp32)
PRK_HD constexpr float tp_coef (int ph, int k)
{
	constexpr float c0[12] = { 0.0017089843750f, 0.0109863281250f, -0.0196533203125f, 0.0332031250000f, -0.0594482421875f, 0.1373291015625f,
		                       0.9721679687500f, -0.1022949218750f, 0.0476074218750f, -0.0266113281250f, 0.0148925781250f, -0.0083007812500f };
	constexpr float c1[12] = { -0.0291748046875f, 0.0292968750000f, -0.0517578125000f, 0.0891113281250f, -0.1665039062500f, 0.4650878906250f,
		                       0.7797851562500f, -0.2003173828125f, 0.1015625000000f, -0.0582275390625f, 0.0330810546875f, -0.0189208984375f };
	return ph == 0 ? c0[k] : ph == 1 ? c1[k] : ph == 2 ? c1[11 - k] : c0[11 - k];
}

struct TpParams {
	const float* inter;       // interleaved frames, frame 0 = stream position 0
	const float* hist;        // frames [-hist_frames, 0) or nullptr (silence)
	long long    n_frames;
	int          C, hist_frames;
	const float* H;           // [channel][h_stride]: kTpCarry floats, then launch-compact samples
	long long    h_stride;
	int          chan0;
	long long    seg0, seg_stride;
	int          seg_jitter;  // same pseudo-random segment offsets as ConvParams::seg_jitter
	float        boot_beta;   // > 0: bootstrap wave, additionally gate on boot_beta * r2max[c]
	const unsigned* r2max;    // [channel] float bits of the largest H^2 of the launch (written by the FFT kernel)
	int          V2;          // samples per segment (2 V)
	int          D;           // delay of the direct branch in samples (L / 2)
	long long    t_skip;      // t <  t_skip : not examined            (first-block rule, cli:418-419)
	long long    t_zero;      // t <  t_zero : direct branch forced to 0
	long long    t_end;       // samples exist for t < t_end
	int          os;          // 2 or 4
	float2*      list;
	long long    list_stride;
	unsigned*    count;
	unsigned     list_cap;    // as in ConvParams
	unsigned*    overflow;
	const float* thr2;
	unsigned*    rawpeak;
};

__device__ __forceinline__ float tp_input_at (const TpParams& p, int c, long long f)
{
	if (f >= 0) return f < p.n_frames ? __ldg (p.inter + f * p.C + c) : 0.f;
	return (p.hist && f >= -(long long)p.hist_frames) ? __ldg (p.hist + (p.hist_frames + f) * p.C + c) : 0.f;
}

template <int PH>
__device__ __forceinline__ float tp_interp (const float (&s)[16], int n)
{
	float a = 0.f;
#pragma unroll
	for (int k = 0; k < 12; ++k) a = fmaf (tp_coef (PH, k), s[12 + n - k], a);
	return a;
}

// both components of a pair (x_d, H) at once: one FFMA2 per tap, the coefficient
// broadcast to the two halves as an immediate
template <int PH>
__device__ __forceinline__ float2 tp_interp2 (const float2 (&s)[16], int n)
{
	float2 a = make_float2 (0.f, 0.f);
#pragma unroll
	for (int k = 0; k < 12; ++k) a = __ffma2_rn (make_float2 (tp_coef (PH, k), tp_coef (PH, k)), s[12 + n - k], a);
	return a;
}

// survivors of one sample (bit q of `keep` = point q) -> list, one atomic per warp
__device__ __forceinline__ void tp_append (float2* lst, unsigned* cnt, unsigned cap, unsigned* ovf, unsigned keep, const float2 (&pt)[5], int lane)
{
	if (__any_sync (0xffffffffu, keep != 0)) {
		// exclusive prefix sum of the per-lane survivor counts
		const int nk  = __popc (keep);
		int       inc = nk;
#pragma unroll
		for (int o = 1; o < 32; o <<= 1) {
			const int v = __shfl_up_sync (0xffffffffu, inc, o);
			if (lane >= o) inc += v;
		}
		unsigned base = 0;
		if (lane == 31) {
			base = atomicAdd (cnt, (unsigned)inc);
			if (base + (unsigned)inc > cap) *ovf = 0x3f800000u;
		}
		base          = __shfl_sync (0xffffffffu, base, 31);
		unsigned pos  = base + (unsigned)(inc - nk);
#pragma unroll
		for (int q = 0; q < 5; ++q) {
			if (keep & (1u << q)) {
				if (pos < cap) lst[pos] = pt[q];
				++pos;
			}
		}
	}
}

__global__ void __launch_bounds__ (256, 4) truepeak_kernel (const TpParams p)
{
	__shared__ __align__ (16) float sh[kTpTile + kTpHalo], sx[kTpTile + kTpHalo], sq[kTpTile + kTpHalo];
	const int       c    = p.chan0 + blockIdx.y;
	const int       tps  = p.V2 / kTpTile; // tiles per segment
	const int       si   = blockIdx.x / tps, tile = blockIdx.x - si * tps;
	const long long u0   = (long long)si * p.V2 + (long long)tile * kTpTile;                        // launch-compact index
	const long long seg  = p.seg0 + si * p.seg_stride + (p.seg_jitter ? (long long)(((unsigned)si * 2654435761u >> 8) % (unsigned)p.seg_stride) : 0);
	const long long t0   = seg * (long long)p.V2 + (long long)tile * kTpTile; // stream time
	if (t0 >= p.t_end) return;
	// the 11 samples of H before the tile: inside the segment, in the previous
	// segment of a contiguous launch, or in the carry of the previous launch; a
	// sparse (bootstrap) launch has no predecessor, its first 11 samples per
	// segment are left to the contiguous passes
	const bool   head_ok = p.seg_stride == 1 || tile > 0;
	const float* Hc      = p.H + (long long)c * p.h_stride + kTpCarry + u0 - kTpHalo;
	const bool   q1      = t0 - kTpHalo < p.t_zero; // tile touches the forced-zero region of the direct branch
	// Interior tile (nearly all of them): every sample exists, is examined, has its
	// direct branch inside the input and no forced zeros.  The pairs (x_d, H) go
	// to shared memory as float2 and every interpolation is a packed FFMA2 chain.
	if (!q1 && head_ok && t0 - kTpHalo >= p.t_skip && t0 + kTpTile <= p.t_end && t0 - kTpHalo - p.D >= 0 && t0 + kTpTile - p.D <= p.n_frames) {
		__shared__ __align__ (16) float2 sp[kTpTile + kTpHalo];
		const float* xc = p.inter + (t0 - kTpHalo - p.D) * p.C + c;
#pragma unroll
		for (int j = 0; j < 4; ++j) {
			const int i = threadIdx.x + 256 * j;
			sp[i]       = make_float2 (__ldg (xc + (long long)i * p.C), __ldg (Hc + i));
		}
		if (threadIdx.x < kTpHalo) {
			const int i = kTpTile + threadIdx.x;
			sp[i]       = make_float2 (__ldg (xc + (long long)i * p.C), __ldg (Hc + i));
		}
		__syncthreads ();
		float2 w[16];
		{
			const float4* s4 = reinterpret_cast<const float4*> (sp) + 2 * threadIdx.x;
#pragma unroll
			for (int v = 0; v < 8; ++v) {
				const float4 a = s4[v];
				w[2 * v]     = make_float2 (a.x, a.y);
				w[2 * v + 1] = make_float2 (a.z, a.w);
			}
		}
		float          thr2f = p.thr2[c];
		if (p.boot_beta > 0.f) thr2f = fmaxf (thr2f, p.boot_beta * __uint_as_float (p.r2max[c]));
		float2*        lstf  = p.list + (long long)c * p.list_stride;
		unsigned*      cntf  = p.count + c;
		const int      lanef = threadIdx.x & 31;
		float          rmax  = 0.f;
#pragma unroll
		for (int n = 0; n < 4; ++n) {
			float2 pt[5];
			pt[0] = w[12 + n];
			pt[1] = tp_interp2<0> (w, n);
			pt[3] = tp_interp2<2> (w, n);
			if (p.os == 4) {
				pt[2] = tp_interp2<1> (w, n);
				pt[4] = tp_interp2<3> (w, n);
			} else {
				pt[2] = pt[4] = make_float2 (0.f, 0.f);
			}
			unsigned keep = 0;
#pragma unroll
			for (int q = 0; q < 5; ++q) {
				rmax = fmaxf (rmax, fabsf (pt[q].x));
				if (fmaf (pt[q].x, pt[q].x, pt[q].y * pt[q].y) >= thr2f && (p.os == 4 || !(q == 2 || q == 4))) keep |= 1u << q;
			}
			tp_append (lstf, cntf, p.list_cap, p.overflow, keep, pt, lanef);
		}
		for (int o = 16; o; o >>= 1) rmax = fmaxf (rmax, __shfl_xor_sync (0xffffffffu, rmax, o));
		if (lanef == 0 && rmax > 0.f) atomicMax (p.rawpeak + c, __float_as_uint (rmax));
		return;
	}
	for (int i = threadIdx.x; i < kTpTile + kTpHalo; i += blockDim.x) {
		const long long t = t0 - kTpHalo + i;
		const float     x = tp_input_at (p, c, t - p.D);
		sh[i]             = (head_ok || i >= kTpHalo) ? Hc[i] : 0.f;
		sx[i]             = x;
		sq[i]             = t < p.t_zero ? 0.f : x;
	}
	__syncthreads ();

	const int j = threadIdx.x;
	float     hs[16], xs[16], qs[16];
	{
		const float4* h4 = reinterpret_cast<const float4*> (sh) + j;
		const float4* x4 = reinterpret_cast<const float4*> (sx) + j;
		const float4* q4 = reinterpret_cast<const float4*> (sq) + j;
#pragma unroll
		for (int v = 0; v < 4; ++v) {
			const float4 a = h4[v], b = x4[v];
			hs[4 * v] = a.x, hs[4 * v + 1] = a.y, hs[4 * v + 2] = a.z, hs[4 * v + 3] = a.w;
			xs[4 * v] = b.x, xs[4 * v + 1] = b.y, xs[4 * v + 2] = b.z, xs[4 * v + 3] = b.w;
			if (q1) {
				const float4 q = q4[v];
				qs[4 * v] = q.x, qs[4 * v + 1] = q.y, qs[4 * v + 2] = q.z, qs[4 * v + 3] = q.w;
			} else {
				qs[4 * v] = b.x, qs[4 * v + 1] = b.y, qs[4 * v + 2] = b.z, qs[4 * v + 3] = b.w;
			}
		}
	}
	float          thr2 = p.thr2[c];
	if (p.boot_beta > 0.f) thr2 = fmaxf (thr2, p.boot_beta * __uint_as_float (p.r2max[c])); // any subset is valid in the bootstrap
	float2*        lst  = p.list + (long long)c * p.list_stride;
	unsigned*      cnt  = p.count + c;
	const int      lane = threadIdx.x & 31;
	float          rawmax = 0.f;
#pragma unroll
	for (int n = 0; n < 4; ++n) {
		const long long t  = t0 + 4 * j + n;
		const bool      in = t < p.t_end;
		const bool      ex = in && t >= p.t_skip && (head_ok || 4 * j + n >= kTpHalo - 1);
		float2 pt[5];
		float  xr[5];
		pt[0] = make_float2 (qs[12 + n], hs[12 + n]);
		xr[0] = xs[12 + n];
		pt[1] = make_float2 (tp_interp<0> (qs, n), tp_interp<0> (hs, n));
		pt[3] = make_float2 (tp_interp<2> (qs, n), tp_interp<2> (hs, n));
		xr[1] = q1 ? tp_interp<0> (xs, n) : pt[1].x;
		xr[3] = q1 ? tp_interp<2> (xs, n) : pt[3].x;
		if (p.os == 4) {
			pt[2] = make_float2 (tp_interp<1> (qs, n), tp_interp<1> (hs, n));
			pt[4] = make_float2 (tp_interp<3> (qs, n), tp_interp<3> (hs, n));
			xr[2] = q1 ? tp_interp<1> (xs, n) : pt[2].x;
			xr[4] = q1 ? tp_interp<3> (xs, n) : pt[4].x;
		} else {
			pt[2] = pt[4] = make_float2 (0.f, 0.f);
			xr[2] = xr[4] = 0.f;
		}
		unsigned keep = 0;
#pragma unroll
		for (int q = 0; q < 5; ++q) {
			if (in) rawmax = fmaxf (rawmax, fabsf (xr[q]));
			if (ex && fmaf (pt[q].x, pt[q].x, pt[q].y * pt[q].y) >= thr2 && (p.os == 4 || !(q == 2 || q == 4))) keep |= 1u << q;
		}
		tp_append (lst, cnt, p.list_cap, p.overflow, keep, pt, lane);
	}
	for (int o = 16; o; o >>= 1) rawmax = fmaxf (rawmax, __shfl_xor_sync (0xffffffffu, rawmax, o));
	if (lane == 0 && rawmax > 0.f) atomicMax (p.rawpeak + c, __float_as_uint (rawmax));
}

// last kTpCarry floats of a contiguous launch's H -> front of the buffer, for the next launch
__global__ void tp_carry_kernel (float* H, long long h_stride, int chan0, long long n_samples)
{
	float* Hc = H + (long long)(chan0 + blockIdx.x) * h_stride;
	if (threadIdx.x < kTpCarry) Hc[threadIdx.x] = Hc[kTpCarry + n_samples - kTpCarry + threadIdx.x];
}

} // namespace prk
