// Integrated loudness (ITU-R BS.1770-4) of the rotated output, device part
// (phaserot_loudness*, definition in include/phaserot_cuda.h).
//
// Rotation and K-weighting are linear, so for the --fixed-write render
//     out[t] = ca x[t] + sa H'[t],  t in [0, F)
// the K-weighted mean square of every 100 ms sub-block is a quadratic form in
// (ca, sa) whose three coefficients are sums over K(x) and the Hilbert branch
// of K(x).  One pass gives the sums; the gate then evaluates any angle set.
//
//   kweight_kernel        K(x): the two biquads, fp64 state, chunk-parallel
//                         (pass 1: zero-state end state of every chunk;
//                          pass 2: re-run from the carried start state)
//   kweight_carry_kernel  start state of every chunk: a warp scan of the
//                         affine chunk maps s -> A^N s + e_k per channel
//   loudness_head_kernel  the K state the trimmed render discards (see below)
//   loudness_stats_kernel Sxx, Sxh, Shh per (sub-block, channel), one FFT
//                         launch of the Hilbert branch at a time
//   loudness_gate_kernel  block energies, absolute and relative gate, fp64
#pragma once

#include <cuda_runtime.h>

namespace prk {

// K-weighting of BS.1770-4: high shelf, then high pass, each a biquad in
// transposed direct form II; a[0] = 1.
struct KwCoef {
	double b[2][3];
	double a[2][3];
};

struct KwState {
	double s[4]; // (s1, s2) of the shelf, (s1, s2) of the high pass
};

__device__ __forceinline__ double kw_step (const KwCoef& k, double (&s)[4], double x)
{
	const double y1 = fma (k.b[0][0], x, s[0]);
	s[0]            = fma (k.b[0][1], x, fma (-k.a[0][1], y1, s[1]));
	s[1]            = fma (k.b[0][2], x, -k.a[0][2] * y1);
	const double y2 = fma (k.b[1][0], y1, s[2]);
	s[2]            = fma (k.b[1][1], y1, fma (-k.a[1][1], y2, s[3]));
	s[3]            = fma (k.b[1][2], y1, -k.a[1][2] * y2);
	return y2;
}

// One thread per (chunk, channel), channel fastest.  Frames [k N, min ((k+1) N, T)) of
// channel c; the input is zero from frame F on.  WRITE = false: run from zero state and
// store the end state in st[k][c].  WRITE = true: run from st[k][c] (the carried start
// state) and write K(x) as float to kx[t][c].
template <bool WRITE>
__global__ void __launch_bounds__ (256) kweight_kernel (const float* __restrict__ x, long long F, long long T, int C, long long N, KwCoef k,
                                                        KwState* __restrict__ st, float* __restrict__ kx)
{
	const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
	const long long n_chunk = (T + N - 1) / N;
	if (i >= n_chunk * C) return;
	const int       c  = (int)(i % C);
	const long long t0 = (i / C) * N, t1 = min (T, t0 + N);
	double          s[4] = { 0., 0., 0., 0. };
	if (WRITE) {
		for (int j = 0; j < 4; ++j) s[j] = st[i].s[j];
	}
	for (long long t = t0; t < t1; ++t) {
		const double in = t < F ? (double)__ldg (x + t * C + c) : 0.;
		const double y  = kw_step (k, s, in);
		if (WRITE) kx[t * C + c] = (float)y;
	}
	if (!WRITE) {
		for (int j = 0; j < 4; ++j) st[i].s[j] = s[j];
	}
}

__device__ __forceinline__ void mat4_acc (const double* __restrict__ M, const double (&v)[4], double (&acc)[4])
{
#pragma unroll
	for (int r = 0; r < 4; ++r) {
#pragma unroll
		for (int q = 0; q < 4; ++q) acc[r] = fma (M[4 * r + q], v[q], acc[r]);
	}
}

// One warp per channel.  st[k][c] holds the zero-state end state e_k of chunk k on entry
// and the start state of chunk k on return: s_0 = 0, s_{k+1} = A^N s_k + e_k.  P[m - 1] =
// A^(m N), m = 1 .. 32, row-major 4 x 4.  32 chunks per step: an inclusive Kogge-Stone
// scan of the e_k inside the warp, then the carry from the previous group.
__global__ void __launch_bounds__ (32) kweight_carry_kernel (KwState* __restrict__ st, long long n_chunk, int C, const double* __restrict__ P)
{
	const int lane = threadIdx.x, c = blockIdx.x;
	double    carry[4] = { 0., 0., 0., 0. };
	for (long long g = 0; g < n_chunk; g += 32) {
		const long long k = g + lane;
		double          v[4];
		for (int j = 0; j < 4; ++j) v[j] = k < n_chunk ? st[k * C + c].s[j] : 0.;
#pragma unroll
		for (int d = 1; d < 32; d <<= 1) {
			double w[4];
#pragma unroll
			for (int j = 0; j < 4; ++j) w[j] = __shfl_up_sync (0xffffffffu, v[j], d);
			if (lane >= d) mat4_acc (P + 16 * (d - 1), w, v);
		}
		// end state of chunk k = A^((lane + 1) N) carry + v
		double e[4] = { v[0], v[1], v[2], v[3] };
		mat4_acc (P + 16 * lane, carry, e);
		double s[4];
#pragma unroll
		for (int j = 0; j < 4; ++j) {
			s[j] = __shfl_up_sync (0xffffffffu, e[j], 1);
			if (lane == 0) s[j] = carry[j];
		}
		if (k < n_chunk) {
			for (int j = 0; j < 4; ++j) st[k * C + c].s[j] = s[j];
		}
#pragma unroll
		for (int j = 0; j < 4; ++j) carry[j] = __shfl_sync (0xffffffffu, e[j], 31);
	}
}

// The trimmed render starts K at t = 0 on H'[t] = H[t + D], so the first D samples of the
// Hilbert branch of x never enter it; the branch the stats read, Hilbert (K(x))[t + D] =
// K(H)[t + D], includes them.  The difference is the zero-input response of K from the
// state K reaches on H[0, D), which decays by ~1e-7 over one 100 ms sub-block at any rate.
// One thread per channel: H0 = Hilbert branch of x (compact staging, H0[c * h_stride +
// kTpCarry + t] = H[t]); zc[c][t] = that response for t in [0, nz).
__global__ void loudness_head_kernel (const float* __restrict__ H0, long long h_stride, int D, KwCoef k, double* __restrict__ zc, int nz)
{
	if (threadIdx.x) return;
	const int    c  = blockIdx.x;
	const float* Hc = H0 + (long long)c * h_stride + kTpCarry;
	double       s[4] = { 0., 0., 0., 0. };
	for (int t = 0; t < D; ++t) kw_step (k, s, (double)Hc[t]);
	for (int t = 0; t < nz; ++t) zc[(long long)c * nz + t] = kw_step (k, s, 0.);
}

// Sums of sub-blocks j0 + blockIdx.x, channel blockIdx.y, over the samples t in [lo, hi)
// whose Hilbert branch H[t + D] is in the staging of the current FFT launch (compact
// layout, H[u] at Hs[c * h_stride + kTpCarry + u - u0]).  Adds to sums[j][c][3]: a
// sub-block cut by a launch boundary takes two launches, in stream order.
__global__ void __launch_bounds__ (256) loudness_stats_kernel (const float* __restrict__ kx, int C, const float* __restrict__ Hs, long long h_stride,
                                                               long long u0, int D, long long step, long long j0, long long lo, long long hi,
                                                               const double* __restrict__ zc, int nz, double* __restrict__ sums)
{
	__shared__ double red[3][256];
	const int       c  = blockIdx.y;
	const long long j  = j0 + blockIdx.x;
	const long long a  = max (lo, j * step), b = min (hi, (j + 1) * step);
	const float*    Hc = Hs + (long long)c * h_stride + kTpCarry;
	double          sxx = 0., sxh = 0., shh = 0.;
	for (long long t = a + threadIdx.x; t < b; t += blockDim.x) {
		const double xk = (double)__ldg (kx + t * C + c);
		double       hk = (double)__ldg (Hc + (t + D - u0));
		if (t < nz) hk -= zc[(long long)c * nz + t];
		sxx = fma (xk, xk, sxx);
		sxh = fma (xk, hk, sxh);
		shh = fma (hk, hk, shh);
	}
	red[0][threadIdx.x] = sxx;
	red[1][threadIdx.x] = sxh;
	red[2][threadIdx.x] = shh;
	__syncthreads ();
	for (int o = 128; o; o >>= 1) {
		if ((int)threadIdx.x < o) {
			for (int q = 0; q < 3; ++q) red[q][threadIdx.x] += red[q][threadIdx.x + o];
		}
		__syncthreads ();
	}
	if (threadIdx.x < 3) sums[(j * C + c) * 3 + threadIdx.x] += red[threadIdx.x][0];
}

// Energy of 400 ms block k (sub-blocks k .. k + 3) at the rotation cs[c] = (ca, sa).
__device__ __forceinline__ double block_energy (const double* __restrict__ sums, int C, const float2* __restrict__ cs, const double* __restrict__ G, long long k,
                                                double inv_len)
{
	double e = 0.;
	for (int c = 0; c < C; ++c) {
		const double ca = cs[c].x, sa = cs[c].y;
		double       q  = 0.;
		for (long long j = k; j < k + 4; ++j) {
			const double* s = sums + (j * C + c) * 3;
			q += ca * ca * s[0] + 2. * ca * sa * s[1] + sa * sa * s[2];
		}
		e = fma (G[c], q * inv_len, e);
	}
	return e;
}

// fixed-order tree sum of (sum, count) over the CTA
__device__ __forceinline__ void gate_reduce (double (&rs)[256], double (&rn)[256], double s, double n)
{
	rs[threadIdx.x] = s;
	rn[threadIdx.x] = n;
	__syncthreads ();
	for (int o = 128; o; o >>= 1) {
		if ((int)threadIdx.x < o) {
			rs[threadIdx.x] += rs[threadIdx.x + o];
			rn[threadIdx.x] += rn[threadIdx.x + o];
		}
		__syncthreads ();
	}
}

// One CTA of 256 threads per angle set: cs[set][c], G[c] channel weights, nb = n_sub - 3 blocks.
__global__ void __launch_bounds__ (256) loudness_gate_kernel (const double* __restrict__ sums, int C, long long nb, long long step, const float2* __restrict__ cs,
                                                              const double* __restrict__ G, double* __restrict__ lufs)
{
	__shared__ double rs[256], rn[256];
	const float2*     csk     = cs + (long long)blockIdx.x * C;
	const double      inv_len = 1.0 / (4.0 * (double)step);
	const double      abs_e   = pow (10.0, (-70.0 + 0.691) / 10.0); // absolute gate, -70 LUFS
	double            s = 0., n = 0.;
	for (long long k = threadIdx.x; k < nb; k += blockDim.x) {
		const double e = block_energy (sums, C, csk, G, k, inv_len);
		if (e > abs_e) s += e, n += 1.;
	}
	gate_reduce (rs, rn, s, n);
	if (rn[0] == 0.) {
		if (threadIdx.x == 0) lufs[blockIdx.x] = -INFINITY;
		return;
	}
	const double rel_e = 0.1 * (rs[0] / rn[0]); // relative gate, -10 LU
	__syncthreads ();
	s = 0., n = 0.;
	for (long long k = threadIdx.x; k < nb; k += blockDim.x) {
		const double e = block_energy (sums, C, csk, G, k, inv_len);
		if (e > abs_e && e > rel_e) s += e, n += 1.;
	}
	gate_reduce (rs, rn, s, n);
	if (threadIdx.x == 0) lufs[blockIdx.x] = rn[0] > 0. ? -0.691 + 10.0 * log10 (rs[0] / rn[0]) : -INFINITY;
}

} // namespace prk
