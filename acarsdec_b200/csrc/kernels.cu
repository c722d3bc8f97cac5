/*
 * CUDA kernels of the acarsdec hot path for sm_100a.
 *
 *  K1  k_channelize<MODE> : u8 IQ / float32 real / CS16 IQ samples -> per-channel NCO mix x
 *                     boxcar(K) -> decimate by K -> |.|  (reference: in_callback rtl.c:334-354;
 *                     rx_callback air.c:291-341; soapy.c:232-254, sdrplay.c:215-236).  FP32-issue bound by the
 *                     reference's rounding sequence: every complex MAC is 4 rounded products
 *                     and 4 rounded sums in tap order, no FMA contraction — reproduced exactly
 *                     (IQ: two rows packed per FFMA2(x, w, -0) / FADD2, see cmac2) so dm is
 *                     bit-identical to the strict-IEEE build of the reference.
 *      k_channelize_dft   : opt-in fast form of the u8 path (ACB_FLAG_FAST_CHANNELIZER): the same bins as a
 *                     shared 4-point DFT across the row quarters + K/4 MACs per channel; HBM-bound
 *                     (bulk copies, packed FFMA2); messages identical, envelope within tolerance.
 *  K2  k_demod<LANES>     : demodMSK + putbit + decodeAcars, 4 or 8 lanes per channel
 *                     (reference: msk.c:67-137, acars.c:246-375), state carried in HBM between
 *                     launches; serial recurrence per channel, parallel across channels/streams.
 *  K3  k_block_fec        : blk_thread's parity/CRC/syndrome repair, one thread per finished frame
 *                     (reference: acars.c:39-215).
 *
 * Numerics contract (SURVEY.md §8a): all order/rounding-sensitive arithmetic uses the
 * explicit round-to-nearest intrinsics, which the compiler never contracts; the TU is also
 * built with -fmad=false.
 */
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>
#include <stdlib.h>

#include <algorithm>

#include "acb_internal.h"
#include "frame_sm.h"
#include "demod_core.h"

namespace acb {

__constant__ float c_h[FLENO];     /* matched filter, built on the host with glibc cosf (msk.c:44-48) */

/* stream-ordered uploads: the caller synchronises `stream` before it launches anything (the context's
 * streams are non-blocking, i.e. not ordered behind the legacy stream a plain cudaMemcpyToSymbol uses) */
int upload_matched_filter(const float *h, cudaStream_t stream);

/* ------------------------------------------------------------------------------------------
 * K1: channelizer
 * ---------------------------------------------------------------------------------------- */

/* (float)u8 - 127.37f  (rtl.c:338-339) for sample `pair` of word wa (row A) and of word wb (row B),
 * row-packed: re = (I_A, I_B), im = (Q_A, Q_B).  The byte is planted in the mantissa of 2^23, the
 * 2^23 removed (exact), then 127.37f subtracted — also exact: the result is a multiple of
 * 2^-17 below 2^7, so the reference's single rounding rounds nothing either. */
__device__ __forceinline__ void cvt_iq(unsigned wa, unsigned wb, int pair, float2 &re, float2 &im)
{
	re = make_float2(__uint_as_float(__byte_perm(wa, 0x4B000000u, pair ? 0x7542 : 0x7540)),
	                 __uint_as_float(__byte_perm(wb, 0x4B000000u, pair ? 0x7542 : 0x7540)));
	im = make_float2(__uint_as_float(__byte_perm(wa, 0x4B000000u, pair ? 0x7543 : 0x7541)),
	                 __uint_as_float(__byte_perm(wb, 0x4B000000u, pair ? 0x7543 : 0x7541)));
	re = __fadd2_rn(__fadd2_rn(re, make_float2(-8388608.0f, -8388608.0f)), make_float2(-127.37f, -127.37f));
	im = __fadd2_rn(__fadd2_rn(im, make_float2(-8388608.0f, -8388608.0f)), make_float2(-127.37f, -127.37f));
}

/* D += (a + jb) * (c + jd) with the reference's rounding: products rounded, (ac - bd) and
 * (ad + bc) rounded, then the accumulate rounded (rtl.c:351) — for two output rows at once,
 * row-packed: a = (a_A, a_B), b = (b_A, b_B), Dre = (Dre_A, Dre_B), Dim = (Dim_A, Dim_B); the
 * table entry (c, d) rides the packed ops' scalar operand.
 * Instruction shape: 4 FFMA2 + 4 FADD2 for the two rows, i.e. 4 packed instructions per complex MAC.
 * Every product is FFMA2(x, w, nz) with nz = -0.0f: rn(x*w + (-0)) = rn(x*w) for every finite
 * x*w, signed zeros included, and an FFMA2 cannot be fused into the FADD2 that consumes it.  nz
 * must be a run-time value (a kernel argument): ptxas turns an FFMA2 with a literal -0 addend
 * back into FMUL2, and contracts mul.rn.f32x2 feeding add.rn.f32x2 into FFMA2 even under
 * -fmad=false, which would skip a product rounding.  tests/test_sass_exact.py checks the SASS. */
__device__ __forceinline__ void cmac2(float2 &dre, float2 &dim, const float2 a, const float2 b, float c, float d, float nz)
{
	const float2 z = make_float2(nz, nz), cc = make_float2(c, c), dd = make_float2(d, d);
	const float2 ac = __ffma2_rn(a, cc, z), bd = __ffma2_rn(b, dd, z);
	const float2 ad = __ffma2_rn(a, dd, z), bc = __ffma2_rn(b, cc, z);
	dre = __fadd2_rn(dre, __fadd2_rn(ac, make_float2(-bd.x, -bd.y)));
	dim = __fadd2_rn(dim, __fadd2_rn(ad, bc));
}

/* cabsf (rtl.c:353): glibc hypotf is (float)sqrt((double)x*x + (double)y*y) for finite input */
__device__ __forceinline__ float envelope(float2 d)
{
	double x = (double)d.x, y = (double)d.y;
	return __double2float_rn(__dsqrt_rn(__dadd_rn(__dmul_rn(x, x), __dmul_rn(y, y))));
}

__device__ __forceinline__ void cp_async16(void *smem, const void *gmem)
{
	unsigned s = (unsigned)__cvta_generic_to_shared(smem);
	asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(s), "l"(gmem) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_group 0;" ::: "memory"); }

/* ------------------------------------------------------------------------------------------
 * K1 pipeline.  One CTA = one 1024-output block x one group of 8 channels; 128 threads, two
 * output rows per thread (rows t and t+128 of a 256-row tile) so every broadcast 16-byte table load
 * (two channels' (c, d)) feeds four complex MACs; the K taps are walked in chunks of 5 sixteen-byte units per row
 * (5 is odd: the strided LDS.128 row reads are conflict free without padding) staged by
 * cp.async into a 2-deep ring together with the matching slice of the table, so the copy of
 * chunk i+1 runs under the arithmetic of chunk i.  Any K that keeps rows 16-byte aligned, up to
 * ACB_MAXK.  Table entries are (c, d) for every MODE: u8 IQ (rtl.c:334-354), one LDS.128 serving
 * two channels of cmac2; float32 real samples, D += wf[i]*S (air.c:314-333); CS16 IQ, same complex
 * MAC as u8 on (float)int16 (soapy.c:239-242 with the /32768.0 folded into the table, sdrplay.c:218-222).
 * ---------------------------------------------------------------------------------------- */

constexpr int C2_ROWS = 256;
enum { IN_U8IQ = 0, IN_F32REAL = 1, IN_CS16IQ = 2 };   /* input sample formats (acb_internal.h: InputKind) */

template <int MODE> struct C2 {
	/* 16-byte units of a row per chunk: odd, so the strided per-thread LDS.128 row reads are conflict free with rows
	 * packed back to back.  (Whole-sector chunks of 6 units with a padded row stride were tried for the 4-byte-per-tap
	 * inputs: no gain, 42.4 % vs 43 % of HBM peak on the real-input kernel — their limit was elsewhere, see
	 * k_channelize_real4.) */
	static constexpr int UNITS = 5;
	static constexpr int ROW_UNITS = UNITS;                      /* shared-memory row stride in units */
	static constexpr int STAGES = 2;                             /* cp.async ring depth */
	static constexpr int TAP_BYTES = MODE == IN_U8IQ ? 2 : 4;    /* input bytes per tap */
	static constexpr int TAPS_PER_UNIT = 16 / TAP_BYTES;
	static constexpr int W_BYTES = 8;                            /* table bytes per (tap, channel): (c, d) */
	static constexpr int CHUNK_TAPS = UNITS * TAPS_PER_UNIT;
	static constexpr int TILE_BYTES = C2_ROWS * ROW_UNITS * 16;
	static constexpr int WF_BYTES = CHUNK_TAPS * CH_GROUP * W_BYTES;
	static constexpr int STAGE_BYTES = TILE_BYTES + WF_BYTES;
};

/* (float)int16 for both halves of a CS16 sample (soapy.c:239-240, sdrplay.c:218-219) of row A (word wa)
 * and row B (word wb), row-packed like cvt_iq: x ^ 0x8000 planted in the mantissa of 2^23, then
 * 2^23 + 2^15 removed — exact */
__device__ __forceinline__ void cvt_cs16(unsigned wa, unsigned wb, float2 &re, float2 &im)
{
	const unsigned va = wa ^ 0x80008000u, vb = wb ^ 0x80008000u;
	re = make_float2(__uint_as_float(__byte_perm(va, 0x4B000000u, 0x7410)), __uint_as_float(__byte_perm(vb, 0x4B000000u, 0x7410)));
	im = make_float2(__uint_as_float(__byte_perm(va, 0x4B000000u, 0x7432)), __uint_as_float(__byte_perm(vb, 0x4B000000u, 0x7432)));
	re = __fadd2_rn(re, make_float2(-8421376.0f, -8421376.0f));
	im = __fadd2_rn(im, make_float2(-8421376.0f, -8421376.0f));
}

/* air.c:317-318: D += wf[i] * S — (c*S, d*S) rounded, then the accumulate rounded.  Scalar
 * products + packed add: ptxas leaves that pair unfused (it contracts FMUL2 -> FADD2). */
__device__ __forceinline__ void rmac(float2 &acc, float sv, const float2 w)
{
	acc = __fadd2_rn(acc, make_float2(__fmul_rn(w.x, sv), __fmul_rn(w.y, sv)));
}

template <int MODE>
__global__ void __launch_bounds__(CH_TILE)
k_channelize(const uint8_t *__restrict__ in, size_t stream_stride, const uint8_t *__restrict__ wf,
              float *__restrict__ dm, int K, int taps, int nch, int ngrp, size_t nsamp, float nz)
{
	/* nz: -0.0f, the addend of cmac2's product FFMA2s (a kernel argument on purpose, see cmac2) */
	using T = C2<MODE>;
	extern __shared__ __align__(16) unsigned char smem[];
	const int t = threadIdx.x;
	const int blk = blockIdx.x, s = blockIdx.y;
	const size_t rowbytes = (size_t)K * T::TAP_BYTES;
	const int U = taps * T::TAP_BYTES / 16;                          /* units of each row that carry taps (taps <= K) */
	const int nchunk = (U + T::UNITS - 1) / T::UNITS;
	const uint8_t *src_blk = in + (size_t)s * stream_stride + (size_t)blk * OUTBLK * rowbytes;
	constexpr int NTILE = OUTBLK / C2_ROWS;
	const int nstep = NTILE * nchunk;

	{
		const int g = blockIdx.z;                                    /* channel group of 8: one CTA each */
		const uint8_t *wsrc = wf + ((size_t)s * ngrp + g) * taps * CH_GROUP * T::W_BYTES;

		auto issue = [&](int step) {
			const int tile = step / nchunk, ck = step - tile * nchunk;
			unsigned char *st = smem + (size_t)(step % T::STAGES) * T::STAGE_BYTES;
			const int uc = min(T::UNITS, U - ck * T::UNITS);         /* units of this chunk */
			const uint8_t *tsrc = src_blk + (size_t)tile * C2_ROWS * rowbytes + (size_t)ck * T::UNITS * 16;
			{
				/* unit u = t + 128*i of the chunk tile lives at (row u/uc, column u%uc): one division
				 * per chunk, then incremental (the address arithmetic is a fifth of the kernel's
				 * instructions otherwise) */
				int row = t / uc, j = t - row * uc;
				const int drow = CH_TILE / uc, dj = CH_TILE - drow * uc;
				unsigned char *dst = st + ((size_t)row * T::ROW_UNITS + j) * 16;
				const uint8_t *src = tsrc + (size_t)row * rowbytes + (size_t)j * 16;
				const size_t dstep = ((size_t)drow * T::ROW_UNITS + dj) * 16, sstep = (size_t)drow * rowbytes + (size_t)dj * 16;
				const size_t dwrap = (size_t)(T::ROW_UNITS - uc) * 16, swrap = rowbytes - (size_t)uc * 16;
				for (int u = t; u < C2_ROWS * uc; u += CH_TILE) {
					cp_async16(dst, src);
					dst += dstep; src += sstep; j += dj;
					if (j >= uc) { j -= uc; dst += dwrap; src += swrap; }
				}
			}
			const int wunits = uc * T::TAPS_PER_UNIT * CH_GROUP * T::W_BYTES / 16;
			const uint8_t *ws = wsrc + (size_t)ck * T::CHUNK_TAPS * CH_GROUP * T::W_BYTES;
			for (int u = t; u < wunits; u += CH_TILE) cp_async16(st + T::TILE_BYTES + (size_t)u * 16, ws + (size_t)u * 16);
			cp_async_commit();
		};

		/* float32 real: acc0 = row A (re, im), acc1 = row B (re, im).  IQ modes, row-packed for cmac2:
		 * acc0 = re (row A, row B), acc1 = im (row A, row B). */
		float2 acc0[CH_GROUP], acc1[CH_GROUP];
#pragma unroll
		for (int c = 0; c < CH_GROUP; c++) acc0[c] = acc1[c] = make_float2(0.f, 0.f);

		/* prologue: STAGES-1 chunks in flight; every iteration commits exactly one group (possibly
		 * empty) so that "all but the newest STAGES-1 groups" always means "chunk `step` landed" */
#pragma unroll
		for (int i = 0; i < T::STAGES - 1; i++) {
			if (i < nstep) issue(i); else cp_async_commit();
		}
		for (int step = 0; step < nstep; step++) {
			if (step + T::STAGES - 1 < nstep) issue(step + T::STAGES - 1); else cp_async_commit();
			asm volatile("cp.async.wait_group %0;" ::"n"(T::STAGES - 1) : "memory");
			__syncthreads();                                         /* chunk `step` visible to all */
			const int tile = step / nchunk, ck = step - tile * nchunk;
			const unsigned char *st = smem + (size_t)(step % T::STAGES) * T::STAGE_BYTES;
			const int uc = min(T::UNITS, U - ck * T::UNITS);
			const uint4 *rowA = reinterpret_cast<const uint4 *>(st) + (size_t)t * T::ROW_UNITS;
			const uint4 *rowB = reinterpret_cast<const uint4 *>(st) + (size_t)(t + CH_TILE) * T::ROW_UNITS;
			for (int j = 0; j < uc; j++) {
				const uint4 qa = rowA[j], qb = rowB[j];
				const unsigned wa[4] = { qa.x, qa.y, qa.z, qa.w }, wb[4] = { qb.x, qb.y, qb.z, qb.w };
				if (MODE == IN_F32REAL) {
					const float2 *wj = reinterpret_cast<const float2 *>(st + T::TILE_BYTES) + (size_t)j * 4 * CH_GROUP;
#pragma unroll
					for (int e = 0; e < 4; e++) {
						const float sa = __uint_as_float(wa[e]), sb = __uint_as_float(wb[e]);
#pragma unroll
						for (int c = 0; c < CH_GROUP; c++) {
							const float2 w = wj[e * CH_GROUP + c];
							rmac(acc0[c], sa, w);
							rmac(acc1[c], sb, w);
						}
					}
				} else {
					/* one float4 = the (c, d) entries of channels 2i and 2i+1 */
					constexpr int SPW = MODE == IN_CS16IQ ? 1 : 2;       /* complex samples per 32-bit word */
					const float4 *wj = reinterpret_cast<const float4 *>(st + T::TILE_BYTES) + (size_t)j * 4 * SPW * CH_GROUP / 2;
#pragma unroll
					for (int e = 0; e < 4; e++) {
#pragma unroll
						for (int h = 0; h < SPW; h++) {
							float2 re, im;
							if (MODE == IN_CS16IQ) cvt_cs16(wa[e], wb[e], re, im);
							else cvt_iq(wa[e], wb[e], h, re, im);
#pragma unroll
							for (int c = 0; c < CH_GROUP; c += 2) {
								const float4 w = wj[((SPW * e + h) * CH_GROUP + c) / 2];
								cmac2(acc0[c], acc1[c], re, im, w.x, w.y, nz);
								cmac2(acc0[c + 1], acc1[c + 1], re, im, w.z, w.w, nz);
							}
						}
					}
				}
			}
			if (ck == nchunk - 1) {                                  /* row complete: |D| out, restart */
				const int nc = min(CH_GROUP, nch - g * CH_GROUP);
#pragma unroll
				for (int half = 0; half < 2; half++) {
					float2 d[CH_GROUP];                              /* (re, im) of this half's row */
#pragma unroll
					for (int c = 0; c < CH_GROUP; c++)
						d[c] = MODE == IN_F32REAL ? (half ? acc1[c] : acc0[c])
						                          : (half ? make_float2(acc0[c].y, acc1[c].y) : make_float2(acc0[c].x, acc1[c].x));
					const size_t m = (size_t)blk * OUTBLK + (size_t)tile * C2_ROWS + t + half * CH_TILE;
					float *o = dm + ((size_t)s * nsamp + m) * nch + g * CH_GROUP;
					if (nc == CH_GROUP && (nch & 3) == 0) {
						reinterpret_cast<float4 *>(o)[0] = make_float4(envelope(d[0]), envelope(d[1]), envelope(d[2]), envelope(d[3]));
						reinterpret_cast<float4 *>(o)[1] = make_float4(envelope(d[4]), envelope(d[5]), envelope(d[6]), envelope(d[7]));
					} else {
#pragma unroll
						for (int c = 0; c < CH_GROUP; c++)
							if (c < nc) o[c] = envelope(d[c]);
					}
				}
#pragma unroll
				for (int c = 0; c < CH_GROUP; c++) acc0[c] = acc1[c] = make_float2(0.f, 0.f);
			}
			__syncthreads();                                         /* stage may be refilled by issue(step+2) */
		}
	}
}

/* The float32 real-input form of the same pipeline with FOUR output rows per thread (64 threads per 256-row tile).
 * air.c:317-318 is D += wf[i]*S: half the arithmetic of a complex tap per table entry, so with two rows per thread the
 * warp-uniform table loads (64 bytes per tap) were a fifth of the instruction stream and the shared-memory pipe, not the
 * FP32 pipe, set the pace (round 1: 43 % of HBM peak, 58 % of this arithmetic's FP32 ceiling).  Four rows per thread
 * halve the table traffic per MAC; same arithmetic, same order, bit-identical results. */
constexpr int R4_THREADS = 64, R4_RPT = C2_ROWS / R4_THREADS;

__global__ void __launch_bounds__(R4_THREADS)
k_channelize_real4(const uint8_t *__restrict__ in, size_t stream_stride, const uint8_t *__restrict__ wf,
                   float *__restrict__ dm, int K, int taps, int nch, int ngrp, size_t nsamp)
{
	constexpr int UNITS = 5, TAPS_PER_UNIT = 4, W_BYTES = 8, CHUNK_TAPS = UNITS * TAPS_PER_UNIT, STAGES = 2;
	constexpr int TILE_BYTES = C2_ROWS * UNITS * 16, STAGE_BYTES = TILE_BYTES + CHUNK_TAPS * CH_GROUP * W_BYTES;
	extern __shared__ __align__(16) unsigned char smem[];
	const int t = threadIdx.x;
	const int blk = blockIdx.x, s = blockIdx.y, g = blockIdx.z;
	const size_t rowbytes = (size_t)K * 4;
	const int U = taps / TAPS_PER_UNIT;                              /* taps is padded to whole units by the caller */
	const int nchunk = (U + UNITS - 1) / UNITS;
	const uint8_t *src_blk = in + (size_t)s * stream_stride + (size_t)blk * OUTBLK * rowbytes;
	constexpr int NTILE = OUTBLK / C2_ROWS;
	const int nstep = NTILE * nchunk;
	const uint8_t *wsrc = wf + ((size_t)s * ngrp + g) * taps * CH_GROUP * W_BYTES;

	auto issue = [&](int step) {
		const int tile = step / nchunk, ck = step - tile * nchunk;
		unsigned char *st = smem + (size_t)(step % STAGES) * STAGE_BYTES;
		const int uc = min(UNITS, U - ck * UNITS);
		const uint8_t *tsrc = src_blk + (size_t)tile * C2_ROWS * rowbytes + (size_t)ck * UNITS * 16;
		int row = t / uc, j = t - row * uc;
		const int drow = R4_THREADS / uc, dj = R4_THREADS - drow * uc;
		unsigned char *dst = st + ((size_t)row * UNITS + j) * 16;
		const uint8_t *src = tsrc + (size_t)row * rowbytes + (size_t)j * 16;
		const size_t dstep = ((size_t)drow * UNITS + dj) * 16, sstep = (size_t)drow * rowbytes + (size_t)dj * 16;
		const size_t dwrap = (size_t)(UNITS - uc) * 16, swrap = rowbytes - (size_t)uc * 16;
		for (int u = t; u < C2_ROWS * uc; u += R4_THREADS) {
			cp_async16(dst, src);
			dst += dstep; src += sstep; j += dj;
			if (j >= uc) { j -= uc; dst += dwrap; src += swrap; }
		}
		const int wunits = uc * TAPS_PER_UNIT * CH_GROUP * W_BYTES / 16;
		const uint8_t *ws = wsrc + (size_t)ck * CHUNK_TAPS * CH_GROUP * W_BYTES;
		for (int u = t; u < wunits; u += R4_THREADS) cp_async16(st + TILE_BYTES + (size_t)u * 16, ws + (size_t)u * 16);
		cp_async_commit();
	};

	float2 acc[R4_RPT][CH_GROUP];
#pragma unroll
	for (int r = 0; r < R4_RPT; r++)
#pragma unroll
		for (int c = 0; c < CH_GROUP; c++) acc[r][c] = make_float2(0.f, 0.f);

	if (0 < nstep) issue(0); else cp_async_commit();
	for (int step = 0; step < nstep; step++) {
		if (step + 1 < nstep) issue(step + 1); else cp_async_commit();
		asm volatile("cp.async.wait_group %0;" ::"n"(STAGES - 1) : "memory");
		__syncthreads();
		const int tile = step / nchunk, ck = step - tile * nchunk;
		const unsigned char *st = smem + (size_t)(step % STAGES) * STAGE_BYTES;
		const int uc = min(UNITS, U - ck * UNITS);
		const uint4 *rows = reinterpret_cast<const uint4 *>(st) + (size_t)t * UNITS;
		for (int j = 0; j < uc; j++) {
			uint4 q[R4_RPT];
#pragma unroll
			for (int r = 0; r < R4_RPT; r++) q[r] = rows[(size_t)r * R4_THREADS * UNITS + j];
			const float2 *wj = reinterpret_cast<const float2 *>(st + TILE_BYTES) + (size_t)j * 4 * CH_GROUP;
#pragma unroll
			for (int e = 0; e < 4; e++) {
				float sv[R4_RPT];
#pragma unroll
				for (int r = 0; r < R4_RPT; r++) sv[r] = __uint_as_float(e == 0 ? q[r].x : e == 1 ? q[r].y : e == 2 ? q[r].z : q[r].w);
#pragma unroll
				for (int c = 0; c < CH_GROUP; c++) {
					const float2 w = wj[e * CH_GROUP + c];
#pragma unroll
					for (int r = 0; r < R4_RPT; r++) rmac(acc[r][c], sv[r], w);
				}
			}
		}
		if (ck == nchunk - 1) {                                  /* rows complete: |D| out, restart */
			const int nc = min(CH_GROUP, nch - g * CH_GROUP);
#pragma unroll
			for (int r = 0; r < R4_RPT; r++) {
				const size_t m = (size_t)blk * OUTBLK + (size_t)tile * C2_ROWS + t + r * R4_THREADS;
				float *o = dm + ((size_t)s * nsamp + m) * nch + g * CH_GROUP;
				if (nc == CH_GROUP && (nch & 3) == 0) {
					reinterpret_cast<float4 *>(o)[0] = make_float4(envelope(acc[r][0]), envelope(acc[r][1]), envelope(acc[r][2]), envelope(acc[r][3]));
					reinterpret_cast<float4 *>(o)[1] = make_float4(envelope(acc[r][4]), envelope(acc[r][5]), envelope(acc[r][6]), envelope(acc[r][7]));
				} else {
#pragma unroll
					for (int c = 0; c < CH_GROUP; c++)
						if (c < nc) o[c] = envelope(acc[r][c]);
				}
#pragma unroll
				for (int c = 0; c < CH_GROUP; c++) acc[r][c] = make_float2(0.f, 0.f);
			}
		}
		__syncthreads();
	}
}

static int launch_channelize_real4(const void *in, size_t stream_stride, const void *wf, float *dm,
                                   int K, int taps, int nch, int nstreams, int nblk, size_t nsamp, cudaStream_t stream)
{
	if (nblk == 0) return 0;
	const int ngrp = (nch + CH_GROUP - 1) / CH_GROUP;
	const size_t smem = 2 * (size_t)(C2_ROWS * 5 * 16 + 20 * CH_GROUP * 8);
	cudaError_t e = cudaFuncSetAttribute(k_channelize_real4, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
	if (e != cudaSuccess) return (int)e;
	e = cudaFuncSetAttribute(k_channelize_real4, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
	if (e != cudaSuccess) return (int)e;
	dim3 grid(nblk, nstreams, ngrp);
	k_channelize_real4<<<grid, R4_THREADS, smem, stream>>>(reinterpret_cast<const uint8_t *>(in), stream_stride,
	                                                      reinterpret_cast<const uint8_t *>(wf), dm, K, taps, nch, ngrp, nsamp);
	return (int)cudaGetLastError();
}

size_t channelize_smem_bytes(int mode)
{
	return mode == IN_F32REAL ? (size_t)C2<IN_F32REAL>::STAGES * C2<IN_F32REAL>::STAGE_BYTES
	       : mode == IN_CS16IQ ? (size_t)C2<IN_CS16IQ>::STAGES * C2<IN_CS16IQ>::STAGE_BYTES
	                           : (size_t)C2<IN_U8IQ>::STAGES * C2<IN_U8IQ>::STAGE_BYTES;
}

template <int MODE>
static int launch_channelize_t(const void *in, size_t stream_stride, const void *wf, float *dm,
                               int K, int taps, int nch, int nstreams, int nblk, size_t nsamp, cudaStream_t stream)
{
	if (nblk == 0) return 0;
	const int ngrp = (nch + CH_GROUP - 1) / CH_GROUP;
	const size_t smem = (size_t)C2<MODE>::STAGES * C2<MODE>::STAGE_BYTES;
	cudaError_t e = cudaFuncSetAttribute(k_channelize<MODE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
	if (e != cudaSuccess) return (int)e;
	/* both kernels ask for the largest shared-memory carve-out: an SM's L1/shared split only
	 * changes when the SM is idle, so kernels that prefer different splits cannot be co-resident
	 * — and the demod of submit i is meant to run underneath the channelizer of submit i+1 */
	e = cudaFuncSetAttribute(k_channelize<MODE>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
	if (e != cudaSuccess) return (int)e;
	dim3 grid(nblk, nstreams, ngrp);
	k_channelize<MODE><<<grid, CH_TILE, smem, stream>>>(reinterpret_cast<const uint8_t *>(in), stream_stride,
	                                                    reinterpret_cast<const uint8_t *>(wf), dm, K, taps, nch, ngrp, nsamp, -0.0f);
	return (int)cudaGetLastError();
}

/* whole 1024-row blocks of any input kind; the caller sends remaining rows to the generic kernel */
int launch_channelize(int mode, const void *in, size_t stream_stride_bytes, const float *wf, float *dm,
                      int K, int taps, int nch, int nstreams, int nblk, size_t nsamp, cudaStream_t stream)
{
	switch (mode) {
	case IN_F32REAL: {
		static const bool two_rows = getenv("ACB_REAL_ROWS") && atoi(getenv("ACB_REAL_ROWS")) == 2;     /* A/B switch: the 2-rows-per-thread form */
		return two_rows ? launch_channelize_t<IN_F32REAL>(in, stream_stride_bytes, wf, dm, K, taps, nch, nstreams, nblk, nsamp, stream)
		                : launch_channelize_real4(in, stream_stride_bytes, wf, dm, K, taps, nch, nstreams, nblk, nsamp, stream);
	}
	case IN_CS16IQ: return launch_channelize_t<IN_CS16IQ>(in, stream_stride_bytes, wf, dm, K, taps, nch, nstreams, nblk, nsamp, stream);
	default: return launch_channelize_t<IN_U8IQ>(in, stream_stride_bytes, wf, dm, K, taps, nch, nstreams, nblk, nsamp, stream);
	}
}

/* ------------------------------------------------------------------------------------------
 * K1, fast form (ACB_FLAG_FAST_CHANNELIZER).  The reference's mixer table is a sampled complex
 * exponential: when (Fr - Fc) is a whole number k of 12.5 kHz steps — the planner's normal outcome,
 * frequencies are rounded to that raster (rtl.c:245-247) — wf[ind] = g*exp(-j*2*pi*k*ind/K) and the
 * boxcar sum D = sum_ind x[ind]*wf[ind] is bin k of a K-point DFT of the row.  Split ind = (K/4)*n1 + n2:
 *
 *     D_c = sum_{n2 < K/4} T_c[n2] * Y_{k_c mod 4}[n2],   Y_r[n2] = sum_{n1 < 4} x[(K/4)*n1 + n2] * (-j)^(r*n1)
 *
 * (k is always even: the float images of Fr and Fc that the reference mixes with are multiples of 8 Hz,
 * so only Y_0 = x0+x1+x2+x3 and Y_2 = x0-x1+x2-x3 occur.)
 *
 * Y_r is a 4-point DFT across the four quarters of the row: additions only, EXACT in float (integer
 * samples), and shared by every channel of the stream; each channel then needs K/4 complex MACs instead
 * of K.  The -127.37 offset of rtl.c:338-339 drops out (a channel is never at bin 0: chooseFc keeps it
 * 25 kHz from the centre).  FP32 work per input sample falls from 8*C to 2.5 + C lane-ops (C = 8: 64 ->
 * 10.5), which moves the kernel from the FP32 roof towards the HBM roof.
 *
 * This is NOT the reference's operation order: the envelope differs from the reference's in the last
 * bits.  Measured (tests/test_gpu_fast.py, tests/test_fast_oracle.py), relative to the total in-band
 * signal: 3e-7 from the exact double-precision DFT bin — the reference, whose table carries float phase
 * rounding (float AMFreq*ind), sits at 1.8e-6 — bit-identical to its CPU restatement
 * (oracle: orc_channelize_dft), and decoded messages identical on every fixture.  The default (exact)
 * kernel above stays bit-identical; this one is what the north star's tolerance (messages bit-exact,
 * float intermediates within tolerance) buys.
 *
 * Shape: one CTA = one 1024-row block of one stream for 8 channels, 16 tiles of 64 rows dealt round-robin
 * to its warps; lane l owns rows l and l+32 of a tile, and every FP32 instruction is packed across those
 * two rows (FADD2/FFMA2: half the issue slots; the twiddle rides FFMA2's scalar-broadcast operand).
 * Whole rows are fetched by bulk copies (cp.async.bulk of one or two rows, completion on the warp's
 * mbarrier) issued by one lane: every 32-byte sector fetched is used, no per-unit addressing.
 * Warps do not synchronise with each other after the twiddles are in shared memory; with one private
 * buffer per warp, the copy of a warp's next tile hides under the other warps' arithmetic.
 * ---------------------------------------------------------------------------------------- */

constexpr int DFT_ROWS = 64;                     /* rows per tile: 2 per lane */

__device__ __forceinline__ float2 ffma2(float2 a, float2 b, float2 c)
{
	float2 d;
	asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(reinterpret_cast<unsigned long long &>(d))
	    : "l"(reinterpret_cast<unsigned long long &>(a)), "l"(reinterpret_cast<unsigned long long &>(b)),
	      "l"(reinterpret_cast<unsigned long long &>(c)));
	return d;
}
__device__ __forceinline__ float2 fsub2(float2 a, float2 b) { return __fadd2_rn(a, make_float2(-b.x, -b.y)); }

/* byte `k` of word wa / wb as 32768 + u, packed (row A, row B): the byte lands in bits 8..15 of the
 * mantissa of 2^15, where the unit weight is */
template <int KB> __device__ __forceinline__ float2 dft_cvt(unsigned wa, unsigned wb)
{
	constexpr unsigned sel = 0x7404u | (KB << 4);
	return make_float2(__uint_as_float(__byte_perm(wa, 0x47000000u, sel)), __uint_as_float(__byte_perm(wb, 0x47000000u, sel)));
}

struct DftAcc { float2 a, b, p, q; };            /* re = a - b, im = p + q; each packed (row A, row B) */

/* acc += y * t for the lane's two rows; t = (Tr, Ti) is warp-uniform.  Passing the same scalar as both
 * halves of the multiplier makes ptxas use FFMA2's broadcast operand form (R.F32): no pair to build.
 * Four independent accumulators keep the dependent FFMA2 chains short. */
__device__ __forceinline__ void dft_mac(DftAcc &acc, float2 yr, float2 yi, float2 t)
{
	const float2 tr = make_float2(t.x, t.x), ti = make_float2(t.y, t.y);
	acc.a = ffma2(yr, tr, acc.a);
	acc.b = ffma2(yi, ti, acc.b);
	acc.p = ffma2(yr, ti, acc.p);
	acc.q = ffma2(yi, tr, acc.q);
}

/* mbarrier + bulk-copy (TMA 1-D) plumbing */
__device__ __forceinline__ unsigned smem_u32(const void *p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(unsigned long long *bar, unsigned count)
{
	asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(unsigned long long *bar, unsigned bytes)
{
	asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned long long *bar, unsigned parity)
{
	asm volatile("{\n\t.reg .pred p;\n\tWAIT_%=:\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t@p bra DONE_%=;\n\tbra WAIT_%=;\n\tDONE_%=:\n\t}"
	             ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
__device__ __forceinline__ void bulk_g2s(void *dst, const void *src, unsigned bytes, unsigned long long *bar)
{
	asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
	             ::"r"(smem_u32(dst)), "l"(src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}

/* one lane of a converged warp, chosen by the hardware: the compiler then knows the guarded block runs once per
 * warp and keeps warp-uniform operands (addresses built from a shuffled warp index) in uniform registers */
__device__ __forceinline__ bool elect_one()
{
	unsigned p;
	asm volatile("{\n\t.reg .pred q;\n\telect.sync _|q, 0xffffffff;\n\tselp.u32 %0, 1, 0, q;\n\t}" : "=r"(p));
	return p != 0;
}

/* Shared-memory plan of one CTA: WARPS warps, each with STAGES private tile buffers of 64 rows. */
template <int UNITS, int WARPS, int STAGES> struct DftPlan {
	static constexpr int ROWBYTES = UNITS * 16;
	/* rows per bulk copy, each copy followed by 16 bytes of padding.  The eight lanes of an LDS.128
	 * phase read eight consecutive rows at the same offset: they hit eight different 16-byte bank groups
	 * when the row stride is an odd number of units (UNITS odd after padding every row), or — UNITS = 20,
	 * stride = 4 mod 8 — when every second row is shifted by one more unit (pad after every two rows). */
	static constexpr int RPC = (UNITS % 8 == 4) ? 2 : 1;
	static constexpr int GROUP = RPC * ROWBYTES + 16;
	static constexpr int TILE_BYTES = DFT_ROWS / RPC * GROUP;
	static __device__ __forceinline__ int row_off(int r) { return (r / RPC) * GROUP + (r % RPC) * ROWBYTES; }
	static constexpr int N2 = UNITS * 2;                                     /* K/4 */
	static constexpr int TW_BYTES = N2 * CH_GROUP * 8;
	static constexpr int BAR_OFF = WARPS * STAGES * TILE_BYTES + TW_BYTES;
	static constexpr int SMEM = BAR_OFF + WARPS * STAGES * 8;
};

template <int UNITS, int WARPS, int STAGES, int MINB, bool FOLD8>
__global__ void __launch_bounds__(32 * WARPS, MINB)
k_channelize_dft(const uint8_t *__restrict__ in, size_t stream_stride, const float2 *__restrict__ tw,
                 const unsigned *__restrict__ meta, float *__restrict__ dm, int nch, int ngrp, size_t nsamp)
{
	using P = DftPlan<UNITS, WARPS, STAGES>;
	constexpr int CU = UNITS / 4;                 /* 16-byte units per quarter row */
	constexpr int N2 = P::N2;
	constexpr int NTILE = OUTBLK / DFT_ROWS;
	extern __shared__ __align__(16) unsigned char smem[];
	const int l = threadIdx.x & 31, w = threadIdx.x >> 5;
	const int blk = blockIdx.x, s = blockIdx.y, g = blockIdx.z;
	unsigned char *mytiles = smem + (size_t)w * STAGES * P::TILE_BYTES;
	const float4 *stw = reinterpret_cast<const float4 *>(smem + (size_t)WARPS * STAGES * P::TILE_BYTES);   /* [ch][n2] (Tr, Ti) */
	unsigned long long *bars = reinterpret_cast<unsigned long long *>(smem + P::BAR_OFF) + w * STAGES;
	const uint8_t *src_blk = in + (size_t)s * stream_stride + (size_t)blk * OUTBLK * P::ROWBYTES;
	const unsigned m = meta[(size_t)s * ngrp + g];    /* residue k_c mod 4 (0 or 2) of channel slot c in bits 2c, 2c+1 */

	if (l == 0)
		for (int i = 0; i < STAGES; i++) mbar_init(bars + i, 1);
	asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
	{
		const uint4 *tsrc = reinterpret_cast<const uint4 *>(tw + ((size_t)s * ngrp + g) * N2 * CH_GROUP);
		uint4 *tdst = reinterpret_cast<uint4 *>(smem + (size_t)WARPS * STAGES * P::TILE_BYTES);
		for (int q = threadIdx.x; q < P::TW_BYTES / 16; q += 32 * WARPS) cp_async16(tdst + q, tsrc + q);
		cp_async_commit();
		cp_async_wait_all();
	}
	__syncthreads();

	/* this warp's tiles: w, w + WARPS, ...; tile n of the warp uses stage n % STAGES */
	const int ntile = (NTILE - w + WARPS - 1) / WARPS;
	auto issue = [&](int n) {
		const int tile = w + n * WARPS;
		unsigned char *st = mytiles + (size_t)(n % STAGES) * P::TILE_BYTES;
		unsigned long long *bar = bars + n % STAGES;
		if (l == 0) {
			mbar_expect_tx(bar, DFT_ROWS * P::ROWBYTES);
			const uint8_t *src = src_blk + (size_t)tile * DFT_ROWS * P::ROWBYTES;
#pragma unroll 4
			for (int i = 0; i < DFT_ROWS / P::RPC; i++)
				bulk_g2s(st + (size_t)i * P::GROUP, src + (size_t)i * P::RPC * P::ROWBYTES, P::RPC * P::ROWBYTES, bar);
		}
	};
	for (int n = 0; n < STAGES && n < ntile; n++) issue(n);
	const int nc = min(CH_GROUP, nch - g * CH_GROUP);

	for (int n = 0; n < ntile; n++) {
		const int tile = w + n * WARPS;
		mbar_wait(bars + n % STAGES, (unsigned)((n / STAGES) & 1));
		const unsigned char *st = mytiles + (size_t)(n % STAGES) * P::TILE_BYTES;
		const uint4 *rowA = reinterpret_cast<const uint4 *>(st + P::row_off(l));
		const uint4 *rowB = reinterpret_cast<const uint4 *>(st + P::row_off(l + 32));
		DftAcc acc[CH_GROUP];
#pragma unroll
		for (int c = 0; c < CH_GROUP; c++) acc[c].a = acc[c].b = acc[c].p = acc[c].q = make_float2(0.f, 0.f);

		if constexpr (!FOLD8) {
			/* unit j covers samples 8j..8j+7 of each quarter: one LDS.128 per quarter and row (their latency
			 * is left to the other warps of the SM to cover) */
	#pragma unroll 1
			for (int j = 0; j < CU; j++) {
				uint4 qa[4], qb[4];
	#pragma unroll
				for (int n1 = 0; n1 < 4; n1++) { qa[n1] = rowA[n1 * CU + j]; qb[n1] = rowB[n1 * CU + j]; }
	#pragma unroll
				for (int eh = 0; eh < 2; eh++) {      /* four samples of each quarter at a time */
					float2 y0r[4], y0i[4], y2r[4], y2i[4];
	#pragma unroll
					for (int k = 0; k < 4; k++) {
						float2 xi[4], xq[4];
	#pragma unroll
						for (int n1 = 0; n1 < 4; n1++) {
							const unsigned wa = eh ? (k < 2 ? qa[n1].z : qa[n1].w) : (k < 2 ? qa[n1].x : qa[n1].y);
							const unsigned wb = eh ? (k < 2 ? qb[n1].z : qb[n1].w) : (k < 2 ? qb[n1].x : qb[n1].y);
							if (k & 1) { xi[n1] = dft_cvt<2>(wa, wb); xq[n1] = dft_cvt<3>(wa, wb); }
							else       { xi[n1] = dft_cvt<0>(wa, wb); xq[n1] = dft_cvt<1>(wa, wb); }
						}
						/* sums carry the 2 x 32768 planted by dft_cvt (exact: < 2^24); differences do not.  Y_0
						 * also sheds the converter's mid-scale 4 x 127.5 here: any constant is invisible to a
						 * channel (its twiddles sum to zero) but a large one costs accumulate precision */
						const float2 sI02 = __fadd2_rn(xi[0], xi[2]), sI13 = __fadd2_rn(xi[1], xi[3]);
						const float2 sQ02 = __fadd2_rn(xq[0], xq[2]), sQ13 = __fadd2_rn(xq[1], xq[3]);
						const float2 bias = make_float2(-131582.0f, -131582.0f);
						y0r[k] = __fadd2_rn(__fadd2_rn(sI02, sI13), bias);
						y0i[k] = __fadd2_rn(__fadd2_rn(sQ02, sQ13), bias);
						y2r[k] = fsub2(sI02, sI13);
						y2i[k] = fsub2(sQ02, sQ13);
					}
					/* channel c's four twiddles: two LDS.128, fetched one channel ahead of their use so the
					 * load latency hides under the previous channel's FFMA2s (the residue dispatch below is a
					 * uniform branch the scheduler does not move loads across) */
					const float4 *tj = stw + (j * 2 + eh) * 2;
					float4 t0 = tj[0], t1 = tj[1];
	#pragma unroll
					for (int c = 0; c < CH_GROUP; c++) {
						const float4 u0 = t0, u1 = t1;
						if (c + 1 < CH_GROUP) { t0 = tj[(c + 1) * (N2 / 2)]; t1 = tj[(c + 1) * (N2 / 2) + 1]; }
						const float2 tt[4] = { make_float2(u0.x, u0.y), make_float2(u0.z, u0.w), make_float2(u1.x, u1.y), make_float2(u1.z, u1.w) };
						if (((m >> (2 * c)) & 3u) == 0) {             /* warp-uniform: k_c mod 4 is 0 or 2 */
	#pragma unroll
							for (int k = 0; k < 4; k++) dft_mac(acc[c], y0r[k], y0i[k], tt[k]);
						} else {
	#pragma unroll
							for (int k = 0; k < 4; k++) dft_mac(acc[c], y2r[k], y2i[k], tt[k]);
						}
					}
				}
			}
		} else {
			/* Bins are even (k = 2k'), so the row folds in half first: z[n] = x[n] + x[n + K/2] and D is bin
			 * k' of the K/2-point DFT of z; the same four-way split of THAT gives
			 *   D = sum_{n2 < K/8} T[n2] * Y'_{k' mod 4}[n2],   Y'_r[n2] = sum_{n1<4} z[(K/8)*n1 + n2] * (-j)^(r*n1)
			 * with the same twiddles T[n2] = exp(-j*2*pi*k*n2/K)/K/127.5 and all four residues in play:
			 * 26 packed additions per n2 (exact) and K/8 complex MACs per channel.  Group g4 covers samples
			 * 4*g4..4*g4+3 of each eighth of the row: one LDS.64 per eighth and row. */
			const unsigned char *ra = st + P::row_off(l), *rb = st + P::row_off(l + 32);
#pragma unroll 1
			for (int g4 = 0; g4 < CU; g4++) {
				uint2 ea[8], eb[8];
#pragma unroll
				for (int e = 0; e < 8; e++) {
					ea[e] = *reinterpret_cast<const uint2 *>(ra + e * (UNITS * 2) + g4 * 8);
					eb[e] = *reinterpret_cast<const uint2 *>(rb + e * (UNITS * 2) + g4 * 8);
				}
				float2 yr[4][4], yi[4][4];            /* [residue][sample of the group] */
#pragma unroll
				for (int k = 0; k < 4; k++) {
					float2 zi[4], zq[4];
#pragma unroll
					for (int n1 = 0; n1 < 4; n1++) {
						const unsigned wa0 = k < 2 ? ea[n1].x : ea[n1].y, wb0 = k < 2 ? eb[n1].x : eb[n1].y;
						const unsigned wa1 = k < 2 ? ea[n1 + 4].x : ea[n1 + 4].y, wb1 = k < 2 ? eb[n1 + 4].x : eb[n1 + 4].y;
						if (k & 1) {
							zi[n1] = __fadd2_rn(dft_cvt<2>(wa0, wb0), dft_cvt<2>(wa1, wb1));
							zq[n1] = __fadd2_rn(dft_cvt<3>(wa0, wb0), dft_cvt<3>(wa1, wb1));
						} else {
							zi[n1] = __fadd2_rn(dft_cvt<0>(wa0, wb0), dft_cvt<0>(wa1, wb1));
							zq[n1] = __fadd2_rn(dft_cvt<1>(wa0, wb0), dft_cvt<1>(wa1, wb1));
						}
					}
					/* every z carries 2 x 32768 from dft_cvt: sums of four carry 262144 (exact, < 2^24) and Y'_0
					 * also sheds the converter's mid-scale 8 x 127.5; differences carry nothing */
					const float2 sI02 = __fadd2_rn(zi[0], zi[2]), sI13 = __fadd2_rn(zi[1], zi[3]);
					const float2 sQ02 = __fadd2_rn(zq[0], zq[2]), sQ13 = __fadd2_rn(zq[1], zq[3]);
					const float2 dI02 = fsub2(zi[0], zi[2]), dI13 = fsub2(zi[1], zi[3]);
					const float2 dQ02 = fsub2(zq[0], zq[2]), dQ13 = fsub2(zq[1], zq[3]);
					const float2 bias = make_float2(-263164.0f, -263164.0f);
					yr[0][k] = __fadd2_rn(__fadd2_rn(sI02, sI13), bias);
					yi[0][k] = __fadd2_rn(__fadd2_rn(sQ02, sQ13), bias);
					yr[2][k] = fsub2(sI02, sI13);
					yi[2][k] = fsub2(sQ02, sQ13);
					yr[1][k] = __fadd2_rn(dI02, dQ13); yi[1][k] = fsub2(dQ02, dI13);      /* (z0-z2) - j(z1-z3) */
					yr[3][k] = fsub2(dI02, dQ13);      yi[3][k] = __fadd2_rn(dQ02, dI13); /* (z0-z2) + j(z1-z3) */
				}
				const float4 *tj = stw + g4 * 2;
				float4 t0 = tj[0], t1 = tj[1];
#pragma unroll
				for (int c = 0; c < CH_GROUP; c++) {
					const float4 u0 = t0, u1 = t1;
					if (c + 1 < CH_GROUP) { t0 = tj[(c + 1) * (N2 / 2)]; t1 = tj[(c + 1) * (N2 / 2) + 1]; }
					const float2 tt[4] = { make_float2(u0.x, u0.y), make_float2(u0.z, u0.w), make_float2(u1.x, u1.y), make_float2(u1.z, u1.w) };
					const unsigned r8 = (m >> (16 + 2 * c)) & 3u;     /* warp-uniform: (k_c / 2) mod 4 */
					if (r8 == 0) {
#pragma unroll
						for (int k = 0; k < 4; k++) dft_mac(acc[c], yr[0][k], yi[0][k], tt[k]);
					} else if (r8 == 1) {
#pragma unroll
						for (int k = 0; k < 4; k++) dft_mac(acc[c], yr[1][k], yi[1][k], tt[k]);
					} else if (r8 == 2) {
#pragma unroll
						for (int k = 0; k < 4; k++) dft_mac(acc[c], yr[2][k], yi[2][k], tt[k]);
					} else {
#pragma unroll
						for (int k = 0; k < 4; k++) dft_mac(acc[c], yr[3][k], yi[3][k], tt[k]);
					}
				}
			}
		}
		/* every lane has its rows in registers: the stage can take the warp's tile n + STAGES */
		__syncwarp();
		if (n + STAGES < ntile) issue(n + STAGES);
		/* |D| out (rtl.c:353) for the lane's two rows */
#pragma unroll
		for (int half = 0; half < 2; half++) {
			float e[CH_GROUP];
#pragma unroll
			for (int c = 0; c < CH_GROUP; c++) {
				const float re = half ? __fadd_rn(acc[c].a.y, -acc[c].b.y) : __fadd_rn(acc[c].a.x, -acc[c].b.x);
				const float im = half ? __fadd_rn(acc[c].p.y, acc[c].q.y) : __fadd_rn(acc[c].p.x, acc[c].q.x);
				e[c] = __fsqrt_rn(__fmaf_rn(re, re, __fmul_rn(im, im)));      /* |D|: half an ulp, this form's tolerance is 1e-5 */
			}
			const size_t mrow = (size_t)blk * OUTBLK + (size_t)tile * DFT_ROWS + l + half * 32;
			float *o = dm + ((size_t)s * nsamp + mrow) * nch + g * CH_GROUP;
			if (nc == CH_GROUP && (nch & 3) == 0) {
				reinterpret_cast<float4 *>(o)[0] = make_float4(e[0], e[1], e[2], e[3]);
				reinterpret_cast<float4 *>(o)[1] = make_float4(e[4], e[5], e[6], e[7]);
			} else {
#pragma unroll
				for (int c = 0; c < CH_GROUP; c++)
					if (c < nc) o[c] = e[c];
			}
		}
	}
}

template <int UNITS, int WARPS, int STAGES, int MINB, bool FOLD8>
static int launch_dft_t(const uint8_t *in, size_t stream_stride, const float2 *tw, const unsigned *meta, float *dm,
                        int nch, int nstreams, int nblk, size_t nsamp, cudaStream_t stream)
{
	const int ngrp = (nch + CH_GROUP - 1) / CH_GROUP;
	constexpr int smem = DftPlan<UNITS, WARPS, STAGES>::SMEM;
	auto kern = k_channelize_dft<UNITS, WARPS, STAGES, MINB, FOLD8>;
	cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
	if (e != cudaSuccess) return (int)e;
	e = cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
	if (e != cudaSuccess) return (int)e;
	dim3 grid(nblk, nstreams, ngrp);
	kern<<<grid, 32 * WARPS, smem, stream>>>(in, stream_stride, tw, meta, dm, nch, ngrp, nsamp);
	return (int)cudaGetLastError();
}

/* The folded fast form with ONE row per lane and the pair packing moved from "two rows" to "(re, im)": a lane's
 * accumulators for channel c are A = (a, p) and B = (q, b), fed by two FFMA2 per complex MAC —
 *     A += (yr, yr) * (Tr, Ti)        B += (yi, yi) * (Tr, Ti)          re = A.x - B.y, im = A.y + B.x
 * — the very same four sums, term for term and in the same order, that the two-rows-per-lane kernel above keeps in
 * a, b, p, q: the envelope is BIT-IDENTICAL to that kernel's (and to the CPU restatement orc_channelize_dft8).  The
 * shared 4-point DFTs run on (I, Q) pairs, exact in float like before.  What changes is the footprint: a warp's tile
 * is 32 rows (10.5 KB instead of 21 KB) and a thread holds one row's worth of state (~100 registers instead of 162),
 * so 16-20 warps fit an SM instead of 10 — the two-row kernel is latency bound at 2.5 warps per scheduler (ncu: issue
 * active 58 %, stall `wait` 35 %) — and the demod warps that share the SMs displace smaller pieces. */
constexpr int DFT1_ROWS = 32;

/* KIND: IN_U8IQ (2 bytes per complex sample, UNITS = K/8 sixteen-byte units per row) or IN_CS16IQ (4 bytes per complex
 * sample: the same kernel with rows twice as long, another converter, and rows padded one by one — 16·UNITS·2 bytes is a
 * multiple of 128, so every row needs its own 16-byte shift to spread the lanes over the bank groups) */
template <int KIND, int UNITS, int WARPS> struct Dft1Plan {
	static constexpr int BPS = KIND == IN_CS16IQ ? 4 : 2;                     /* bytes per complex sample */
	static constexpr int ROWBYTES = UNITS * 8 * BPS;
	static constexpr int RPC = (KIND != IN_CS16IQ && UNITS % 8 == 4) ? 2 : 1; /* rows per bulk copy, see DftPlan */
	static constexpr int GROUP = RPC * ROWBYTES + 16;
	static constexpr int TILE_BYTES = DFT1_ROWS / RPC * GROUP;
	static __device__ __forceinline__ int row_off(int r) { return (r / RPC) * GROUP + (r % RPC) * ROWBYTES; }
	static constexpr int N2 = UNITS * 2;                                      /* K/4: twiddles are stored for the 4-way split */
	static constexpr int TW_BYTES = N2 * CH_GROUP * 8;
	static constexpr int BAR_OFF = WARPS * TILE_BYTES + TW_BYTES;
	static constexpr int SMEM = BAR_OFF + WARPS * 8;
};

/* bytes `KB`, `KB+1` (I, Q of one sample) of word w as (32768 + I, 32768 + Q) */
template <int KB> __device__ __forceinline__ float2 dft1_cvt(unsigned w)
{
	constexpr unsigned si = 0x7404u | (KB << 4), sq = 0x7404u | ((KB + 1) << 4);
	return make_float2(__uint_as_float(__byte_perm(w, 0x47000000u, si)), __uint_as_float(__byte_perm(w, 0x47000000u, sq)));
}
/* CS16: the two 16-bit halves of w (already XORed, see the kernel) planted in the mantissa of 2^23: (2^23 + lo, 2^23 + hi) */
__device__ __forceinline__ float2 dft1_cvt16(unsigned w)
{
	return make_float2(__uint_as_float(__byte_perm(w, 0x4B000000u, 0x7410)), __uint_as_float(__byte_perm(w, 0x4B000000u, 0x7432)));
}

template <int KIND, int UNITS, int WARPS, int MINB, bool PF>
__global__ void __launch_bounds__(32 * WARPS, MINB)
k_channelize_dft1(const uint8_t *__restrict__ in, size_t stream_stride, const float2 *__restrict__ tw,
                  const unsigned *__restrict__ meta, float *__restrict__ dm, int nch, int ngrp, size_t nsamp)
{
	using P = Dft1Plan<KIND, UNITS, WARPS>;
	constexpr int CU = UNITS / 4;                 /* groups of 4 samples per eighth of a row */
	constexpr int N2 = P::N2;
	constexpr int NTILE = OUTBLK / DFT1_ROWS;
	extern __shared__ __align__(16) unsigned char smem[];
	const int l = threadIdx.x & 31;
	const int w = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0);     /* warp-uniform for the compiler too: the bulk-copy operands stay in uniform registers */
	const int blk = blockIdx.x, s = blockIdx.y, g = blockIdx.z;
	unsigned char *mytile = smem + (size_t)w * P::TILE_BYTES;
	const float4 *stw = reinterpret_cast<const float4 *>(smem + (size_t)WARPS * P::TILE_BYTES);   /* [ch][n2] (Tr, Ti) */
	unsigned long long *bar = reinterpret_cast<unsigned long long *>(smem + P::BAR_OFF) + w;
	const uint8_t *src_blk = in + (size_t)s * stream_stride + (size_t)blk * OUTBLK * P::ROWBYTES;
	const unsigned m = __shfl_sync(0xffffffffu, meta[(size_t)s * ngrp + g], 0);    /* (k_c / 2) mod 4 of channel slot c in bits 16 + 2c, 17 + 2c */

	if (l == 0) mbar_init(bar, 1);
	asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
	/* Which Y a channel multiplies is its bin's residue (k_c / 2) mod 4 — warp-uniform, so a branch, not selects.  To
	 * make that branch cheap the CTA works on its channel slots SORTED by residue (a stable counting sort of the eight
	 * 2-bit fields, once per CTA): slot j holds channel perm[j], the twiddles are staged in slot order, the envelope is
	 * stored through perm[], and the MAC section below is four straight-line columns (one per residue) that a warp walks
	 * left to right, moving one column over where the next slot's residue is larger: one compare + branch per slot
	 * instead of a compare-and-branch chain per channel (ncu, chain form: 137 BRA + 97 ISETP per 320 FFMA2). */
	unsigned pw = 0;                             /* perm[j] in bits 3j .. 3j+2 */
	int bnd0, bnd1, bnd2;                        /* first slot whose residue is > 0, > 1, > 2 */
	{
		int cnt[4] = { 0, 0, 0, 0 };
#pragma unroll
		for (int c = 0; c < CH_GROUP; c++) {
			const unsigned r = (m >> (16 + 2 * c)) & 3u;
#pragma unroll
			for (int q = 0; q < 4; q++) cnt[q] += (r == (unsigned)q);
		}
		bnd0 = cnt[0]; bnd1 = bnd0 + cnt[1]; bnd2 = bnd1 + cnt[2];
		int pos[4] = { 0, bnd0, bnd1, bnd2 };
#pragma unroll
		for (int c = 0; c < CH_GROUP; c++) {
			const unsigned r = (m >> (16 + 2 * c)) & 3u;
			int at = 0;
#pragma unroll
			for (int q = 0; q < 4; q++) { at = (r == (unsigned)q) ? pos[q] : at; pos[q] += (r == (unsigned)q); }
			pw |= (unsigned)c << (3 * at);
		}
	}
	{
		const uint4 *tsrc = reinterpret_cast<const uint4 *>(tw + ((size_t)s * ngrp + g) * N2 * CH_GROUP);
		uint4 *tdst = reinterpret_cast<uint4 *>(smem + (size_t)WARPS * P::TILE_BYTES);
		constexpr int PER = N2 * 8 / 16;         /* 16-byte pieces per channel */
		for (int q = threadIdx.x; q < P::TW_BYTES / 16; q += 32 * WARPS) {
			const int j = q / PER, off = q - j * PER;
			cp_async16(tdst + q, tsrc + ((pw >> (3 * j)) & 7u) * PER + off);
		}
		cp_async_commit();
		cp_async_wait_all();
	}
	__syncthreads();

	/* this warp's tiles: w, w + WARPS, ...; the streaming inputs (CS16) may end inside a block: tiles that start past
	 * the last row are not touched, the last one reads up to 31 rows of slack behind the input (context.cu allocates it) */
	const size_t rows_left = nsamp - (size_t)blk * OUTBLK;
	const int tiles_here = rows_left >= (size_t)OUTBLK ? NTILE : (int)((rows_left + DFT1_ROWS - 1) / DFT1_ROWS);
	const int ntile = (tiles_here - w + WARPS - 1) / WARPS;
	auto issue = [&](int n) {
		if (elect_one()) {
			mbar_expect_tx(bar, DFT1_ROWS * P::ROWBYTES);
			const uint8_t *src = src_blk + (size_t)(w + n * WARPS) * DFT1_ROWS * P::ROWBYTES;
#pragma unroll
			for (int i = 0; i < DFT1_ROWS / P::RPC; i++)
				bulk_g2s(mytile + (size_t)i * P::GROUP, src + (size_t)i * P::RPC * P::ROWBYTES, P::RPC * P::ROWBYTES, bar);
		}
	};
	if (ntile > 0) issue(0);
	const int nc = min(CH_GROUP, nch - g * CH_GROUP);

	for (int n = 0; n < ntile; n++) {
		const int tile = w + n * WARPS;
		mbar_wait(bar, (unsigned)(n & 1));
		const unsigned char *ra = mytile + P::row_off(l);
		float2 A[CH_GROUP], B[CH_GROUP];
#pragma unroll
		for (int c = 0; c < CH_GROUP; c++) A[c] = B[c] = make_float2(0.f, 0.f);

#pragma unroll 1
		for (int g4 = 0; g4 < CU; g4++) {
			uint2 e8[8];
			uint4 e16[8];
#pragma unroll
			for (int e = 0; e < 8; e++) {
				if (KIND == IN_CS16IQ) e16[e] = *reinterpret_cast<const uint4 *>(ra + e * (UNITS * 4) + g4 * 16);
				else e8[e] = *reinterpret_cast<const uint2 *>(ra + e * (UNITS * 2) + g4 * 8);
			}
			float2 Y[4][4];                       /* [residue][sample of the group] = (re, im) */
#pragma unroll
			for (int k = 0; k < 4; k++) {
				float2 z[4];
#pragma unroll
				for (int n1 = 0; n1 < 4; n1++) {
					if (KIND == IN_CS16IQ) {
						/* int16 v as the unsigned v + 32768 (XOR 0x8000) in the first half of the row, as 32767 - v (XOR 0x7fff) in
						 * the second: both planted in the mantissa of 2^23, their DIFFERENCE is v0 + v1 + 1, exact (operands in
						 * [2^23, 2^24)) — one XOR per word, two PRMT, one packed subtraction per folded sample */
						const uint4 a = e16[n1], b = e16[n1 + 4];
						const unsigned w0 = (k == 0 ? a.x : k == 1 ? a.y : k == 2 ? a.z : a.w) ^ 0x80008000u;
						const unsigned w1 = (k == 0 ? b.x : k == 1 ? b.y : k == 2 ? b.z : b.w) ^ 0x7fff7fffu;
						z[n1] = fsub2(dft1_cvt16(w0), dft1_cvt16(w1));
					} else {
						const unsigned w0 = k < 2 ? e8[n1].x : e8[n1].y, w1 = k < 2 ? e8[n1 + 4].x : e8[n1 + 4].y;
						z[n1] = (k & 1) ? __fadd2_rn(dft1_cvt<2>(w0), dft1_cvt<2>(w1)) : __fadd2_rn(dft1_cvt<0>(w0), dft1_cvt<0>(w1));
					}
				}
				/* u8: every z carries 2 x 32768 from the converter: sums of four carry 262144 (exact, < 2^24) and Y'_0 also
				 * sheds the converter's mid-scale 8 x 127.5; CS16: every z carries + 1, |z| < 2^17; differences carry nothing */
				const float2 s02 = __fadd2_rn(z[0], z[2]), s13 = __fadd2_rn(z[1], z[3]);
				const float2 d02 = fsub2(z[0], z[2]);
				const float2 wj = make_float2(__fadd_rn(z[1].y, -z[3].y), __fadd_rn(z[3].x, -z[1].x));   /* -j (z1 - z3) */
				const float y0bias = KIND == IN_CS16IQ ? -4.0f : -263164.0f;
				Y[0][k] = __fadd2_rn(__fadd2_rn(s02, s13), make_float2(y0bias, y0bias));
				Y[2][k] = fsub2(s02, s13);
				Y[1][k] = __fadd2_rn(d02, wj);    /* (z0 - z2) - j (z1 - z3) */
				Y[3][k] = fsub2(d02, wj);         /* (z0 - z2) + j (z1 - z3) */
			}
			const float4 *tj = stw + g4 * 2;
			float4 nu0 = make_float4(0.f, 0.f, 0.f, 0.f), nu1 = nu0;
			if (PF) { nu0 = tj[0]; nu1 = tj[1]; }
#define ACB_DFT1_MAC(J, R)                                                                 \
			{                                                                                      \
				const float4 u0 = PF ? nu0 : tj[(J) * (N2 / 2)], u1 = PF ? nu1 : tj[(J) * (N2 / 2) + 1];   \
				/* PF: loaded one slot ahead, whichever column that was */                             \
				if (PF && (J) + 1 < CH_GROUP) { nu0 = tj[((J) + 1) * (N2 / 2)]; nu1 = tj[((J) + 1) * (N2 / 2) + 1]; } \
				const float2 tt[4] = { make_float2(u0.x, u0.y), make_float2(u0.z, u0.w),               \
				                       make_float2(u1.x, u1.y), make_float2(u1.z, u1.w) };             \
				_Pragma("unroll") for (int k = 0; k < 4; k++) {                                        \
					A[J] = ffma2(make_float2(Y[R][k].x, Y[R][k].x), tt[k], A[J]);                          \
					B[J] = ffma2(make_float2(Y[R][k].y, Y[R][k].y), tt[k], B[J]);                          \
				}                                                                                      \
			}
#define ACB_DFT1_C0(J) if ((J) >= bnd0) goto c1_##J; ACB_DFT1_MAC(J, 0)
#define ACB_DFT1_C1(J) c1_##J: if ((J) >= bnd1) goto c2_##J; ACB_DFT1_MAC(J, 1)
#define ACB_DFT1_C2(J) c2_##J: if ((J) >= bnd2) goto c3_##J; ACB_DFT1_MAC(J, 2)
#define ACB_DFT1_C3(J) c3_##J: ACB_DFT1_MAC(J, 3)
#define ACB_DFT1_COL(C) C(0) C(1) C(2) C(3) C(4) C(5) C(6) C(7)
			ACB_DFT1_COL(ACB_DFT1_C0) goto macs_done;
			ACB_DFT1_COL(ACB_DFT1_C1) goto macs_done;
			ACB_DFT1_COL(ACB_DFT1_C2) goto macs_done;
			ACB_DFT1_COL(ACB_DFT1_C3)
			macs_done:;
#undef ACB_DFT1_COL
#undef ACB_DFT1_C3
#undef ACB_DFT1_C2
#undef ACB_DFT1_C1
#undef ACB_DFT1_C0
#undef ACB_DFT1_MAC
		}
		/* every lane has its row in registers: the buffer can take the warp's next tile */
		__syncwarp();
		if (n + 1 < ntile) issue(n + 1);
		float e[CH_GROUP];
#pragma unroll
		for (int c = 0; c < CH_GROUP; c++) {
			const float re = __fadd_rn(A[c].x, -B[c].y), im = __fadd_rn(A[c].y, B[c].x);
			e[c] = __fsqrt_rn(__fmaf_rn(re, re, __fmul_rn(im, im)));
		}
		const size_t mrow = (size_t)blk * OUTBLK + (size_t)tile * DFT1_ROWS + l;
		float *o = dm + ((size_t)s * nsamp + mrow) * nch + g * CH_GROUP;
		/* slot j is channel perm[j]: eight 4-byte stores into the lane's own 32-byte sector */
#pragma unroll
		for (int j = 0; j < CH_GROUP; j++) {
			const int c = (int)((pw >> (3 * j)) & 7u);
			if (c < nc && mrow < nsamp) o[c] = e[j];
		}
	}
}

template <int KIND, int UNITS, int WARPS, int MINB, bool PF>
static int launch_dft1_t(const uint8_t *in, size_t stream_stride, const float2 *tw, const unsigned *meta, float *dm,
                         int nch, int nstreams, int nblk, size_t nsamp, cudaStream_t stream)
{
	const int ngrp = (nch + CH_GROUP - 1) / CH_GROUP;
	constexpr int smem = Dft1Plan<KIND, UNITS, WARPS>::SMEM;
	auto kern = k_channelize_dft1<KIND, UNITS, WARPS, MINB, PF>;
	cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
	if (e != cudaSuccess) return (int)e;
	e = cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
	if (e != cudaSuccess) return (int)e;
	dim3 grid(nblk, nstreams, ngrp);
	kern<<<grid, 32 * WARPS, smem, stream>>>(in, stream_stride, tw, meta, dm, nch, ngrp, nsamp);
	return (int)cudaGetLastError();
}

/* ------------------------------------------------------------------------------------------
 * Fast form of the REAL-input channelizer (air.c:291-341 with the table of air.c:278-285): wf[i] = exp(-j*2*pi*k*i/K)/K is
 * a sampled exponential with k = (Fc - Fr + rate/4) / 12.5 kHz a whole number whenever the channels and the tuner
 * centre sit on the 12.5 kHz raster (air.c:66 puts Fc there), so D is bin k of the K-point DFT of a REAL row:
 *   D = sum_{n2 < K/4} T[n2] * Y_r[n2],  r = k mod 4,  T[n2] = exp(-j*2*pi*k*n2/K)/K,
 *   Y_0 = (x0 + x2) + (x1 + x3)   Y_2 = (x0 + x2) - (x1 + x3)          real
 *   Y_1 = (x0 - x2) - j (x1 - x3) Y_3 = (x0 - x2) + j (x1 - x3)        x_q = x[(K/4) q + n2]
 * 6 additions per n2 shared by all channels, then K/4 real x complex (r even: one FFMA2 per n2) or complex x complex
 * (r odd: two) MACs per channel instead of K: 8 channels cost ~10 FP32 lane-ops per input sample where the reference's
 * order costs 32 — the kernel becomes a memory streamer.  Same shape as k_channelize_dft1: one row per lane, whole rows
 * by cp.async.bulk into a private 32-row tile per warp, channel slots sorted so that the MAC section is straight-line
 * columns (r = 0 | r = 2 | r odd; residues 1 and 3 accumulate the same two sums and differ in one sign at the end).
 * NOT the reference's operation order (tolerance: include/acars_b200.h); bit-identical to oracle's orc_channelize_rdft.
 * ---------------------------------------------------------------------------------------- */
/* LPR lanes share a row: lane l works on row l % ROWS of the warp's tile and takes the h-th contiguous range of n2 pairs,
 * h = l / ROWS; the LPR partial sums are added pairwise (h ^ 1, then h ^ 2, ...) at the end.  A row of K floats is 800 bytes
 * and more: with one lane per row a warp's tile is 26-103 KB, 8 warps or fewer fit an SM and the kernel sits at 29 % issue
 * utilisation waiting for its own dependent FFMA2 chains (ncu, K = 200: 0.93 ms); LPR = K/100 keeps the tile at 13 KB. */
template <int K8, int LPR, int WARPS> struct RdftPlan {
	static constexpr int K = K8 * 8;
	static constexpr int ROWS = 32 / LPR;                             /* rows per warp tile */
	static constexpr int ROWBYTES = K * 4;
	static constexpr int GROUP = ROWBYTES + 16;                       /* every row shifted by one more 16-byte unit */
	static constexpr int TILE_BYTES = ROWS * GROUP;
	static constexpr int N2 = K / 4;
	static constexpr int TW_BYTES = N2 * CH_GROUP * 8;
	static constexpr int BAR_OFF = WARPS * TILE_BYTES + TW_BYTES;
	static constexpr int SMEM = BAR_OFF + WARPS * 8;
	static constexpr int PER = (K8 + LPR - 1) / LPR;                  /* n2 pairs per lane */
};

template <int K8, int LPR, int WARPS, int MINB>
__global__ void __launch_bounds__(32 * WARPS, MINB)
k_channelize_rdft(const uint8_t *__restrict__ in, size_t stream_stride, const float2 *__restrict__ tw,
                  const unsigned *__restrict__ meta, float *__restrict__ dm, int nch, int ngrp, size_t nsamp)
{
	using P = RdftPlan<K8, LPR, WARPS>;
	constexpr int N2 = P::N2, ROWS = P::ROWS;
	constexpr int NTILE = OUTBLK / ROWS;
	extern __shared__ __align__(16) unsigned char smem[];
	const int l = threadIdx.x & 31;
	const int w = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0);
	const int blk = blockIdx.x, s = blockIdx.y, g = blockIdx.z;
	unsigned char *mytile = smem + (size_t)w * P::TILE_BYTES;
	const float4 *stw = reinterpret_cast<const float4 *>(smem + (size_t)WARPS * P::TILE_BYTES);   /* [slot][n2] (Tr, Ti) */
	unsigned long long *bar = reinterpret_cast<unsigned long long *>(smem + P::BAR_OFF) + w;
	const uint8_t *src_blk = in + (size_t)s * stream_stride + (size_t)blk * OUTBLK * P::ROWBYTES;
	const unsigned m = __shfl_sync(0xffffffffu, meta[(size_t)s * ngrp + g], 0);    /* k_c mod 4 of channel c in bits 2c, 2c + 1 */

	if (l == 0) mbar_init(bar, 1);
	asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
	/* slots sorted by column: residue 0, residue 2, odd residues (stable); perm[j] in bits 3j.., sign of slot j in bit j */
	unsigned pw = 0, neg = 0;
	int bnd0, bnd1;
	{
		int cnt[3] = { 0, 0, 0 };
#pragma unroll
		for (int c = 0; c < CH_GROUP; c++) {
			const unsigned r = (m >> (2 * c)) & 3u;
			const int cls = r == 0 ? 0 : r == 2 ? 1 : 2;
#pragma unroll
			for (int q = 0; q < 3; q++) cnt[q] += (cls == q);
		}
		bnd0 = cnt[0]; bnd1 = bnd0 + cnt[1];
		int pos[3] = { 0, bnd0, bnd1 };
#pragma unroll
		for (int c = 0; c < CH_GROUP; c++) {
			const unsigned r = (m >> (2 * c)) & 3u;
			const int cls = r == 0 ? 0 : r == 2 ? 1 : 2;
			int at = 0;
#pragma unroll
			for (int q = 0; q < 3; q++) { at = (cls == q) ? pos[q] : at; pos[q] += (cls == q); }
			pw |= (unsigned)c << (3 * at);
			neg |= (unsigned)(r == 3) << at;
		}
	}
	{
		const uint4 *tsrc = reinterpret_cast<const uint4 *>(tw + ((size_t)s * ngrp + g) * N2 * CH_GROUP);
		uint4 *tdst = reinterpret_cast<uint4 *>(smem + (size_t)WARPS * P::TILE_BYTES);
		constexpr int PER16 = N2 * 8 / 16;
		for (int q = threadIdx.x; q < P::TW_BYTES / 16; q += 32 * WARPS) {
			const int j = q / PER16, off = q - j * PER16;
			cp_async16(tdst + q, tsrc + ((pw >> (3 * j)) & 7u) * PER16 + off);
		}
		cp_async_commit();
		cp_async_wait_all();
	}
	__syncthreads();

	const size_t rows_left = nsamp - (size_t)blk * OUTBLK;
	const int tiles_here = rows_left >= (size_t)OUTBLK ? NTILE : (int)((rows_left + ROWS - 1) / ROWS);
	const int ntile = (tiles_here - w + WARPS - 1) / WARPS;
	auto issue = [&](int n) {
		if (elect_one()) {
			mbar_expect_tx(bar, ROWS * P::ROWBYTES);
			const uint8_t *src = src_blk + (size_t)(w + n * WARPS) * ROWS * P::ROWBYTES;
#pragma unroll
			for (int i = 0; i < ROWS; i++)
				bulk_g2s(mytile + (size_t)i * P::GROUP, src + (size_t)i * P::ROWBYTES, P::ROWBYTES, bar);
		}
	};
	if (ntile > 0) issue(0);
	const int nc = min(CH_GROUP, nch - g * CH_GROUP);
	const int row = l % ROWS, h = l / ROWS;
	const int gp0 = h * P::PER, gp1 = min(K8, gp0 + P::PER);

	for (int n = 0; n < ntile; n++) {
		const int tile = w + n * WARPS;
		mbar_wait(bar, (unsigned)(n & 1));
		const unsigned char *ra = mytile + (size_t)row * P::GROUP;
		float2 A[CH_GROUP], B[CH_GROUP];
#pragma unroll
		for (int c = 0; c < CH_GROUP; c++) A[c] = B[c] = make_float2(0.f, 0.f);

#pragma unroll 1
		for (int gp = gp0; gp < gp1; gp++) {              /* n2 = 2 gp, 2 gp + 1 */
			const float2 x0 = *reinterpret_cast<const float2 *>(ra + 0 * P::K + gp * 8);
			const float2 x1 = *reinterpret_cast<const float2 *>(ra + 1 * P::K + gp * 8);
			const float2 x2 = *reinterpret_cast<const float2 *>(ra + 2 * P::K + gp * 8);
			const float2 x3 = *reinterpret_cast<const float2 *>(ra + 3 * P::K + gp * 8);
			const float2 s02 = __fadd2_rn(x0, x2), s13 = __fadd2_rn(x1, x3);
			const float2 y0 = __fadd2_rn(s02, s13), y2 = fsub2(s02, s13);
			const float2 d02 = fsub2(x0, x2), d13 = fsub2(x1, x3);
			const float4 *tj = stw + gp;
#define ACB_RDFT_E(J, Y)                                                                   \
			{                                                                                      \
				const float4 u = tj[(J) * (N2 / 2)];                                                   \
				A[J] = ffma2(make_float2(Y.x, Y.x), make_float2(u.x, u.y), A[J]);                      \
				A[J] = ffma2(make_float2(Y.y, Y.y), make_float2(u.z, u.w), A[J]);                      \
			}
#define ACB_RDFT_O(J)                                                                      \
			{                                                                                      \
				const float4 u = tj[(J) * (N2 / 2)];                                                   \
				A[J] = ffma2(make_float2(d02.x, d02.x), make_float2(u.x, u.y), A[J]);                  \
				B[J] = ffma2(make_float2(d13.x, d13.x), make_float2(u.x, u.y), B[J]);                  \
				A[J] = ffma2(make_float2(d02.y, d02.y), make_float2(u.z, u.w), A[J]);                  \
				B[J] = ffma2(make_float2(d13.y, d13.y), make_float2(u.z, u.w), B[J]);                  \
			}
#define ACB_RDFT_C0(J) if ((J) >= bnd0) goto r1_##J; ACB_RDFT_E(J, y0)
#define ACB_RDFT_C1(J) r1_##J: if ((J) >= bnd1) goto r2_##J; ACB_RDFT_E(J, y2)
#define ACB_RDFT_C2(J) r2_##J: ACB_RDFT_O(J)
#define ACB_RDFT_COL(C) C(0) C(1) C(2) C(3) C(4) C(5) C(6) C(7)
			ACB_RDFT_COL(ACB_RDFT_C0) goto rmacs_done;
			ACB_RDFT_COL(ACB_RDFT_C1) goto rmacs_done;
			ACB_RDFT_COL(ACB_RDFT_C2)
			rmacs_done:;
#undef ACB_RDFT_COL
#undef ACB_RDFT_C2
#undef ACB_RDFT_C1
#undef ACB_RDFT_C0
#undef ACB_RDFT_O
#undef ACB_RDFT_E
		}
		__syncwarp();
		if (n + 1 < ntile) issue(n + 1);
		/* the row's LPR partial sums, pairwise: (p0 + p1) + (p2 + p3) ... — both partners compute the same sum */
#pragma unroll
		for (int step = ROWS; step < 32; step *= 2) {
#pragma unroll
			for (int j = 0; j < CH_GROUP; j++) {
				A[j].x = __fadd_rn(A[j].x, __shfl_xor_sync(0xffffffffu, A[j].x, step));
				A[j].y = __fadd_rn(A[j].y, __shfl_xor_sync(0xffffffffu, A[j].y, step));
				B[j].x = __fadd_rn(B[j].x, __shfl_xor_sync(0xffffffffu, B[j].x, step));
				B[j].y = __fadd_rn(B[j].y, __shfl_xor_sync(0xffffffffu, B[j].y, step));
			}
		}
		const size_t mrow = (size_t)blk * OUTBLK + (size_t)tile * ROWS + row;
		if (h == 0 && mrow < nsamp) {
			float *o = dm + ((size_t)s * nsamp + mrow) * nch + g * CH_GROUP;
#pragma unroll
			for (int j = 0; j < CH_GROUP; j++) {
				/* r = 1: D = (A.x + B.y) + j (A.y - B.x); r = 3: the other signs; r even: B is zero */
				const float sg = ((neg >> j) & 1u) ? -1.0f : 1.0f;
				const float re = __fadd_rn(A[j].x, __fmul_rn(sg, B[j].y)), im = __fadd_rn(A[j].y, -__fmul_rn(sg, B[j].x));
				const float e = __fsqrt_rn(__fmaf_rn(re, re, __fmul_rn(im, im)));
				const int c = (int)((pw >> (3 * j)) & 7u);
				if (c < nc) o[c] = e;
			}
		}
	}
}

template <int K8, int LPR, int WARPS, int MINB>
static int launch_rdft_t(const uint8_t *in, size_t stream_stride, const float2 *tw, const unsigned *meta, float *dm,
                         int nch, int nstreams, int nblk, size_t nsamp, cudaStream_t stream)
{
	const int ngrp = (nch + CH_GROUP - 1) / CH_GROUP;
	constexpr int smem = RdftPlan<K8, LPR, WARPS>::SMEM;
	auto kern = k_channelize_rdft<K8, LPR, WARPS, MINB>;
	cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
	if (e != cudaSuccess) return (int)e;
	e = cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
	if (e != cudaSuccess) return (int)e;
	dim3 grid(nblk, nstreams, ngrp);
	kern<<<grid, 32 * WARPS, smem, stream>>>(in, stream_stride, tw, meta, dm, nch, ngrp, nsamp);
	return (int)cudaGetLastError();
}

/* the Airspy rates: 2.5 MS/s (K = 200), 3 (240), 5 (400), 6 (480), 10 (800) */
bool channelize_rdft_supports(int K) { return K == 200 || K == 240 || K == 400 || K == 480 || K == 800; }
/* lanes per row of k_channelize_rdft (the CPU restatement needs it: it fixes the order of the partial sums) */
int channelize_rdft_lanes_per_row(int K) { return K >= 800 ? 8 : K >= 400 ? 4 : 2; }

/* float32 real input (air.c), taps == K, every channel on the 12.5 kHz raster around Fc; `nsamp` output rows per stream,
 * any count (the input buffer carries 32 rows of slack).  stream_stride in bytes. */
int launch_channelize_rdft(const void *in, size_t stream_stride, const float *tw, const unsigned *meta, float *dm,
                           int K, int nch, int nstreams, size_t nsamp, cudaStream_t stream)
{
	if (nsamp == 0) return 0;
	const uint8_t *i8 = reinterpret_cast<const uint8_t *>(in);
	const float2 *t4 = reinterpret_cast<const float2 *>(tw);
	const int nblk = (int)((nsamp + OUTBLK - 1) / OUTBLK);
	const int w2 = getenv("ACB_FAST_WARPS") ? atoi(getenv("ACB_FAST_WARPS")) : 4;
#define ACB_RDFT_GO(K8, LPR, W, M) launch_rdft_t<K8, LPR, W, M>(i8, stream_stride, t4, meta, dm, nch, nstreams, nblk, nsamp, stream)
	/* 13-16 KB of tile per warp everywhere; 4 warps per CTA: 16 warps per SM at K = 200, 12 at the other rates */
	if (K == 200) return w2 == 2 ? ACB_RDFT_GO(25, 2, 2, 7) : ACB_RDFT_GO(25, 2, 4, 4);
	if (K == 240) return ACB_RDFT_GO(30, 2, 4, 3);
	if (K == 400) return ACB_RDFT_GO(50, 4, 4, 3);
	if (K == 480) return ACB_RDFT_GO(60, 4, 4, 3);
	if (K == 800) return ACB_RDFT_GO(100, 8, 4, 3);
#undef ACB_RDFT_GO
	return (int)cudaErrorInvalidValue;
}

bool channelize_dft_supports(int K) { return K == 160 || K == 192; }

/* u8 IQ, K in {160, 192} (the reference's two rates), taps == K, every channel on the 12.5 kHz raster
 * around Fc (context.cu checks and builds tw/meta) */
int launch_channelize_dft(const void *in, size_t stream_stride, const float *tw, const unsigned *meta, float *dm,
                          int K, int nch, int nstreams, int nblk, size_t nsamp, bool fold8, cudaStream_t stream)
{
	if (nblk == 0) return 0;
	const uint8_t *i8 = reinterpret_cast<const uint8_t *>(in);
	const float2 *t4 = reinterpret_cast<const float2 *>(tw);
	/* the two-rows-per-lane kernel: 2 warps per CTA, one tile buffer per warp; K=160: 44.5 KB of shared memory and <= 200
	 * registers -> 5 CTAs = 10 warps per SM (measured: 0.97 ms for the 4-way split; 3 or 4 warps per CTA 1.09-1.43 ms; two
	 * buffers per warp with half the warps 1.73 ms) */
	const int minb = getenv("ACB_DFT_MINB") ? atoi(getenv("ACB_DFT_MINB")) : 0;     /* experiment switch: register cap */
	/* default: the folded form with one row per lane, 2 warps per CTA (profiles/r2_dft1b.jsonl: 0.660 ms / 78.7 % of HBM peak at
	 * 592 streams x 16 blocks, 82.9 % at 4736 x 8, against 0.896 ms / 58.0 % for two rows per lane; in the pipeline at 4736
	 * streams 1442-1465 vs 1165 Gsamples/s).  ACB_FAST_ROWS=2 selects the two-row kernel, ACB_FAST_WARPS=4 four warps per CTA,
	 * ACB_FAST_PF=0 twiddle loads in place instead of one slot ahead (no measurable difference): comparison switches, all
	 * bit-identical and tested. */
	const int rows1 = getenv("ACB_FAST_ROWS") ? atoi(getenv("ACB_FAST_ROWS")) : 1;
	if (fold8 && rows1 == 1) {
		const int w2 = getenv("ACB_FAST_WARPS") ? atoi(getenv("ACB_FAST_WARPS")) : 2;
		const bool pf = getenv("ACB_FAST_PF") ? atoi(getenv("ACB_FAST_PF")) != 0 : true;   /* experiment switch: twiddles one slot ahead */
#define ACB_DFT1_GO(U, W, M, F) launch_dft1_t<IN_U8IQ, U, W, M, F>(i8, stream_stride, t4, meta, dm, nch, nstreams, nblk, nsamp, stream)
		if (K == 160) return w2 != 2 ? ACB_DFT1_GO(20, 4, 4, true) : pf ? ACB_DFT1_GO(20, 2, 8, true) : ACB_DFT1_GO(20, 2, 8, false);
		if (K == 192) return w2 != 2 ? ACB_DFT1_GO(24, 4, 4, true) : pf ? ACB_DFT1_GO(24, 2, 8, true) : ACB_DFT1_GO(24, 2, 8, false);
#undef ACB_DFT1_GO
	}
	if (K == 160 && fold8 && minb == 8) return launch_dft_t<20, 2, 1, 8, true>(i8, stream_stride, t4, meta, dm, nch, nstreams, nblk, nsamp, stream);
	if (K == 160 && fold8 && minb == 6) return launch_dft_t<20, 2, 1, 6, true>(i8, stream_stride, t4, meta, dm, nch, nstreams, nblk, nsamp, stream);
	if (K == 160) return fold8 ? launch_dft_t<20, 2, 1, 5, true>(i8, stream_stride, t4, meta, dm, nch, nstreams, nblk, nsamp, stream)
	                           : launch_dft_t<20, 2, 1, 5, false>(i8, stream_stride, t4, meta, dm, nch, nstreams, nblk, nsamp, stream);
	if (K == 192) return fold8 ? launch_dft_t<24, 2, 1, 4, true>(i8, stream_stride, t4, meta, dm, nch, nstreams, nblk, nsamp, stream)
	                           : launch_dft_t<24, 2, 1, 4, false>(i8, stream_stride, t4, meta, dm, nch, nstreams, nblk, nsamp, stream);
	return (int)cudaErrorInvalidValue;
}

/* CS16 IQ (soapy.c / sdrplay.c), same conditions as above; `nsamp` output rows per stream, any count: the last block may be
 * partial (the input buffer carries 32 rows of slack).  stream_stride in bytes. */
int launch_channelize_dft_cs16(const void *in, size_t stream_stride, const float *tw, const unsigned *meta, float *dm,
                               int K, int nch, int nstreams, size_t nsamp, cudaStream_t stream)
{
	if (nsamp == 0) return 0;
	const uint8_t *i8 = reinterpret_cast<const uint8_t *>(in);
	const float2 *t4 = reinterpret_cast<const float2 *>(tw);
	const int nblk = (int)((nsamp + OUTBLK - 1) / OUTBLK);
	/* a warp's tile is 32 rows x (4K + 16) bytes = 20.5 KB at K = 160: 2 warps per CTA -> 5 CTAs = 10 warps per SM */
	const int w2 = getenv("ACB_FAST_WARPS") ? atoi(getenv("ACB_FAST_WARPS")) : 2;
#define ACB_DFT1_GO(U, W, M) launch_dft1_t<IN_CS16IQ, U, W, M, true>(i8, stream_stride, t4, meta, dm, nch, nstreams, nblk, nsamp, stream)
	if (K == 160) return w2 == 1 ? ACB_DFT1_GO(20, 1, 8) : ACB_DFT1_GO(20, 2, 5);
	if (K == 192) return w2 == 1 ? ACB_DFT1_GO(24, 1, 8) : ACB_DFT1_GO(24, 2, 4);
#undef ACB_DFT1_GO
	return (int)cudaErrorInvalidValue;
}

/* SDRplay's stream callback delivers I and Q as separate int16 arrays (sdrplay.c:196-205): out[s][i] = (xi[s][i], xq[s][i])
 * as the interleaved CS16 sample the channelizer reads.  Pure data movement, 8 bytes per sample. */
__global__ void __launch_bounds__(256)
k_interleave_cs16(const int16_t *__restrict__ xi, const int16_t *__restrict__ xq, size_t plane_stride,
                  uint32_t *__restrict__ out, size_t out_stride, size_t nsamples)
{
	const int s = blockIdx.y;
	const uint16_t *pi = reinterpret_cast<const uint16_t *>(xi) + (size_t)s * plane_stride;
	const uint16_t *pq = reinterpret_cast<const uint16_t *>(xq) + (size_t)s * plane_stride;
	uint32_t *o = out + (size_t)s * out_stride;
	for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < nsamples; i += (size_t)gridDim.x * blockDim.x)
		o[i] = (uint32_t)pi[i] | ((uint32_t)pq[i] << 16);
}

int launch_interleave_cs16(const int16_t *xi, const int16_t *xq, size_t plane_stride, uint32_t *out, size_t out_stride,
                           size_t nsamples, int nstreams, cudaStream_t stream)
{
	if (nsamples == 0) return 0;
	const unsigned gx = (unsigned)std::min<size_t>((nsamples + 255) / 256, 1184);
	k_interleave_cs16<<<dim3(gx, nstreams), 256, 0, stream>>>(xi, xq, plane_stride, out, out_stride, nsamples);
	return (int)cudaGetLastError();
}

/* Rows the pipeline kernel does not take (K that breaks 16-byte row alignment; the < 1024 rows
 * left over by a real-input submit of arbitrary length): one thread per (output, channel),
 * straight from global memory, same arithmetic.  Correctness path, not tuned. */
template <int MODE>
__global__ void __launch_bounds__(128)
k_channelize_generic(const uint8_t *__restrict__ in, size_t stream_stride, const uint8_t *__restrict__ wf,
                     float *__restrict__ dm, int K, int taps, int nch, int ngrp, size_t row0, size_t nrows, size_t nsamp)
{
	const size_t gid = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
	const int s = blockIdx.y;
	if (gid >= nrows * nch) return;
	const size_t m = row0 + gid / nch;
	const int ch = (int)(gid % nch);
	float dr = 0.f, di = 0.f;
	const float2 *w = reinterpret_cast<const float2 *>(wf) + ((size_t)s * ngrp + ch / CH_GROUP) * taps * CH_GROUP + (ch % CH_GROUP);
	if (MODE == IN_F32REAL) {
		const float *p = reinterpret_cast<const float *>(in + (size_t)s * stream_stride) + m * K;
		for (int i = 0; i < taps; i++) {
			const float2 ww = w[(size_t)i * CH_GROUP];
			dr = __fadd_rn(dr, __fmul_rn(ww.x, p[i]));
			di = __fadd_rn(di, __fmul_rn(ww.y, p[i]));
		}
	} else if (MODE == IN_CS16IQ) {
		const short *p = reinterpret_cast<const short *>(in + (size_t)s * stream_stride) + m * K * 2;
		for (int ind = 0; ind < taps; ind++) {
			const float a = (float)p[2 * ind], b = (float)p[2 * ind + 1];
			const float2 ww = w[(size_t)ind * CH_GROUP];
			dr = __fadd_rn(dr, __fsub_rn(__fmul_rn(a, ww.x), __fmul_rn(b, ww.y)));
			di = __fadd_rn(di, __fadd_rn(__fmul_rn(a, ww.y), __fmul_rn(b, ww.x)));
		}
	} else {
		const uint8_t *p = in + (size_t)s * stream_stride + m * K * 2;
		for (int ind = 0; ind < taps; ind++) {
			float a = __fadd_rn((float)p[2 * ind], -127.37f), b = __fadd_rn((float)p[2 * ind + 1], -127.37f);
			float2 ww = w[(size_t)ind * CH_GROUP];
			float pr = __fsub_rn(__fmul_rn(a, ww.x), __fmul_rn(b, ww.y));
			float pi = __fadd_rn(__fmul_rn(a, ww.y), __fmul_rn(b, ww.x));
			dr = __fadd_rn(dr, pr);
			di = __fadd_rn(di, pi);
		}
	}
	dm[((size_t)s * nsamp + m) * nch + ch] = envelope(make_float2(dr, di));
}

int launch_channelize_generic(int mode, const void *in, size_t stream_stride, const void *wf, float *dm,
                              int K, int taps, int nch, int nstreams, size_t row0, size_t nrows, size_t nsamp, cudaStream_t stream)
{
	if (nrows == 0) return 0;
	const int ngrp = (nch + CH_GROUP - 1) / CH_GROUP;
	const size_t total = nrows * nch;
	dim3 grid((unsigned)((total + 127) / 128), nstreams);
	const uint8_t *i8 = (const uint8_t *)in, *w8 = (const uint8_t *)wf;
	if (mode == IN_F32REAL) k_channelize_generic<IN_F32REAL><<<grid, 128, 0, stream>>>(i8, stream_stride, w8, dm, K, taps, nch, ngrp, row0, nrows, nsamp);
	else if (mode == IN_CS16IQ) k_channelize_generic<IN_CS16IQ><<<grid, 128, 0, stream>>>(i8, stream_stride, w8, dm, K, taps, nch, ngrp, row0, nrows, nsamp);
	else k_channelize_generic<IN_U8IQ><<<grid, 128, 0, stream>>>(i8, stream_stride, w8, dm, K, taps, nch, ngrp, row0, nrows, nsamp);
	return (int)cudaGetLastError();
}

/* ------------------------------------------------------------------------------------------
 * K2: MSK demodulator + bit/byte framing, one channel per lane
 *
 * The recurrence is serial per channel (VCO phase -> ring -> matched filter -> PLL -> VCO step,
 * with the frame synchroniser resetting the PLL), so the kernel is latency bound; what it can
 * do is (a) never diverge: every lane runs "up to 6 samples, then one bit" per outer iteration
 * (the bit clock fires every 5.2 samples), (b) expose the 6 independent sincos evaluations of an
 * iteration to the scheduler at once, (c) use a branch-free table sincos (20 FP64 ops) instead
 * of the library one (~45 + slow path), (d) prefetch the 6 envelope samples.
 * ---------------------------------------------------------------------------------------- */

/* acars.c:350-366: queue the finished block.  lvl = 10*log10(lvlsum/bitcount) is left to the host
 * (glibc log10) so the float matches the reference bit for bit.  Out of line and by value: it
 * runs once per frame, and keeping it away from the loop keeps the loop's state in registers. */
static __device__ __noinline__ void emit_frame(const ChainState *st, RawFrame *ring, RingCtl *ctl, unsigned cap,
                                               int stream, int chn, int len, int err, double lvlsum, int bitcount,
                                               unsigned long long pos, unsigned long long soh_pos)
{
	/* blk_thread drops blocks shorter than 13 bytes unseen (acars.c:124-129): they never take a slot, so a
	 * ring sized for the shortest deliverable frame (19 bytes on air = 792 samples) cannot be overrun by a
	 * transmitter sending degenerate frames; the host adds the count to raw_frames / fec_dropped */
	if (len < 13) { atomicAdd(&ctl->short_frames, 1u); return; }
	const unsigned slot = atomicAdd(&ctl->count, 1u);
	if (slot >= cap) return;                       /* overflow: counted by the host (frames_lost), decoding goes on */
	RawFrame *f = ring + slot;
	f->stream = stream; f->chn = chn;
	f->len = len; f->err = err;
	f->lvlsum = lvlsum; f->bitcount = bitcount; f->pad0 = 0;          /* pad0: FEC status, set by k_block_fec */
	f->pos = pos; f->soh_pos = soh_pos;
	f->crc[0] = st->crc[0]; f->crc[1] = st->crc[1];
	for (int i = 0; i < 6; i++) f->pad1[i] = 0;            /* the record goes to the host as a whole */
	const uint2 *src = reinterpret_cast<const uint2 *>(st->txt);
	uint2 *dst = reinterpret_cast<uint2 *>(f->txt);
	for (int i = 0; i < TXTCAP / 8; i++) dst[i] = src[i];
}

/* accessor for frame_sm.h: state in registers, text in the chain's HBM record */
struct DevFrameAcc {
	DemodRegs &r;
	ChainState *st;
	RawFrame *ring;
	RingCtl *ctl;
	unsigned cap;
	int stream, chn;
	bool leader;             /* the lane of the channel's group that owns the HBM side effects */

	__device__ __forceinline__ int &state() { return r.state; }
	__device__ __forceinline__ int &nbits() { return r.nbits; }
	__device__ __forceinline__ int &bitcount() { return r.bitcount; }
	__device__ __forceinline__ int &blk_len() { return r.blk_len; }
	__device__ __forceinline__ int &blk_err() { return r.blk_err; }
	__device__ __forceinline__ unsigned &msk_s() { return r.S; }
	__device__ __forceinline__ double &msk_df() { return r.df; }
	__device__ __forceinline__ double &lvlsum() { return r.lvlsum; }
	__device__ __forceinline__ void txt_put(int i, unsigned char c) { if (leader) st->txt[i] = c; }
	/* only the leader's value is ever stored (crc_put); the shadows' reads are don't-cares */
	__device__ __forceinline__ unsigned char txt_get(int i) { return leader ? st->txt[i] : (unsigned char)0; }
	__device__ __forceinline__ void crc_put(int i, unsigned char c) { if (leader) st->crc[i] = c; }
	bool v2;                 /* demod_core.h's loop: the bit's sample position is pos0 + fire_n (r.pos is only set at the end) */
	__device__ __forceinline__ unsigned long long bit_pos() const { return v2 ? r.pos0 + (unsigned long long)(long long)r.fire_n : r.pos; }
	__device__ __forceinline__ bool frame_begin() { r.soh_pos = bit_pos(); return true; }   /* acars.c:283-292 */
	__device__ __forceinline__ void frame_emit()
	{
		if (leader) emit_frame(st, ring, ctl, cap, stream, chn, r.blk_len, r.blk_err, r.lvlsum, r.bitcount, bit_pos(), r.soh_pos);
	}
};

/* cos/sin of k*pi/32 as double-double (hi, lo), built on the host in long double */
__device__ double2 g_sc_cos[64], g_sc_sin[64];

int upload_sincos_table(const double *cos_hi_lo, const double *sin_hi_lo, cudaStream_t stream)
{
	cudaError_t e = cudaMemcpyToSymbolAsync(g_sc_cos, cos_hi_lo, sizeof(double) * 128, 0, cudaMemcpyHostToDevice, stream);
	if (e != cudaSuccess) return (int)e;
	e = cudaMemcpyToSymbolAsync(g_sc_sin, sin_hi_lo, sizeof(double) * 128, 0, cudaMemcpyHostToDevice, stream);
	if (e != cudaSuccess) return (int)e;
	return (int)cudaStreamSynchronize(stream);      /* the sources are the caller's stack arrays */
}

/* cos(p), sin(p) for p in [0, 2*pi] — the VCO phase after msk.c:82-83.  p = k*pi/32 + r with
 * |r| <= pi/64 (three-part pi/32, so r keeps full relative accuracy next to the zeros of sin and
 * cos, which are table points with exact entries); short Taylor polynomials for sin r and
 * cos r - 1; angle addition against the double-double table.  Max error measured against 80-bit
 * references: 1.7 ulp (typ. < 0.6), i.e. the class of CUDA's own sincos; see DESIGN.md for why
 * ~1 ulp here is invisible after the (float) rounding of in*cexp(-j p) (msk.c:90). */
constexpr double SC_MAGIC = 6755399441055744.0;     /* 1.5 * 2^52 */
__device__ __forceinline__ void sincos_vco(double p, const double2 *tcos, const double2 *tsin, double &sn, double &cs)
{
	const double t = fma(p, 0x1.45f306dc9c883p+3, SC_MAGIC);               /* p * 32/pi, rounded to integer */
	const int k = __double2loint(t) & 63;
	const double kd = t - SC_MAGIC;
	double r = fma(-kd, 0x1.921fb54442d18p-4, p);
	r = fma(-kd, 0x1.1a62633145c07p-58, r);
	r = fma(-kd, -0x1.f1976b7ed8fbcp-114, r);
	const double r2 = r * r;
	double sp = fma(r2, (1.0 / 362880), (-1.0 / 5040));
	sp = fma(sp, r2, (1.0 / 120));
	sp = fma(sp, r2, (-1.0 / 6));
	const double sr = fma(r * r2, sp, r);                    /* sin r */
	double cp = fma(r2, (1.0 / 40320), (-1.0 / 720));
	cp = fma(cp, r2, (1.0 / 24));
	cp = fma(cp, r2, (-0.5));
	const double cm = r2 * cp;                               /* cos r - 1 */
	const double2 C = tcos[k], S = tsin[k];
	cs = C.x + fma(-S.x, sr, fma(C.x, cm, C.y));
	sn = S.x + fma(C.x, sr, fma(S.x, cm, S.y));
}

/* lanes per channel: 4 (8 channels per warp), or 8 (4 channels per warp, one mixer evaluation per lane
 * instead of two) for contexts small enough that the doubled warp count still fits one warp per SM
 * sub-partition (context.cu decides) */

/* One warp = 8 channels of one stream x 4 lanes per channel.  The 4 lanes of a channel run the
 * SAME recurrence on the same inputs (identical registers, no communication needed) except for
 * the mixer: lane `sub` evaluates in*cexp(-j phi) for candidate samples sub and 4+sub and drops
 * the result into the channel's ring in shared memory.  SIMT lanes are the one way to get the
 * independent sincos evaluations of a bit period executed side by side: as straight-line code of
 * one lane, ptxas schedules them back to back (6 x 16 dependent FP64 ops x 8 cycles).  Only the
 * group leader touches HBM state (frame text, frame ring, state write-back). */
template <int DEMOD_GROUP>
__global__ void __launch_bounds__(32)
k_demod(ChainState *__restrict__ states, const float *__restrict__ dm, int nsamp, int nch, int nstreams,
        int wps, RawFrame *__restrict__ ring, RingCtl *__restrict__ ctl, unsigned cap)
{
	constexpr int DEMOD_CPW = 32 / DEMOD_GROUP;      /* channels per warp */
	__shared__ float s_h[FLENO + 3];
	/* rows FLEN.. : one scratch row per lane of the group, for mixer outputs past the bit instant */
	__shared__ float s_re[FLEN + DEMOD_GROUP][DEMOD_CPW], s_im[FLEN + DEMOD_GROUP][DEMOD_CPW];
	__shared__ double2 s_cos[64], s_sin[64];

	for (int i = threadIdx.x; i < FLENO; i += 32) s_h[i] = c_h[i];
	for (int i = threadIdx.x; i < 64; i += 32) { s_cos[i] = g_sc_cos[i]; s_sin[i] = g_sc_sin[i]; }

	const int lane = threadIdx.x;
	const int grp = lane / DEMOD_GROUP, sub = lane % DEMOD_GROUP;
	const int warp = blockIdx.x;
	const int s = warp / wps;
	const int ch_raw = (warp - s * wps) * DEMOD_CPW + grp;
	const bool valid = ch_raw < nch;                 /* surplus groups shadow the last channel, silently */
	const int ch = valid ? ch_raw : nch - 1;
	const bool leader = valid && sub == 0;

	ChainState *st = states + (size_t)s * nch + ch;
	DemodRegs r;
	r.phi = st->phi; r.df = st->df; r.lvlsum = st->lvlsum; r.clk = st->clk; r.bitcount = st->bitcount;
	r.S = st->S; r.idx = st->idx; r.nbits = st->nbits; r.state = st->state; r.outbits = st->outbits;
	r.blk_len = st->blk_len; r.blk_err = st->blk_err; r.pos = st->pos; r.soh_pos = st->soh_pos;
	for (int k = sub; k < FLEN; k += DEMOD_GROUP) { s_re[k][grp] = st->inb_re[k]; s_im[k][grp] = st->inb_im[k]; }
	__syncwarp();

	DevFrameAcc acc{ r, st, ring, ctl, cap, s, ch, leader, false };

	const double TWO_PI = 2.0 * M_PI;
	const double S0 = 1800.0 / 12500 * 2.0 * M_PI;             /* msk.c:81 */
	const double THR = 3 * M_PI / 2.0;                         /* msk.c:96,100 */
	const double INV_S0 = 1.0 / (1800.0 / 12500 * 2.0 * M_PI);
	const double PLLC = (double)0.52f;                         /* msk.c:66 (float constant) */
	const double PLLK = (1.0 - (double)0.52f) * (double)38e-4f;/* msk.c:130 (1.0-PLLC)*PLLG */

	const float *in = dm + (size_t)s * nsamp * nch + ch;
	const unsigned long long pos0 = r.pos;
	double clkd = (double)r.clk;             /* MskClk: a float value carried in a double register */
	/* which of the six candidate phases this lane mixes: 4 lanes -> samples sub and 4 + sub (the latter
	 * only for sub < 2; lanes 2, 3 get phase 4 or 5 for their discarded second evaluation, as before);
	 * 8 lanes -> sample sub (lanes 6, 7 idle on phase 5) */
	long long pick[DEMOD_LOOK];
#pragma unroll
	for (int k = 0; k < DEMOD_LOOK; k++) {
		bool mine;
		if (DEMOD_GROUP == 4) mine = k < 4 ? (sub == k) : ((sub & 1) == (k - 4));
		else mine = k < DEMOD_LOOK - 1 ? (sub == k) : (sub >= k);
		pick[k] = mine ? -1LL : 0LL;
	}
	int n = 0;
	/* channels of a warp consume 5 or 6 samples per iteration each, so they finish a few
	 * iterations apart: finished groups idle through empty iterations (m = 0) */
	while (__any_sync(0xffffffffu, n < nsamp)) {
		const int m = max(0, min(DEMOD_LOOK, nsamp - n));
		/* this lane's two candidate samples */
		const int k1 = sub, k2 = DEMOD_GROUP + sub;
		const float x1 = in[(size_t)min(n + k1, nsamp - 1) * nch];
		const float x2 = DEMOD_GROUP == 4 ? in[(size_t)min(n + k2, nsamp - 1) * nch] : 0.f;
		if (n + 2 * DEMOD_LOOK < nsamp) asm volatile("prefetch.global.L1 [%0];" ::"l"(in + (size_t)(n + 2 * DEMOD_LOOK) * nch));

		/* VCO step is constant until the next bit (msk.c:81): MskDf only changes in the bit path */
		const double sv = __dadd_rn(S0, r.df);
		const double fire_at = __dadd_rn(THR, -__dmul_rn(sv, 0.5));
		/* 1/sv for the phase-index fast path below: three Newton steps from 1/S0 (|sv/S0 - 1| < 2e-2),
		 * off the critical path */
		double inv_s = INV_S0;
		inv_s = fma(inv_s, fma(-sv, inv_s, 1.0), inv_s);
		inv_s = fma(inv_s, fma(-sv, inv_s, 1.0), inv_s);
		inv_s = fma(inv_s, fma(-sv, inv_s, 1.0), inv_s);

		/* the two cheap serial chains of the next samples: phase (msk.c:82-83) and bit clock
		 * (msk.c:95-96), each rounded step by step exactly like the reference's loop; straight-line
		 * code (selects, no branches) */
		double pk[DEMOD_LOOK], ck[DEMOD_LOOK];
		{
			double p = r.phi, c = clkd;
#pragma unroll
			for (int k = 0; k < DEMOD_LOOK; k++) {
				p = __dadd_rn(p, sv);
				p = (p >= TWO_PI) ? __dadd_rn(p, -TWO_PI) : p;
				c = round_to_f32<false>(__dadd_rn(c, sv));
				pk[k] = p;
				ck[k] = c;
			}
		}
		/* first of the m available samples at which the clock fires (msk.c:96), if any; the state
		 * after `cnt` samples is picked with bit masks (a select chain on the index would be
		 * turned into a local-memory array by the compiler) */
		int cnt = m;                 /* samples consumed this iteration */
		bool fired = false;
#pragma unroll
		for (int k = DEMOD_LOOK - 1; k >= 0; k--) {
			const bool f = (k < m) & (ck[k] >= fire_at);
			cnt = f ? k + 1 : cnt;
			fired = fired | f;
		}
		double p;
		{
			long long pb = (cnt == 0) ? __double_as_longlong(r.phi) : 0, cb = (cnt == 0) ? __double_as_longlong(clkd) : 0;
#pragma unroll
			for (int k = 0; k < DEMOD_LOOK; k++) {
				const long long mk = -(long long)(cnt == k + 1);
				pb |= __double_as_longlong(pk[k]) & mk;
				cb |= __double_as_longlong(ck[k]) & mk;
			}
			p = __longlong_as_double(pb);
			clkd = __longlong_as_double(cb);
		}
		/* mixer (msk.c:86-91): in * cexp(-j phi), this lane's share */
		if (DEMOD_GROUP == 4) {
			/* lane-dependent picks as mask selects: written as a ?: chain on `sub` the compiler branches,
			 * and the lanes of a group then run the arms one after the other */
			const double p1 = __longlong_as_double((__double_as_longlong(pk[0]) & pick[0]) | (__double_as_longlong(pk[1]) & pick[1]) |
			                                       (__double_as_longlong(pk[2]) & pick[2]) | (__double_as_longlong(pk[3]) & pick[3]));
			const double p2 = __longlong_as_double((__double_as_longlong(pk[4]) & pick[4]) | (__double_as_longlong(pk[5]) & pick[5]));
			double sn1, cs1, sn2, cs2;
			sincos_vco(p1, s_cos, s_sin, sn1, cs1);
			sincos_vco(p2, s_cos, s_sin, sn2, cs2);
			const double xd1 = (double)x1, xd2 = (double)x2;
			const float re1 = __double2float_rn(__dmul_rn(xd1, cs1)), im1 = __double2float_rn(__dmul_rn(xd1, -sn1));
			const float re2 = __double2float_rn(__dmul_rn(xd2, cs2)), im2 = __double2float_rn(__dmul_rn(xd2, -sn2));
			unsigned row1 = r.idx + k1, row2 = r.idx + k2;
			row1 = (row1 >= FLEN) ? row1 - FLEN : row1;
			row2 = (row2 >= FLEN) ? row2 - FLEN : row2;
			row1 = (k1 < cnt) ? row1 : FLEN + sub;                 /* past the bit instant: scratch row */
			row2 = (k2 < cnt && k2 < DEMOD_LOOK) ? row2 : FLEN + sub;
			__syncwarp();          /* the previous bit's matched filter has read the rows being replaced */
			s_re[row1][grp] = re1; s_im[row1][grp] = im1;
			s_re[row2][grp] = re2; s_im[row2][grp] = im2;
			__syncwarp();
		} else {                   /* one candidate sample per lane (lanes 6, 7 of the group idle here) */
			const double p1 = __longlong_as_double((__double_as_longlong(pk[0]) & pick[0]) | (__double_as_longlong(pk[1]) & pick[1]) |
			                                       (__double_as_longlong(pk[2]) & pick[2]) | (__double_as_longlong(pk[3]) & pick[3]) |
			                                       (__double_as_longlong(pk[4]) & pick[4]) | (__double_as_longlong(pk[5]) & pick[5]));
			double sn1, cs1;
			sincos_vco(p1, s_cos, s_sin, sn1, cs1);
			const double xd1 = (double)x1;
			const float re1 = __double2float_rn(__dmul_rn(xd1, cs1)), im1 = __double2float_rn(__dmul_rn(xd1, -sn1));
			unsigned row1 = r.idx + k1;
			row1 = (row1 >= FLEN) ? row1 - FLEN : row1;
			row1 = (k1 < cnt && k1 < DEMOD_LOOK) ? row1 : FLEN + sub;
			__syncwarp();
			s_re[row1][grp] = re1; s_im[row1][grp] = im1;
			__syncwarp();
		}
		r.idx = (r.idx + cnt) % FLEN;
		r.phi = p;
		r.pos = pos0 + (unsigned long long)(n + cnt - 1);       /* the sample that fired the bit */

		if (fired) {
			clkd = round_to_f32<false>(__dadd_rn(clkd, -THR));

			/* matched filter (msk.c:103-107): 11 taps out of the x12 oversampled half cosine.
			 * Phase index o = (int)(12*(MskClk/s + 0.5)): with inv_s good to 1e-15 the product gives
			 * the value to ~1e-14; only when that lands within 1e-9 of an integer (where the
			 * truncation could differ) is the reference's exact division sequence replayed. */
			double u = fma(__dmul_rn(clkd, inv_s), 12.0, 6.0);
			if (fabs(u - rint(u)) < 1e-9) u = __dmul_rn(12.0, __dadd_rn(__ddiv_rn(clkd, sv), 0.5));
			int o = __double2int_rz(u);
			o = min(max(o, 0), MFLTOVER);
			float vr = 0.f, vi = 0.f;
			const float *hp = s_h + o;
			int kk = r.idx;
#pragma unroll
			for (int j = 0; j < FLEN; j++) {
				const float hh = hp[MFLTOVER * j];
				vr = __fadd_rn(vr, __fmul_rn(hh, s_re[kk][grp]));
				vi = __fadd_rn(vi, __fmul_rn(hh, s_im[kk][grp]));
				kk = (kk + 1 == FLEN) ? 0 : kk + 1;
			}
			/* normalise (msk.c:110-113) */
			const float lvl = envelope(make_float2(vr, vi));
			const double d = __dadd_rn((double)lvl, 1e-8);
			vr = __double2float_rn(__ddiv_rn((double)vr, d));
			vi = __double2float_rn(__ddiv_rn((double)vi, d));
			r.lvlsum = __dadd_rn(r.lvlsum, (double)__fmul_rn(__fmul_rn(lvl, lvl), 0.25f));
			r.bitcount++;

			/* decision + phase error (msk.c:115-127) */
			float vo;
			double dphi;
			if (r.S & 1u) { vo = vi; dphi = (vo >= 0.f) ? (double)(-vr) : (double)vr; }
			else          { vo = vr; dphi = (vo >= 0.f) ? (double)vi : (double)(-vi); }
			const float bitv = (r.S & 2u) ? -vo : vo;

			/* putbit (msk.c:53-63) */
			r.outbits >>= 1;
			if (bitv > 0.f) r.outbits |= 0x80u;
			if (--r.nbits <= 0) frame_byte(acc, (unsigned char)r.outbits);
			r.S++;

			/* PLL filter (msk.c:130) — after putbit, so a frame resync's MskDf=0 is filtered too */
			r.df = __dadd_rn(__dmul_rn(PLLC, r.df), __dmul_rn(PLLK, dphi));
		}
		n += cnt;
	}
	if (!leader) return;
	r.pos = pos0 + (unsigned long long)nsamp;
	r.clk = (float)clkd;

	st->phi = r.phi; st->df = r.df; st->lvlsum = r.lvlsum; st->clk = r.clk; st->bitcount = r.bitcount;
	st->S = r.S; st->idx = r.idx; st->nbits = r.nbits; st->state = r.state; st->outbits = r.outbits;
	st->blk_len = r.blk_len; st->blk_err = r.blk_err; st->pos = r.pos; st->soh_pos = r.soh_pos;
#pragma unroll
	for (int k = 0; k < FLEN; k++) { st->inb_re[k] = s_re[k][grp]; st->inb_im[k] = s_im[k][grp]; }
}

/* K2, current form: the loop lives in demod_core.h (shared with the CPU tests' single-lane emulation).
 * One warp per CTA so chains spread over all SMs; L lanes per channel, 32/L channels per warp; state in
 * registers across the whole launch, ring and tables in shared memory, state written back at the end
 * (channel_t's role between demodMSK calls, msk.c:71-72, 134-135). */
struct WarpEnv {
	static __device__ __forceinline__ bool any(bool x) { return __any_sync(0xffffffffu, x) != 0; }
	static __device__ __forceinline__ bool all(bool x) { return __all_sync(0xffffffffu, x) != 0; }
	static __device__ __forceinline__ void sync() { __syncwarp(); }
	static __device__ __forceinline__ int max(int x) { return __reduce_max_sync(0xffffffffu, x); }
};

__device__ DcF4 g_h2[MFLTOVER + 1][3];           /* matched filter, transposed: g_h2[o] = h[o + 12 j] (msk.c:104-107) */

int upload_matched_filter(const float *h, cudaStream_t stream)
{
	float t[MFLTOVER + 1][12];
	for (int o = 0; o <= MFLTOVER; o++)
		for (int j = 0; j < 12; j++) t[o][j] = j < FLEN ? h[o + MFLTOVER * j] : 0.f;
	cudaError_t e = cudaMemcpyToSymbolAsync(c_h, h, sizeof(float) * FLENO, 0, cudaMemcpyHostToDevice, stream);
	if (e != cudaSuccess) return (int)e;
	e = cudaMemcpyToSymbolAsync(g_h2, t, sizeof(t), 0, cudaMemcpyHostToDevice, stream);
	if (e != cudaSuccess) return (int)e;
	return (int)cudaStreamSynchronize(stream);
}

template <int L, bool F2F, bool PIN, int MINB = 1>     /* MINB = 0: no occupancy request */
__global__ void __launch_bounds__(32, MINB)
k_demod2(ChainState *__restrict__ states, const float *__restrict__ dm, int nsamp, int nch, int nstreams,
         int wps, RawFrame *__restrict__ ring, RingCtl *__restrict__ ctl, unsigned cap)
{
	constexpr int CPW = 32 / L;                  /* channels per warp */
	__shared__ DemodShared<CPW> sm;
	const int lane = threadIdx.x;
	for (int i = lane; i < 64; i += 32) {
		sm.tcos[i].x = g_sc_cos[i].x; sm.tcos[i].y = g_sc_cos[i].y;
		sm.tsin[i].x = g_sc_sin[i].x; sm.tsin[i].y = g_sc_sin[i].y;
	}
	for (int i = lane; i < (MFLTOVER + 1) * 3; i += 32) (&sm.h2[0][0])[i] = (&g_h2[0][0])[i];

	const int grp = lane / L, sub = lane % L;
	/* chains (stream, channel) are numbered stream-major and dealt CPW to a warp, across stream boundaries: a
	 * warp of 32 single-lane chains serves four 8-channel streams */
	const long long nchain = (long long)nstreams * nch;
	const long long g_raw = (long long)blockIdx.x * CPW + grp;
	const bool valid = g_raw < nchain;               /* surplus groups of the last warp shadow the last chain, silently */
	const long long g = valid ? g_raw : nchain - 1;
	const int s = (int)(g / nch), ch = (int)(g - (long long)s * nch);
	const bool leader = valid && sub == 0;
	(void)wps;

	ChainState *st = states + (size_t)s * nch + ch;
	DemodRegs r;
	r.phi = st->phi; r.df = st->df; r.lvlsum = st->lvlsum; r.clk = st->clk; r.bitcount = st->bitcount;
	r.S = st->S; r.idx = st->idx; r.nbits = st->nbits; r.state = st->state; r.outbits = st->outbits;
	r.blk_len = st->blk_len; r.blk_err = st->blk_err; r.pos = st->pos; r.soh_pos = st->soh_pos;
	for (int k = sub; k < FLEN; k += L) {
		DcF2 v;
		v.x = st->inb_re[k]; v.y = st->inb_im[k];
		sm.ring[k][grp] = v;
		sm.ring[k + FLEN][grp] = v;
	}
	__syncwarp();

	DevFrameAcc acc{ r, st, ring, ctl, cap, s, ch, leader, true };
	demod_run<L, F2F, PIN, WarpEnv>(r, sm, dm + (size_t)s * nsamp * nch + ch, nch, nsamp, sub, grp, acc);

	if (!leader) return;
	st->phi = r.phi; st->df = r.df; st->lvlsum = r.lvlsum; st->clk = r.clk; st->bitcount = r.bitcount;
	st->S = r.S; st->idx = r.idx; st->nbits = r.nbits; st->state = r.state; st->outbits = r.outbits;
	st->blk_len = r.blk_len; st->blk_err = r.blk_err; st->pos = r.pos; st->soh_pos = r.soh_pos;
#pragma unroll
	for (int k = 0; k < FLEN; k++) { st->inb_re[k] = sm.ring[k][grp].x; st->inb_im[k] = sm.ring[k][grp].y; }
}

template <int LANES, bool F2F, bool PIN, int MINB = 1>
static int launch_demod_t(ChainState *st, const float *dm, int nsamp, int nch, int nstreams,
                          RawFrame *ring, RingCtl *ctl, unsigned cap, cudaStream_t stream)
{
	constexpr int CPW = 32 / LANES;
	const int wps = (nch + CPW - 1) / CPW;
	const long long nchain = (long long)nstreams * nch;
	const int grid = (int)((nchain + CPW - 1) / CPW);    /* one warp per CTA so that chains spread over all SMs */
	cudaError_t e = cudaFuncSetAttribute(k_demod2<LANES, F2F, PIN, MINB>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
	if (e != cudaSuccess) return (int)e;
	k_demod2<LANES, F2F, PIN, MINB><<<grid, 32, 0, stream>>>(st, dm, nsamp, nch, nstreams, wps, ring, ctl, cap);
	return (int)cudaGetLastError();
}

/* The pinned forms (2, 4, 8 lanes) in two register budgets.  Told that one CTA per SM is all it asks for
 * (__launch_bounds__(32, 1)), ptxas spends 144 instead of 124 registers on a wider schedule: 1.4 % fewer instructions and 9 %
 * less time where the kernel is latency bound (592 streams, 4 lanes: 2.75 -> 2.51 ms under ncu) — and two warps per SM fewer
 * where it is not (2368 streams forced to 4 lanes: 16 -> 14 warps per SM, 4.31 -> 5.76 ms).  So: the wide schedule while
 * there are at most 8 warps per SM, the lean one beyond. */
template <int LANES, bool F2F>
static int launch_demod_pinned(ChainState *st, const float *dm, int nsamp, int nch, int nstreams,
                               RawFrame *ring, RingCtl *ctl, unsigned cap, cudaStream_t stream)
{
	int dev = 0, sm_count = 0;               /* asked per launch: contexts of one process may sit on different devices */
	if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&sm_count, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || sm_count <= 0)
		sm_count = 148;
	const long long warps = ((long long)nstreams * nch * LANES + 31) / 32;
	return warps <= 8LL * sm_count ? launch_demod_t<LANES, F2F, true, 1>(st, dm, nsamp, nch, nstreams, ring, ctl, cap, stream)
	                               : launch_demod_t<LANES, F2F, true, 0>(st, dm, nsamp, nch, nstreams, ring, ctl, cap, stream);
}

template <int LANES>
static int launch_demod_v1(ChainState *st, const float *dm, int nsamp, int nch, int nstreams,
                           RawFrame *ring, RingCtl *ctl, unsigned cap, cudaStream_t stream)
{
	constexpr int CPW = 32 / LANES;
	const int wps = (nch + CPW - 1) / CPW;
	cudaError_t e = cudaFuncSetAttribute(k_demod<LANES>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
	if (e != cudaSuccess) return (int)e;
	k_demod<LANES><<<nstreams * wps, 32, 0, stream>>>(st, dm, nsamp, nch, nstreams, wps, ring, ctl, cap);
	return (int)cudaGetLastError();
}

/* Lanes per channel.  Every lane of a channel's group repeats the serial part of a bit period and the group
 * only splits the six mixer evaluations, so fewer lanes = fewer instructions per channel; more lanes = a
 * shorter chain per bit.  The kernel is latency bound until there are several warps per scheduler, so: the
 * most lanes that still leave about one warp per SM sub-partition, the fewest once the chains alone fill
 * the machine. */
int demod_pick_lanes(long long nchains, int sm_count)
{
	/* measured on B200 (profiles/r2_ab_demod.jsonl, 8 channels per stream): 592 streams: 8 or 4 lanes (2.9 ms per 16
	 * blocks), 1 lane 4.0 ms; 2368 streams: 1 lane 4.1 ms, 4 lanes 4.5 ms, 8 lanes 7.7 ms; 4736 x 8 blocks: 1 lane 2.4 ms,
	 * 4 lanes 4.4 ms: the fewest lanes that still put a warp on every scheduler */
	const long long slots = 4LL * sm_count;      /* one warp per scheduler */
	for (int lanes = 1; lanes < 8; lanes *= 2)
		if (nchains * lanes >= 32 * slots) return lanes;
	return 8;
}

/* lanes: 1, 2, 4 or 8 lanes per channel, each in its measured-best form (profiles/r2_ab_demod_pinning.jsonl): loop
 * constants pinned in registers for 2, 4, 8 lanes (592 streams, 4 lanes: 2.75 vs 3.08 ms), not pinned for 1 lane (4736
 * streams: 2.18 vs 2.30 ms alone, and the pipelined step is no slower); + 32 = the other choice; + 16 = bit clock rounded
 * with the F2F conversion pair instead of integer ops (round_to_f32); negative (-4, -8) = the round-1 kernel, kept for
 * A/B runs */
int launch_demod(ChainState *st, const float *dm, int nsamp, int nch, int nstreams,
                 RawFrame *ring, RingCtl *ctl, unsigned cap, int lanes, cudaStream_t stream)
{
#define ACB_DEMOD_ARGS st, dm, nsamp, nch, nstreams, ring, ctl, cap, stream
	switch (lanes) {
	case -8: return launch_demod_v1<8>(ACB_DEMOD_ARGS);
	case -4: return launch_demod_v1<4>(ACB_DEMOD_ARGS);
	case 8: return launch_demod_pinned<8, false>(ACB_DEMOD_ARGS);
	case 2: return launch_demod_pinned<2, false>(ACB_DEMOD_ARGS);
	case 1: return launch_demod_t<1, false, false>(ACB_DEMOD_ARGS);
	case 17: return launch_demod_t<1, true, false>(ACB_DEMOD_ARGS);          /* F2F bit clock at one lane: no different (profiles/r2_notes.md) */
	case 24: return launch_demod_pinned<8, true>(ACB_DEMOD_ARGS);
	case 20: return launch_demod_pinned<4, true>(ACB_DEMOD_ARGS);
	case 40: return launch_demod_t<8, false, false>(ACB_DEMOD_ARGS);
	case 36: return launch_demod_t<4, false, false>(ACB_DEMOD_ARGS);
	case 34: return launch_demod_t<2, false, false>(ACB_DEMOD_ARGS);
	case 33: return launch_demod_t<1, false, true>(ACB_DEMOD_ARGS);
	default: return launch_demod_pinned<4, false>(ACB_DEMOD_ARGS);
	}
#undef ACB_DEMOD_ARGS
}

/* ------------------------------------------------------------------------------------------
 * K3: block FEC, one thread per finished frame (blk_thread, acars.c:123-207; fixprerr acars.c:39-64;
 * fixdberr acars.c:66-90).  Integer only.  Works in place on the frame ring right behind the demod:
 * status in RawFrame::pad0 (1 = deliver, 2 = drop), err = parity errors found, txt repaired and
 * parity-stripped.  CRC and syndrome tables are generated in shared memory per CTA (syndrom.h:15-48,
 * 52-295) rather than stored.
 * ---------------------------------------------------------------------------------------- */

constexpr int FEC_SYN_BYTES = 252;      /* covers len <= 250 (the reference table has 242 rows; a
                                           241-byte block indexes past it there, see hostmath.cpp) */

__device__ __forceinline__ unsigned fec_crc_step(const unsigned short *tab, unsigned crc, unsigned c)
{
	return ((crc >> 8) ^ tab[(crc ^ c) & 0xffu]) & 0xffffu;               /* update_crc, syndrom.h:49 */
}

__device__ __forceinline__ bool fec_crc_bytes_hit(const unsigned short *syn, unsigned crc)
{
	bool hit = false;
#pragma unroll
	for (int i = 0; i < 16; i++) hit |= (syn[i] == crc);                  /* acars.c:57-62, 70-74 */
	return hit;
}

__global__ void __launch_bounds__(128)
k_block_fec(RawFrame *__restrict__ ring, const RingCtl *__restrict__ ctl, unsigned cap)
{
	__shared__ unsigned short s_crc[256];
	__shared__ unsigned short s_syn[8 * FEC_SYN_BYTES];
	/* the grid is sized for the busiest step (one thread per frame up to 75 776 frames, then a stride loop); CTAs
	 * with no frame leave before building the tables */
	if (blockIdx.x * blockDim.x >= min(ctl->count, cap)) return;
	for (int b = threadIdx.x; b < 256; b += blockDim.x) {
		unsigned r = b;
		for (int k = 0; k < 8; k++) r = (r & 1u) ? (r >> 1) ^ 0x8408u : r >> 1;
		s_crc[b] = (unsigned short)r;
	}
	__syncthreads();
	if (threadIdx.x < 8) {                                                /* one bit position per thread */
		unsigned r = s_crc[1u << threadIdx.x];
		for (int p = 0; p < FEC_SYN_BYTES; p++) {
			s_syn[threadIdx.x + 8 * p] = (unsigned short)r;
			r = fec_crc_step(s_crc, r, 0);
		}
	}
	__syncthreads();

	const unsigned count = min(ctl->count, cap);
	for (unsigned f = blockIdx.x * blockDim.x + threadIdx.x; f < count; f += gridDim.x * blockDim.x) {
		RawFrame *fr = ring + f;
		unsigned char *txt = fr->txt;
		const int len = fr->len;
		int status = 2;
		do {
			if (len < 13 || len > 250) break;                                 /* acars.c:124-129 */
			txt[12] = (unsigned char)((txt[12] & 0x83u) | 0x02u);             /* force STX/ETX, acars.c:132-133 */
			int bad[3], nbad = 0;
			unsigned crc = 0;
			for (int i = 0; i < len; i++) {
				const unsigned c = txt[i];
				if ((__popc(c) & 1) == 0) { if (nbad < 3) bad[nbad] = i; nbad++; }
				crc = fec_crc_step(s_crc, crc, c);
			}
			if (nbad > 3) break;                                              /* acars.c:145-152 */
			crc = fec_crc_step(s_crc, crc, fr->crc[0]);
			crc = fec_crc_step(s_crc, crc, fr->crc[1]);
			fr->err = nbad;
			bool ok = true;
			if (nbad) {
				/* fixprerr, depth first in the reference's order: bit of the first bad byte outermost */
				ok = false;
				const int p0 = 8 * (len - bad[0] + 1), p1 = nbad > 1 ? 8 * (len - bad[1] + 1) : 0, p2 = nbad > 2 ? 8 * (len - bad[2] + 1) : 0;
				for (int i0 = 0; i0 < 8 && !ok; i0++) {
					const unsigned c0 = crc ^ s_syn[i0 + p0];
					if (nbad == 1) {
						if (c0 == 0 || fec_crc_bytes_hit(s_syn, c0)) { txt[bad[0]] ^= (unsigned char)(1u << i0); ok = true; }
						continue;
					}
					for (int i1 = 0; i1 < 8 && !ok; i1++) {
						const unsigned c1 = c0 ^ s_syn[i1 + p1];
						if (nbad == 2) {
							if (c1 == 0 || fec_crc_bytes_hit(s_syn, c1)) {
								txt[bad[1]] ^= (unsigned char)(1u << i1); txt[bad[0]] ^= (unsigned char)(1u << i0); ok = true;
							}
							continue;
						}
						for (int i2 = 0; i2 < 8 && !ok; i2++) {
							const unsigned c2 = c1 ^ s_syn[i2 + p2];
							if (c2 == 0 || fec_crc_bytes_hit(s_syn, c2)) {
								txt[bad[2]] ^= (unsigned char)(1u << i2); txt[bad[1]] ^= (unsigned char)(1u << i1);
								txt[bad[0]] ^= (unsigned char)(1u << i0); ok = true;
							}
						}
					}
				}
			} else if (crc) {
				/* fixdberr: single wrong bit in the BCS, else two wrong bits in one byte */
				ok = fec_crc_bytes_hit(s_syn, crc);
				for (int k = 0; k < len && !ok; k++) {
					const int base = 8 * (len - k + 1);
					for (int i = 0; i < 8 && !ok; i++)
						for (int j = 0; j < 8 && !ok; j++)
							if (i != j && (crc ^ s_syn[i + base] ^ s_syn[j + base]) == 0) {
								txt[k] ^= (unsigned char)((1u << i) | (1u << j));
								ok = true;
							}
				}
			}
			if (!ok) break;
			int still = 0;                                                    /* acars.c:194-207 */
			for (int i = 0; i < len; i++) {
				const unsigned c = txt[i];
				still += ((__popc(c) & 1) == 0);
				txt[i] = (unsigned char)(c & 0x7fu);
			}
			status = still ? 2 : 1;
		} while (0);
		fr->pad0 = status;
	}
}

int launch_block_fec(RawFrame *ring, const RingCtl *ctl, unsigned cap, cudaStream_t stream)
{
	k_block_fec<<<592, 128, 0, stream>>>(ring, ctl, cap);
	return (int)cudaGetLastError();
}

} // namespace acb
