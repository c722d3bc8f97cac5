/*
 * TEST INFRASTRUCTURE — NOT PRODUCT CODE.  See acars_oracle.h for scope and parity status.
 *
 * Restatement of the reference's algorithm for the hot path; every function cites the
 * reference file:line it follows.  Build: -O2 -ffp-contract=off (strict IEEE, no FMA
 * contraction), the same flags as the in-place reference build it is pinned against.
 * Third-party arithmetic on the path is glibc libm only (sincos, hypotf, cosf, sincosf,
 * log10); this file calls the same entry points the reference reaches.
 */
#define _GNU_SOURCE
#include <math.h>
#include <pthread.h>
#include <stdlib.h>
#include <string.h>
#include <time.h>
#include "acars_oracle.h"

/* ------------------------------------------------------------------ tables */

/* msk.c:44-48 — half-cosine matched filter, oversampled x12, negative lobes clamped */
void orc_build_h(float *h)
{
	for (int i = 0; i < ORC_FLENO; i++) {
		h[i] = cosf(2.0 * M_PI * 600.0 / ORC_INTRATE / ORC_MFLTOVER * (i - (ORC_FLENO - 1) / 2));
		if (h[i] < 0) h[i] = 0;
	}
}

/* syndrom.h:15-49 — the table there is the reflected CCITT CRC (poly 0x8408, "Kermit"),
 * stepped one byte at a time; this computes the same step bitwise. */
uint16_t orc_crc_step(uint16_t crc, uint8_t c)
{
	crc ^= c;
	for (int k = 0; k < 8; k++)
		crc = (crc & 1) ? (uint16_t)((crc >> 1) ^ 0x8408) : (uint16_t)(crc >> 1);
	return crc;
}

/* syndrom.h:52-295 — syndrom[bit + 8*p] is the CRC left by a single wrong bit `bit` in the
 * byte that sits p bytes before the end of (text + 2 CRC bytes); CRC is linear, init 0. */
uint16_t orc_syndrome(int bit, int p)
{
	uint16_t crc = orc_crc_step(0, (uint8_t)(1u << bit));
	while (p-- > 0) crc = orc_crc_step(crc, 0);
	return crc;
}

/* syndrom.h:4-13 used as numbits[c]&1: 1 when the byte has an odd number of set bits */
int orc_odd_parity(uint8_t c)
{
	c ^= c >> 4; c ^= c >> 2; c ^= c >> 1;
	return c & 1;
}

/* ------------------------------------------------------------------ channelizer front-end */

/* rtl.c:245-247 — MHz string value to Hz, rounded to the 12.5 kHz raster */
int orc_round_freq(double mhz)
{
	return ((int)(1000000 * mhz + ORC_INTRATE / 2) / ORC_INTRATE) * ORC_INTRATE;
}

/* rtl.c:255 — channel[].Fr is an int assigned from a float cast of the frequency */
int orc_stored_fr(unsigned fd) { return (int)(float)fd; }

/* rtl.c:131-168 — pick the tuner centre: highest Fc (1 Hz steps, downward) such that every
 * channel is >= 2*INTRATE from DC, <= rate/2 - 2*INTRATE away, and no two are mirror images */
unsigned orc_choose_fc(const unsigned *freqs, int n, int K)
{
	unsigned f[64];
	int rate = ORC_INTRATE * K;
	if (n > 64) return 0;
	memcpy(f, freqs, n * sizeof(unsigned));
	for (int i = 1; i < n; i++)            /* ascending sort (the reference bubble-sorts) */
		for (int j = i; j > 0 && f[j - 1] > f[j]; j--) { unsigned t = f[j]; f[j] = f[j - 1]; f[j - 1] = t; }
	if ((long long)f[n - 1] - f[0] > rate - 4 * ORC_INTRATE) return 0;
	long long fc;
	for (fc = (long long)f[n - 1] + 2 * ORC_INTRATE; fc > (long long)f[0] - 2 * ORC_INTRATE; fc--) {
		int k;
		for (k = 0; k < n; k++) {
			long long d = llabs(fc - f[k]);
			if (d > rate / 2 - 2 * ORC_INTRATE) break;
			if (d < 2 * ORC_INTRATE) break;
			if (k > 0 && fc - f[k - 1] == (long long)f[k] - fc) break;
		}
		if (k == n) break;
	}
	return (unsigned)fc;
}

/* rtl.c:283-286 — per-channel table: NCO x boxcar(K) x 1/127.5 scaling, one float complex per tap */
void orc_build_wf(int fr_stored, unsigned fc, int K, float *wf)
{
	float rate = (float)(ORC_INTRATE * K);
	float am = (float)(((float)fr_stored - (float)fc) / rate * 2.0 * M_PI);
	for (int ind = 0; ind < K; ind++) {
		float ph = am * ind, sn, cs;
		sincosf(-ph, &sn, &cs);                 /* cexpf(-j ph), rtl.c:285 */
		float re = cs / (float)K, im = sn / (float)K;   /* complex / int */
		wf[2 * ind] = (float)((double)re / 127.5);      /* complex / double, stored float */
		wf[2 * ind + 1] = (float)((double)im / 127.5);
	}
}

/* rtl.c:334-354 — u8 IQ -> per channel |sum_k (x_k - 127.37) * wf_k| over K samples, no overlap.
 * float complex arithmetic spelled out: product (ac-bd, ad+bc), then accumulate, in tap order. */
void orc_channelize(const uint8_t *iq, int nout, int K, int nch, const float *wf, float *dm)
{
	for (int m = 0; m < nout; m++) {
		const uint8_t *p = iq + (size_t)m * K * 2;
		for (int ch = 0; ch < nch; ch++) {
			const float *w = wf + (size_t)ch * 2 * K;
			float dr = 0, di = 0;
			for (int ind = 0; ind < K; ind++) {
				float a = (float)p[2 * ind] - 127.37f, b = (float)p[2 * ind + 1] - 127.37f;
				float c = w[2 * ind], d = w[2 * ind + 1];
				float pr = a * c - b * d, pi = a * d + b * c;
				dr = dr + pr;
				di = di + pi;
			}
			dm[(size_t)ch * nout + m] = hypotf(dr, di);     /* cabsf, rtl.c:353 */
		}
	}
}

/* Generalisation used by BASELINE configs 3 and 5 ("FIR taps=165", "tap sweep 65-513"): the
 * reference only has taps == K; with taps < K the first `taps` samples of every K-sample row are
 * weighted by an arbitrary complex table, in the same rounded operation order (rtl.c:350-353).
 * This restatement IS the definition (parity unpinned beyond taps == K, where it reduces to
 * orc_channelize). */
void orc_channelize_fir(const uint8_t *iq, int nout, int K, int taps, int nch, const float *wf, float *dm)
{
	for (int m = 0; m < nout; m++) {
		const uint8_t *p = iq + (size_t)m * K * 2;
		for (int ch = 0; ch < nch; ch++) {
			const float *w = wf + (size_t)ch * 2 * taps;
			float dr = 0, di = 0;
			for (int ind = 0; ind < taps; ind++) {
				float a = (float)p[2 * ind] - 127.37f, b = (float)p[2 * ind + 1] - 127.37f;
				float c = w[2 * ind], d = w[2 * ind + 1];
				float pr = a * c - b * d, pi = a * d + b * c;
				dr = dr + pr;
				di = di + pi;
			}
			dm[(size_t)ch * nout + m] = hypotf(dr, di);
		}
	}
}

/* The product's opt-in FAST channelizer (ACB_FLAG_FAST_CHANNELIZER, k_channelize_dft) — not in the
 * reference: this restatement is its definition, operation for operation, so the GPU kernel can be held
 * to it bit for bit while the CPU tests hold IT to the reference (envelope within the reference's own
 * table rounding, decoded messages identical; tests/test_fast_oracle.py).
 *
 * rtl.c:283-286 builds wf[ind] = cexpf(-j*AMFreq*ind)/K/127.5, a sampled complex exponential.  When the
 * offset the reference mixes with — float image of the stored Fr minus float image of Fc — is a whole,
 * even number k of 12.5 kHz steps, D = sum_ind x[ind]*wf[ind] is bin k of a K-point DFT of the row:
 *   D = sum_{n2<K/4} T[n2] * Y_r[n2],  T[n2] = exp(-j*2*pi*k*n2/K)/K/127.5,  r = k mod 4 (0 or 2),
 *   Y_0 = x0+x1+x2+x3 - 4*127.5,  Y_2 = x0-x1+x2-x3,  x_q = x[(K/4)*q + n2]   (exact in float). */
int orc_fast_plan(const unsigned *freqs_hz, int nch, int K, unsigned fc, int *kbin, float *tw)
{
	const int N2 = K / 4;
	for (int ch = 0; ch < nch; ch++) {
		const float d = (float)orc_stored_fr(freqs_hz[ch]) - (float)fc;
		const float kf = d / (float)ORC_INTRATE;
		const int k = (int)kf;
		if ((float)k != kf || (k & 1) || k == 0 || k <= -K / 2 || k >= K / 2) return 0;
		kbin[ch] = k;
		for (int n2 = 0; n2 < N2; n2++) {
			const double ph = -2.0 * M_PI * (double)(((long long)k * n2) % K) / (double)K;
			tw[((size_t)ch * N2 + n2) * 2] = (float)(cos(ph) / K / 127.5);
			tw[((size_t)ch * N2 + n2) * 2 + 1] = (float)(sin(ph) / K / 127.5);
		}
	}
	return 1;
}

void orc_channelize_dft(const uint8_t *iq, int nout, int K, int nch, const int *kbin, const float *tw, float *dm)
{
	const int N2 = K / 4;
	for (int m = 0; m < nout; m++) {
		const uint8_t *p = iq + (size_t)m * K * 2;
		for (int ch = 0; ch < nch; ch++) {
			const int r = ((kbin[ch] % 4) + 4) % 4;
			const float *t = tw + (size_t)ch * N2 * 2;
			float a = 0, b = 0, pp = 0, q = 0;          /* re = a - b, im = pp + q: four FMA chains in n2 order */
			for (int n2 = 0; n2 < N2; n2++) {
				const int i0 = p[2 * n2], i1 = p[2 * (N2 + n2)], i2 = p[2 * (2 * N2 + n2)], i3 = p[2 * (3 * N2 + n2)];
				const int q0 = p[2 * n2 + 1], q1 = p[2 * (N2 + n2) + 1], q2 = p[2 * (2 * N2 + n2) + 1], q3 = p[2 * (3 * N2 + n2) + 1];
				const float yr = r == 0 ? (float)(i0 + i1 + i2 + i3 - 510) : (float)(i0 - i1 + i2 - i3);
				const float yi = r == 0 ? (float)(q0 + q1 + q2 + q3 - 510) : (float)(q0 - q1 + q2 - q3);
				const float tr = t[2 * n2], ti = t[2 * n2 + 1];
				a = fmaf(yr, tr, a);
				b = fmaf(yi, ti, b);
				pp = fmaf(yr, ti, pp);
				q = fmaf(yi, tr, q);
			}
			const float re = a - b, im = pp + q;
			dm[(size_t)ch * nout + m] = sqrtf(fmaf(re, re, im * im));
		}
	}
}

/* Folded variant of the same (k is even, k = 2k'): z[n] = x[n] + x[n+K/2], then the four-way split of the
 * K/2-point DFT of z: D = sum_{n2<K/8} T[n2] * Y'_r[n2], r = k' mod 4, same twiddles T[n2], n2 < K/8,
 *   Y'_0 = z0+z1+z2+z3 - 8*127.5, Y'_2 = z0-z1+z2-z3, Y'_1 = (z0-z2) - j(z1-z3), Y'_3 = (z0-z2) + j(z1-z3),
 *   z_q = z[(K/8)*q + n2].  `tw` is the table of orc_fast_plan (K/4 entries per channel, first K/8 used). */
void orc_channelize_dft8(const uint8_t *iq, int nout, int K, int nch, const int *kbin, const float *tw, float *dm)
{
	const int N2 = K / 4, N8 = K / 8;
	for (int m = 0; m < nout; m++) {
		const uint8_t *p = iq + (size_t)m * K * 2;
		for (int ch = 0; ch < nch; ch++) {
			const int r = (((kbin[ch] / 2) % 4) + 4) % 4;
			const float *t = tw + (size_t)ch * N2 * 2;
			float a = 0, b = 0, pp = 0, q = 0;
			for (int n2 = 0; n2 < N8; n2++) {
				int zi[4], zq[4];
				for (int n1 = 0; n1 < 4; n1++) {
					zi[n1] = p[2 * (N8 * n1 + n2)] + p[2 * (N8 * (n1 + 4) + n2)];
					zq[n1] = p[2 * (N8 * n1 + n2) + 1] + p[2 * (N8 * (n1 + 4) + n2) + 1];
				}
				int yr, yi;
				switch (r) {
				case 0: yr = zi[0] + zi[1] + zi[2] + zi[3] - 1020; yi = zq[0] + zq[1] + zq[2] + zq[3] - 1020; break;
				case 2: yr = zi[0] - zi[1] + zi[2] - zi[3]; yi = zq[0] - zq[1] + zq[2] - zq[3]; break;
				case 1: yr = (zi[0] - zi[2]) + (zq[1] - zq[3]); yi = (zq[0] - zq[2]) - (zi[1] - zi[3]); break;
				default: yr = (zi[0] - zi[2]) - (zq[1] - zq[3]); yi = (zq[0] - zq[2]) + (zi[1] - zi[3]); break;
				}
				const float fr = (float)yr, fi = (float)yi, tr = t[2 * n2], ti = t[2 * n2 + 1];
				a = fmaf(fr, tr, a);
				b = fmaf(fi, ti, b);
				pp = fmaf(fr, ti, pp);
				q = fmaf(fi, tr, q);
			}
			const float re = a - b, im = pp + q;
			dm[(size_t)ch * nout + m] = sqrtf(fmaf(re, re, im * im));
		}
	}
}

/* The same folded form for CS16 IQ input (soapy.c:232-254, sdrplay.c:215-236): oscillator[ind] = cexpf(-j*AMFreq*ind)/K is a
 * sampled exponential too; with (float)Fr - (float)Fc a whole even number k of 12.5 kHz steps, D is bin k of the row's
 * K-point DFT.  Twiddles carry the variant's power-of-two scale (soapy.c:242 divides by 32768, sdrplay.c:225 by 4).
 * No mid-scale term: the samples are signed. */
int orc_fast_plan_cs16(int variant, const unsigned *freqs_hz, int nch, int K, unsigned fc, int *kbin, float *tw)
{
	const int N2 = K / 4;
	const double scale = variant == 0 ? 1.0 / 32768.0 : 0.25;
	for (int ch = 0; ch < nch; ch++) {
		const float d = (float)freqs_hz[ch] - (float)fc;
		const float kf = d / (float)ORC_INTRATE;
		const int k = (int)kf;
		if ((float)k != kf || (k & 1) || k == 0 || k <= -K / 2 || k >= K / 2) return 0;
		kbin[ch] = k;
		for (int n2 = 0; n2 < N2; n2++) {
			const double ph = -2.0 * M_PI * (double)(((long long)k * n2) % K) / (double)K;
			tw[((size_t)ch * N2 + n2) * 2] = (float)(cos(ph) / K * scale);
			tw[((size_t)ch * N2 + n2) * 2 + 1] = (float)(sin(ph) / K * scale);
		}
	}
	return 1;
}

void orc_channelize_dft8_cs16(const int16_t *iq, int nout, int K, int nch, const int *kbin, const float *tw, float *dm)
{
	const int N2 = K / 4, N8 = K / 8;
	for (int m = 0; m < nout; m++) {
		const int16_t *p = iq + (size_t)m * K * 2;
		for (int ch = 0; ch < nch; ch++) {
			const int r = (((kbin[ch] / 2) % 4) + 4) % 4;
			const float *t = tw + (size_t)ch * N2 * 2;
			float a = 0, b = 0, pp = 0, q = 0;
			for (int n2 = 0; n2 < N8; n2++) {
				int zi[4], zq[4];
				for (int n1 = 0; n1 < 4; n1++) {
					zi[n1] = p[2 * (N8 * n1 + n2)] + p[2 * (N8 * (n1 + 4) + n2)];
					zq[n1] = p[2 * (N8 * n1 + n2) + 1] + p[2 * (N8 * (n1 + 4) + n2) + 1];
				}
				int yr, yi;
				switch (r) {
				case 0: yr = zi[0] + zi[1] + zi[2] + zi[3]; yi = zq[0] + zq[1] + zq[2] + zq[3]; break;
				case 2: yr = zi[0] - zi[1] + zi[2] - zi[3]; yi = zq[0] - zq[1] + zq[2] - zq[3]; break;
				case 1: yr = (zi[0] - zi[2]) + (zq[1] - zq[3]); yi = (zq[0] - zq[2]) - (zi[1] - zi[3]); break;
				default: yr = (zi[0] - zi[2]) - (zq[1] - zq[3]); yi = (zq[0] - zq[2]) + (zi[1] - zi[3]); break;
				}
				const float fr = (float)yr, fi = (float)yi, tr = t[2 * n2], ti = t[2 * n2 + 1];
				a = fmaf(fr, tr, a);
				b = fmaf(fi, ti, b);
				pp = fmaf(fr, ti, pp);
				q = fmaf(fi, tr, q);
			}
			const float re = a - b, im = pp + q;
			dm[(size_t)ch * nout + m] = sqrtf(fmaf(re, re, im * im));
		}
	}
}

/* ------------------------------------------------------------------ Airspy front-end (air.c) */

/* air.c:42-64 with filter == 0 (every rate but 5 MS/s): centre of the span on the 12.5 kHz raster */
unsigned orc_air_choose_fc(unsigned minf, unsigned maxf)
{
	return ((maxf + minf) / 2 + ORC_INTRATE / 2) / ORC_INTRATE * ORC_INTRATE;
}

/* air.c:263-285 — the mixer table is generated by a double phase accumulator, the IF offset is
 * rate/4, and the unit vector is cexpf of the float-rounded phase */
void orc_air_build_wf(int fr, int fc, unsigned rate, float *wf)
{
	const unsigned K = rate / ORC_INTRATE;
	const double step = 2.0 * M_PI * (double)(unsigned)(fc - fr + rate / 4) / (double)rate;
	double ph = 0;
	for (unsigned i = 0; i < K; i++) {
		float sn, cs;
		sincosf((float)-ph, &sn, &cs);
		wf[2 * i] = cs / (float)K;
		wf[2 * i + 1] = sn / (float)K;
		ph += step;
		if (ph > 2.0 * M_PI) ph -= 2.0 * M_PI;
		if (ph < -2.0 * M_PI) ph += 2.0 * M_PI;
	}
}

/* Fast form of the same (k_channelize_rdft restated operation for operation): with Fc and the channels on the 12.5 kHz
 * raster the table of orc_air_build_wf is exp(-j*2*pi*k*i/K)/K, k = (Fc - Fr + rate/4)/12500, and D is bin k of the REAL
 * row's K-point DFT; split over the row's quarters,
 *   D = sum_{n2<K/4} T[n2] * Y_r[n2],  r = k mod 4,  T[n2] = exp(-j*2*pi*k*n2/K)/K,
 *   Y_0 = (x0+x2)+(x1+x3), Y_2 = (x0+x2)-(x1+x3), Y_1 = (x0-x2) - j(x1-x3), Y_3 = (x0-x2) + j(x1-x3), x_q = x[(K/4)q + n2]. */
int orc_fast_plan_air(const int *freqs_hz, int nch, int K, int fc, int *kbin, float *tw)
{
	const int N2 = K / 4;
	const unsigned rate = (unsigned)K * ORC_INTRATE;
	if (K & 7) return 0;
	for (int ch = 0; ch < nch; ch++) {
		const unsigned off = (unsigned)(fc - freqs_hz[ch] + (int)(rate / 4));      /* air.c:278 */
		if (off % ORC_INTRATE) return 0;
		const int k = (int)(off / ORC_INTRATE);
		if (k <= 0 || k >= K) return 0;
		kbin[ch] = k;
		for (int n2 = 0; n2 < N2; n2++) {
			const double ph = -2.0 * M_PI * (double)(((long long)k * n2) % K) / (double)K;
			tw[((size_t)ch * N2 + n2) * 2] = (float)(cos(ph) / K);
			tw[((size_t)ch * N2 + n2) * 2 + 1] = (float)(sin(ph) / K);
		}
	}
	return 1;
}

/* `lpr` lanes of the kernel share a row (K/100 rounded down to a power of two: 2, 4, 4, 8 for K = 200, 400, 480, 800): lane h
 * sums the h-th range of ceil(K/8 / lpr) n2 PAIRS in n2 order, the partial sums are added pairwise (h^1, then h^2, ...). */
void orc_channelize_rdft(const float *x, int nout, int K, int nch, const int *kbin, const float *tw, float *dm)
{
	const int N2 = K / 4, K8 = K / 8;
	const int lpr = K >= 800 ? 8 : K >= 400 ? 4 : 2, per = (K8 + lpr - 1) / lpr;
	for (int m = 0; m < nout; m++) {
		const float *p = x + (size_t)m * K;
		for (int ch = 0; ch < nch; ch++) {
			const int r = kbin[ch] & 3;
			const float *t = tw + (size_t)ch * N2 * 2;
			float ax[8] = { 0 }, ay[8] = { 0 }, bx[8] = { 0 }, by[8] = { 0 };   /* A = sum Ye*T (or (x0-x2)*T), B = sum (x1-x3)*T */
			for (int h = 0; h < lpr; h++) {
				const int g0 = h * per, g1 = g0 + per < K8 ? g0 + per : K8;
				for (int n2 = 2 * g0; n2 < 2 * g1; n2++) {
					const float x0 = p[n2], x1 = p[N2 + n2], x2 = p[2 * N2 + n2], x3 = p[3 * N2 + n2];
					const float tr = t[2 * n2], ti = t[2 * n2 + 1];
					if (r == 0 || r == 2) {
						const float s02 = x0 + x2, s13 = x1 + x3;
						const float y = r == 0 ? s02 + s13 : s02 - s13;
						ax[h] = fmaf(y, tr, ax[h]);
						ay[h] = fmaf(y, ti, ay[h]);
					} else {
						const float d02 = x0 - x2, d13 = x1 - x3;
						ax[h] = fmaf(d02, tr, ax[h]);
						ay[h] = fmaf(d02, ti, ay[h]);
						bx[h] = fmaf(d13, tr, bx[h]);
						by[h] = fmaf(d13, ti, by[h]);
					}
				}
			}
			for (int step = 1; step < lpr; step *= 2)
				for (int h = 0; h < lpr; h += 2 * step) {
					ax[h] += ax[h + step]; ay[h] += ay[h + step]; bx[h] += bx[h + step]; by[h] += by[h + step];
				}
			const float sg = r == 3 ? -1.0f : 1.0f;
			const float re = ax[0] + sg * by[0], im = ay[0] - sg * bx[0];
			dm[(size_t)ch * nout + m] = sqrtf(fmaf(re, re, im * im));
		}
	}
}

/* air.c:291-341 — D += wf[i]*S over K consecutive REAL samples per output; the reference carries
 * D and the tap index across transfers of arbitrary size, which is the same sequence of rounded
 * operations as walking the concatenated stream row by row */
void orc_channelize_real(const float *x, int nout, int K, int nch, const float *wf, float *dm)
{
	for (int m = 0; m < nout; m++) {
		const float *p = x + (size_t)m * K;
		for (int ch = 0; ch < nch; ch++) {
			const float *w = wf + (size_t)ch * 2 * K;
			float dr = 0, di = 0;
			for (int i = 0; i < K; i++) {
				float pr = w[2 * i] * p[i], pi = w[2 * i + 1] * p[i];
				dr = dr + pr;
				di = di + pi;
			}
			dm[(size_t)ch * nout + m] = hypotf(dr, di);
		}
	}
}

/* ------------------------------------------------------------------ CS16 front-ends */

/* soapy.c:159-162 (float per-tap phase) / sdrplay.c:133-137 (double per-tap phase, rounded to
 * float by cexpf's argument); channel[].Fr is a float in both */
void orc_cs16_build_osc(int variant, unsigned freq_hz, unsigned fc, int K, float *osc)
{
	float fr = (float)freq_hz;
	double dstep = (fr - (float)fc) / (float)(ORC_INTRATE * K) * 2.0 * M_PI;
	float fstep = (float)dstep;
	for (int ind = 0; ind < K; ind++) {
		float sn, cs;
		if (variant == 0) sincosf(-(fstep * ind), &sn, &cs);
		else sincosf((float)-(dstep * ind), &sn, &cs);
		osc[2 * ind] = cs / (float)K;
		osc[2 * ind + 1] = sn / (float)K;
	}
}

/* soapy.c:238-243: D += v * osc[ind] / 32768.0 — the float complex product is widened to double,
 * divided, added to D in double and the sum stored back to float.  sdrplay.c:218-225: D += v*osc in
 * float, envelope cabsf(D)/4.  The references carry D and ind across reads: same operation order. */
void orc_channelize_cs16(int variant, const int16_t *iq, int nout, int K, int nch, const float *osc, float *dm)
{
	for (int m = 0; m < nout; m++) {
		const int16_t *p = iq + (size_t)m * K * 2;
		for (int ch = 0; ch < nch; ch++) {
			const float *w = osc + (size_t)ch * 2 * K;
			float dr = 0, di = 0;
			for (int ind = 0; ind < K; ind++) {
				float a = (float)p[2 * ind], b = (float)p[2 * ind + 1];
				float c = w[2 * ind], d = w[2 * ind + 1];
				float pr = a * c - b * d, pi = a * d + b * c;
				if (variant == 0) {
					dr = (float)((double)dr + (double)pr / 32768.0);
					di = (float)((double)di + (double)pi / 32768.0);
				} else {
					dr = dr + pr;
					di = di + pi;
				}
			}
			float e = hypotf(dr, di);
			dm[(size_t)ch * nout + m] = variant == 1 ? e / 4 : e;   /* variant 2: plain D += v*w, |D| (what the
			                                                           product computes with folded tables) */
		}
	}
}

/* A CS16 context with the caller's table (acb_set_wf; taps <= K): the complex MAC of rtl.c:350-352 on (float)int16 with
 * no bias, product (ac-bd, ad+bc) rounded, then the accumulate rounded, over the first `taps` samples of every K-sample
 * row in tap order.  No reference has this mode; with the folded planner tables and taps == K it is
 * orc_channelize_cs16 (tests/test_cs16_oracle.py). */
void orc_channelize_cs16_table(const int16_t *iq, int nout, int K, int taps, int nch, const float *wf, float *dm)
{
	for (int m = 0; m < nout; m++) {
		const int16_t *p = iq + (size_t)m * K * 2;
		for (int ch = 0; ch < nch; ch++) {
			const float *w = wf + (size_t)ch * 2 * taps;
			float dr = 0, di = 0;
			for (int ind = 0; ind < taps; ind++) {
				float a = (float)p[2 * ind], b = (float)p[2 * ind + 1];
				float c = w[2 * ind], d = w[2 * ind + 1];
				float pr = a * c - b * d, pi = a * d + b * c;
				dr = dr + pr;
				di = di + pi;
			}
			dm[(size_t)ch * nout + m] = hypotf(dr, di);
		}
	}
}

/* ------------------------------------------------------------------ frame sync (acars.c) */

#define SYN 0x16
#define SOH 0x01
#define STX 0x02
#define ETX 0x83
#define ETB 0x97
#define DLE 0x7f
#define MAXPERR 3

static void sink_msg(orc_sink_t *s, const orc_msg_t *m)
{
	if (!s) return;
	if (s->nmsg == s->capmsg) {
		s->capmsg = s->capmsg ? 2 * s->capmsg : 64;
		s->msgs = realloc(s->msgs, s->capmsg * sizeof(orc_msg_t));
	}
	s->msgs[s->nmsg++] = *m;
}

/* acars.c:239-244 */
static void frame_reset(orc_chan_t *c)
{
	c->state = ORC_WSYN;
	c->MskDf = 0;
	c->nbits = 1;
}

/* acars.c:350-369 — level estimate and hand-off to the block queue */
static void frame_put(orc_chan_t *c, orc_sink_t *sink)
{
	c->blk.lvl = (float)(10 * log10(c->MskLvlSum / c->MskBitCount));
	sink_msg(sink, &c->blk);
	c->have_blk = 0;
	c->state = ORC_END;
	c->nbits = 8;
}

/* acars.c:246-375 — one assembled byte (or one bit while hunting for SYN) */
void orc_decode_byte(orc_chan_t *c, orc_sink_t *sink)
{
	unsigned char r = c->outbits;
	switch (c->state) {
	case ORC_WSYN:
		if (r == SYN || r == (unsigned char)~SYN) {
			if (r != SYN) c->MskS ^= 2;             /* inverted polarity, acars.c:258-259 */
			c->state = ORC_SYN2; c->nbits = 8;
		} else
			c->nbits = 1;
		return;
	case ORC_SYN2:
		if (r == SYN) { c->state = ORC_SOH1; c->nbits = 8; return; }
		if (r == (unsigned char)~SYN) { c->MskS ^= 2; c->nbits = 8; return; }
		frame_reset(c);
		return;
	case ORC_SOH1:
		if (r != SOH) { frame_reset(c); return; }
		c->have_blk = 1;
		c->blk.chn = c->chn; c->blk.len = 0; c->blk.err = 0;
		c->state = ORC_TXT; c->nbits = 8;
		c->MskLvlSum = 0; c->MskBitCount = 0;
		return;
	case ORC_TXT:
		c->blk.txt[c->blk.len++] = r;
		if (!orc_odd_parity(r) && ++c->blk.err > MAXPERR + 1) { frame_reset(c); return; }
		if (r == ETX || r == ETB) { c->state = ORC_CRC1; c->nbits = 8; return; }
		if (c->blk.len > 20 && r == DLE) {            /* missed the end of text, acars.c:324-333 */
			c->blk.len -= 3;
			c->blk.crc[0] = c->blk.txt[c->blk.len];
			c->blk.crc[1] = c->blk.txt[c->blk.len + 1];
			frame_put(c, sink);
			return;
		}
		if (c->blk.len > 240) { frame_reset(c); return; }
		c->nbits = 8;
		return;
	case ORC_CRC1:
		c->blk.crc[0] = r; c->state = ORC_CRC2; c->nbits = 8;
		return;
	case ORC_CRC2:
		c->blk.crc[1] = r;
		frame_put(c, sink);
		return;
	case ORC_END:
		frame_reset(c);
		c->nbits = 8;
		return;
	}
}

/* ------------------------------------------------------------------ block FEC (acars.c:39-215) */

/* acars.c:39-64 */
static int fix_parity_errs(orc_msg_t *m, uint16_t crc, const int *pr, int pn)
{
	if (pn > 0) {
		for (int i = 0; i < 8; i++)
			if (fix_parity_errs(m, crc ^ orc_syndrome(i, m->len - *pr + 1), pr + 1, pn - 1)) {
				m->txt[*pr] ^= (1 << i);
				return 1;
			}
		return 0;
	}
	if (crc == 0) return 1;
	for (int i = 0; i < 16; i++)
		if (orc_syndrome(i & 7, i >> 3) == crc) return 1;
	return 0;
}

/* acars.c:66-90 */
static int fix_double_err(orc_msg_t *m, uint16_t crc)
{
	for (int i = 0; i < 16; i++)
		if (orc_syndrome(i & 7, i >> 3) == crc) return 1;
	for (int k = 0; k < m->len; k++) {
		int p = m->len - k + 1;
		for (int i = 0; i < 8; i++)
			for (int j = 0; j < 8; j++) {
				if (i == j) continue;
				if ((crc ^ orc_syndrome(i, p) ^ orc_syndrome(j, p)) == 0) {
					m->txt[k] ^= (1 << i);
					m->txt[k] ^= (1 << j);
					return 1;
				}
			}
	}
	return 0;
}

/* acars.c:123-209 — returns 1 when the reference would call outputmsg(), 0 when it drops */
int orc_block_fec(orc_msg_t *m)
{
	int pr[MAXPERR], pn = 0;
	uint16_t crc = 0;
	if (m->len < 13) return 0;
	m->txt[12] &= (ETX | STX);
	m->txt[12] |= (ETX & STX);
	for (int i = 0; i < m->len; i++)
		if (!orc_odd_parity(m->txt[i])) { if (pn < MAXPERR) pr[pn] = i; pn++; }
	if (pn > MAXPERR) return 0;
	m->err = pn;
	for (int i = 0; i < m->len; i++) crc = orc_crc_step(crc, m->txt[i]);
	crc = orc_crc_step(crc, m->crc[0]);
	crc = orc_crc_step(crc, m->crc[1]);
	if (pn) { if (!fix_parity_errs(m, crc, pr, pn)) return 0; }
	else if (crc && !fix_double_err(m, crc)) return 0;
	pn = 0;
	for (int i = 0; i < m->len; i++) {
		if (!orc_odd_parity(m->txt[i])) pn++;
		m->txt[i] &= 0x7f;
	}
	return pn == 0;
}

/* ------------------------------------------------------------------ MSK demodulator (msk.c) */

void orc_chan_init(orc_chan_t *c, int chn)
{
	memset(c, 0, sizeof(*c));      /* msk.c:34-40 */
	c->chn = chn;
	c->nbits = 8;                  /* acars.c:230-234 */
	c->state = ORC_WSYN;
}

/* msk.c:53-63 */
static inline void put_bit(orc_chan_t *c, float v, orc_sink_t *sink)
{
	c->outbits >>= 1;
	if (v > 0) c->outbits |= 0x80;
	if (sink && sink->bits && sink->nbits < sink->capbits) sink->bits[sink->nbits++] = v > 0;
	c->nbit_total++;
	if (--c->nbits <= 0) orc_decode_byte(c, sink);
}

/* msk.c:67-137 — numerics contract of SURVEY.md §8(a): double VCO, float ring, float MF */
void orc_demod(orc_chan_t *c, const float *h, const float *dm, int len, orc_sink_t *sink)
{
	const double pllc = (double)0.52f, pllg = (double)38e-4f;     /* msk.c:65-66, float constants */
	unsigned idx = c->idx;
	double p = c->MskPhi;
	for (int n = 0; n < len; n++) {
		double s = 1800.0 / ORC_INTRATE * 2.0 * M_PI + c->MskDf;    /* msk.c:81 */
		double sn, cs;
		p += s;
		if (p >= 2.0 * M_PI) p -= 2.0 * M_PI;
		sincos(-p, &sn, &cs);                                      /* cexp(-p*I), msk.c:90 */
		c->inb_re[idx] = (float)((double)dm[n] * cs);
		c->inb_im[idx] = (float)((double)dm[n] * sn);
		idx = (idx + 1) % ORC_FLEN;

		c->MskClk = (float)((double)c->MskClk + s);                /* msk.c:95, float state */
		if ((double)c->MskClk >= 3 * M_PI / 2.0 - s / 2) {
			float vr = 0, vi = 0, lvl, vo;
			double dphi, d;
			int o;
			c->MskClk = (float)((double)c->MskClk - 3 * M_PI / 2.0);
			o = (int)(ORC_MFLTOVER * ((double)c->MskClk / s + 0.5));   /* msk.c:103 */
			if (o > ORC_MFLTOVER) o = ORC_MFLTOVER;
			for (int j = 0; j < ORC_FLEN; j++, o += ORC_MFLTOVER) {
				unsigned k = (j + idx) % ORC_FLEN;
				vr = vr + h[o] * c->inb_re[k];
				vi = vi + h[o] * c->inb_im[k];
			}
			lvl = hypotf(vr, vi);                                  /* cabsf, msk.c:110 */
			d = (double)lvl + 1e-8;
			vr = (float)((double)vr / d);
			vi = (float)((double)vi / d);
			c->MskLvlSum += lvl * lvl / 4;
			c->MskBitCount++;
			if (c->MskS & 1) { vo = vi; dphi = (vo >= 0) ? -vr : vr; }
			else             { vo = vr; dphi = (vo >= 0) ? vi : -vi; }
			put_bit(c, (c->MskS & 2) ? -vo : vo, sink);
			c->MskS++;
			c->MskDf = pllc * c->MskDf + (1.0 - pllc) * pllg * dphi;   /* msk.c:130 */
		}
	}
	c->idx = idx;
	c->MskPhi = p;
}

/* ------------------------------------------------------------------ whole path, one stream */

struct orc_stream {
	int K, nch;
	float *wf, *dm;
	float h[ORC_FLENO];
	orc_chan_t *ch;
	orc_sink_t raw;
	orc_msg_t *out; int nout, capout;
};

orc_stream_t *orc_stream_new(int K, int nch, const float *wf)
{
	orc_stream_t *s = calloc(1, sizeof(*s));
	s->K = K; s->nch = nch;
	s->wf = malloc(sizeof(float) * 2 * K * nch);
	memcpy(s->wf, wf, sizeof(float) * 2 * K * nch);
	s->dm = malloc(sizeof(float) * ORC_OUTBLK * nch);
	s->ch = malloc(sizeof(orc_chan_t) * nch);
	for (int i = 0; i < nch; i++) orc_chan_init(&s->ch[i], i);
	orc_build_h(s->h);
	return s;
}

void orc_stream_free(orc_stream_t *s)
{
	if (!s) return;
	free(s->wf); free(s->dm); free(s->ch); free(s->raw.msgs); free(s->out); free(s);
}

/* rtl.c:314-361: channelize one block for all channels, then demod channel by channel;
 * decoded blocks go through the FEC in emission order (block-major, channel, time). */
int orc_stream_blocks(orc_stream_t *s, const uint8_t *iq, int nblk)
{
	for (int b = 0; b < nblk; b++) {
		orc_channelize(iq + (size_t)b * ORC_OUTBLK * s->K * 2, ORC_OUTBLK, s->K, s->nch, s->wf, s->dm);
		for (int c = 0; c < s->nch; c++)
			orc_demod(&s->ch[c], s->h, s->dm + (size_t)c * ORC_OUTBLK, ORC_OUTBLK, &s->raw);
		for (int i = 0; i < s->raw.nmsg; i++) {
			orc_msg_t m = s->raw.msgs[i];
			if (!orc_block_fec(&m)) continue;
			if (s->nout == s->capout) {
				s->capout = s->capout ? 2 * s->capout : 64;
				s->out = realloc(s->out, s->capout * sizeof(orc_msg_t));
			}
			s->out[s->nout++] = m;
		}
		s->raw.nmsg = 0;
	}
	return s->nout;
}

int orc_stream_msgs(orc_stream_t *s, orc_msg_t *out, int max)
{
	int n = s->nout < max ? s->nout : max;
	memcpy(out, s->out, n * sizeof(orc_msg_t));
	memmove(s->out, s->out + n, (s->nout - n) * sizeof(orc_msg_t));
	s->nout -= n;
	return n;
}

orc_chan_t *orc_stream_chan(orc_stream_t *s, int ch) { return &s->ch[ch]; }
const float *orc_stream_dm(orc_stream_t *s, int ch) { return s->dm + (size_t)ch * ORC_OUTBLK; }

/* ------------------------------------------------------------------ CPU baseline ("port") */

typedef struct { int K, nch, nbuf, nblk; const float *wf; const uint8_t *iq; } bench_arg_t;

static void *bench_thread(void *a)
{
	bench_arg_t *b = a;
	orc_stream_t *s = orc_stream_new(b->K, b->nch, b->wf);
	size_t blk = (size_t)ORC_OUTBLK * b->K * 2;
	for (int i = 0; i < b->nblk; i++) orc_stream_blocks(s, b->iq + (size_t)(i % b->nbuf) * blk, 1);
	orc_stream_free(s);
	return NULL;
}

double orc_bench_streams(int nthreads, int K, int nch, const float *wf, const uint8_t *iq, int nbuf, int nblk)
{
	pthread_t th[256];
	bench_arg_t a = { K, nch, nbuf, nblk, wf, iq };
	struct timespec t0, t1;
	if (nthreads > 256) nthreads = 256;
	clock_gettime(CLOCK_MONOTONIC, &t0);
	for (int i = 0; i < nthreads; i++) pthread_create(&th[i], NULL, bench_thread, &a);
	for (int i = 0; i < nthreads; i++) pthread_join(th[i], NULL);
	clock_gettime(CLOCK_MONOTONIC, &t1);
	return (t1.tv_sec - t0.tv_sec) + 1e-9 * (t1.tv_nsec - t0.tv_nsec);
}
