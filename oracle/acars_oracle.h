/*
 * TEST INFRASTRUCTURE — NOT PRODUCT CODE.
 *
 * CPU restatement (oracle) of acarsdec's per-channel DSP hot path, written from the
 * reference's behaviour, re-entrant (no globals), plain C + glibc libm.
 * Parity status: PINNED — tests/test_oracle_vs_reference.py checks every function below
 * bit-for-bit against the unmodified reference compiled in place (oracle/_ref, built by
 * oracle/Makefile with -O2 -ffp-contract=off) on test.wav (the 7 known messages of
 * SURVEY.md §4) and on seeded synthetic IQ; tests/golden/ holds the resulting vectors.
 * Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline leg may use this.
 */
#ifndef ACARS_ORACLE_H
#define ACARS_ORACLE_H
#include <stdint.h>

#define ORC_INTRATE 12500      /* acarsdec.h:31 */
#define ORC_OUTBLK 1024        /* RTLOUTBUFSZ rtl.c:49 */
#define ORC_FLEN 11            /* msk.c:25 */
#define ORC_MFLTOVER 12        /* msk.c:26 */
#define ORC_FLENO 133          /* msk.c:27 */
#define ORC_TXTMAX 250         /* acarsdec.h:55 */

enum { ORC_WSYN, ORC_SYN2, ORC_SOH1, ORC_TXT, ORC_CRC1, ORC_CRC2, ORC_END }; /* acarsdec.h:88 */

typedef struct {               /* msgblk_t minus pointers/time (acarsdec.h:48-57) */
	int chn, len, err;
	float lvl;
	unsigned char txt[ORC_TXTMAX];
	unsigned char crc[2];
} orc_msg_t;

typedef struct {               /* channel_t's demod + framing state (acarsdec.h:76-89) */
	int chn;
	double MskPhi, MskDf, MskLvlSum;
	float MskClk;
	int MskBitCount;
	unsigned MskS, idx;
	float inb_re[ORC_FLEN], inb_im[ORC_FLEN];
	unsigned char outbits;
	int nbits;
	int state;
	int have_blk;
	orc_msg_t blk;
	uint64_t nbit_total;       /* not in the reference: number of putbit() calls, for tests */
} orc_chan_t;

typedef struct {               /* where decoded (pre-FEC) blocks and raw bits go */
	orc_msg_t *msgs; int nmsg, capmsg;
	uint8_t *bits; int64_t nbits, capbits;   /* optional raw-bit trace (1 = putbit saw v>0) */
} orc_sink_t;

/* tables */
void orc_build_h(float *h /*133*/);                                   /* msk.c:44-48 */
uint16_t orc_crc_step(uint16_t crc, uint8_t c);                       /* syndrom.h:49 */
uint16_t orc_syndrome(int bit, int bytes_from_end);                   /* syndrom.h:52- */
int orc_odd_parity(uint8_t c);                                        /* numbits[c]&1, syndrom.h:4 */

/* channelizer front-end (rtl.c) */
unsigned orc_choose_fc(const unsigned *freqs, int n, int K);          /* rtl.c:131-168 */
int  orc_round_freq(double mhz);                                      /* rtl.c:245-247 */
int  orc_stored_fr(unsigned fd);                                      /* rtl.c:255 */
void orc_build_wf(int fr_stored, unsigned fc, int K, float *wf /*2K, re/im interleaved*/); /* rtl.c:283-286 */
void orc_channelize(const uint8_t *iq, int nout, int K, int nch,
                    const float *wf /*nch x 2K*/, float *dm /*nch x nout*/);              /* rtl.c:334-354 */

/* generalised FIR of BASELINE configs 3/5 (no reference implementation: taps < K weight only the
 * first `taps` samples of each K-sample row; same complex-float arithmetic as orc_channelize) */
void orc_channelize_fir(const uint8_t *iq, int nout, int K, int taps, int nch,
                        const float *wf /*nch x 2*taps*/, float *dm /*nch x nout*/);

/* the product's opt-in fast channelizer (no reference implementation: this is its definition; see the .c) */
int  orc_fast_plan(const unsigned *freqs_hz, int nch, int K, unsigned fc, int *kbin /*nch*/, float *tw /*nch x K/4 x 2*/);
void orc_channelize_dft(const uint8_t *iq, int nout, int K, int nch, const int *kbin, const float *tw, float *dm /*nch x nout*/);
void orc_channelize_dft8(const uint8_t *iq, int nout, int K, int nch, const int *kbin, const float *tw, float *dm);   /* folded variant */
/* the folded form on CS16 IQ (variant 0 = soapy.c, 1 = sdrplay.c: the power-of-two scale in the twiddles) */
int  orc_fast_plan_cs16(int variant, const unsigned *freqs_hz, int nch, int K, unsigned fc, int *kbin, float *tw);
/* the real-input (air.c) fast form: bin k = (Fc - Fr + rate/4)/12500 of the real row's DFT, 4-way split */
int  orc_fast_plan_air(const int *freqs_hz, int nch, int K, int fc, int *kbin, float *tw);
void orc_channelize_rdft(const float *x, int nout, int K, int nch, const int *kbin, const float *tw, float *dm);
void orc_channelize_dft8_cs16(const int16_t *iq, int nout, int K, int nch, const int *kbin, const float *tw, float *dm);

/* Airspy front-end (air.c): float32 real samples at IF = rate/4 */
unsigned orc_air_choose_fc(unsigned minf, unsigned maxf);                 /* air.c:42-64, no-filter branch */
void orc_air_build_wf(int fr, int fc, unsigned rate, float *wf /*2K*/);    /* air.c:263-285 */
void orc_channelize_real(const float *x, int nout, int K, int nch,
                         const float *wf /*nch x 2K*/, float *dm /*nch x nout*/);      /* air.c:291-341 */

/* CS16 front-ends: variant 0 = soapy.c, 1 = sdrplay.c */
void orc_cs16_build_osc(int variant, unsigned freq_hz, unsigned fc, int K, float *osc /*2K*/); /* soapy.c:159-162, sdrplay.c:133-137 */
void orc_channelize_cs16(int variant, const int16_t *iq /*interleaved I,Q*/, int nout, int K, int nch,
                         const float *osc /*nch x 2K*/, float *dm /*nch x nout*/);          /* soapy.c:232-254, sdrplay.c:215-236 */
/* a CS16 context with the caller's table (no reference implementation): plain D += v*w over the first `taps` samples */
void orc_channelize_cs16_table(const int16_t *iq, int nout, int K, int taps, int nch,
                               const float *wf /*nch x 2*taps*/, float *dm /*nch x nout*/);

/* demod + framing (msk.c, acars.c) */
void orc_chan_init(orc_chan_t *c, int chn);                           /* msk.c:30-51, acars.c:230-234 */
void orc_demod(orc_chan_t *c, const float *h, const float *dm, int len, orc_sink_t *sink); /* msk.c:67-137 */
void orc_decode_byte(orc_chan_t *c, orc_sink_t *sink);                /* acars.c:246-375 */
int  orc_block_fec(orc_msg_t *m);                                     /* acars.c:123-209; 1 = output, 0 = dropped */

/* whole-path convenience used by bench.py's cpu_baseline("port") leg and the tests */
typedef struct orc_stream orc_stream_t;
orc_stream_t *orc_stream_new(int K, int nch, const float *wf);
void orc_stream_free(orc_stream_t *s);
/* process nblk blocks of 1024*K*2 bytes; appends fixed messages; returns #messages so far */
int  orc_stream_blocks(orc_stream_t *s, const uint8_t *iq, int nblk);
int  orc_stream_msgs(orc_stream_t *s, orc_msg_t *out, int max);
orc_chan_t *orc_stream_chan(orc_stream_t *s, int ch);
const float *orc_stream_dm(orc_stream_t *s, int ch);
/* run `nthreads` independent streams (same iq for all) over nblk blocks, return seconds */
double orc_bench_streams(int nthreads, int K, int nch, const float *wf, const uint8_t *iq, int nbuf, int nblk);

#endif
