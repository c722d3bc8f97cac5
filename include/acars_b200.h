/*
 * acars_b200 — C ABI of the B200-native acarsdec hot path
 * (u8 IQ -> per-channel mix+boxcar+decimate -> |.| -> demodMSK -> ACARS frame sync -> block FEC).
 *
 * Two layers, both plain C:
 *
 *  1. The context API below (acb_*): N independent IQ streams x C channels per GPU, the
 *     superset needed beyond MAXNBCHANNELS=16 (acarsdec.h:30).  Every entry point cites the
 *     reference interface it replaces.
 *  2. The reference's own symbols (initMsk/demodMSK/initAcars/decodeAcars/deinitAcars and the
 *     initRtl/runRtlSample/runRtlCancel/runRtlClose front-end trio) exported by
 *     libacarsdec_compat.so, declared in include/acarsdec_compat.h, implemented as a thin shim
 *     over this API so that acarsdec.c links against it unchanged.
 *
 * There is no CPU fallback: every processing call fails with ACB_ERR_CUDA when no sm_100
 * device / kernel image is available.
 */
#ifndef ACARS_B200_H
#define ACARS_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ACB_INTRATE 12500   /* acarsdec.h:31  INTRATE */
#define ACB_OUTBLK 1024     /* rtl.c:49       RTLOUTBUFSZ: output samples per IQ block */
#define ACB_TXTMAX 250      /* acarsdec.h:55  msgblk_t.txt */
#define ACB_MAXK 2048       /* rtl.c:39 caps rtlMult at 320; wideband configs go beyond */

enum {
	ACB_OK = 0,
	ACB_ERR_ARG = -1,       /* bad argument */
	ACB_ERR_CUDA = -2,      /* CUDA runtime error / no device (see acb_last_error) */
	ACB_ERR_NOMEM = -3,
	ACB_ERR_OVERFLOW = -4,  /* device message ring overflowed: frames were lost */
	ACB_ERR_PLAN = -5       /* frequency plan impossible (rtl.c:149-152) */
};

typedef struct acb_ctx acb_ctx_t;

typedef struct {
	int device;             /* CUDA ordinal */
	int K;                  /* rtlMult: input rate = K*12500, taps == decimation (rtl.c:213-214) */
	int nstreams;           /* independent IQ streams served by this context */
	int nch;                /* channels per stream */
	int max_blocks;         /* largest nblk a submit call may carry (sizes device staging) */
	int flags;              /* ACB_FLAG_* */
	int taps;               /* FIR length per output: 0 = K (the reference: boxcar x NCO over the whole
	                           decimation period, rtl.c:283-286).  1..K selects the generalised case of
	                           BASELINE configs 3/5: only the first `taps` samples of every K-sample row
	                           are weighted (tables from acb_set_wf, nch x 2*taps floats), same arithmetic */
} acb_config_t;

#define ACB_FLAG_NO_INPUT_STAGING 1   /* caller only uses acb_submit_device / acb_submit_dm_* */
#define ACB_FLAG_CS16_INPUT 4         /* SoapySDR / SDRplay front-ends (soapy.c, sdrplay.c): int16 I,Q samples;
                                         use acb_set_plan_cs16 / acb_submit_cs16_host (or _planar_host) */
#define ACB_FLAG_FAST_CHANNELIZER 8    /* u8 IQ contexts planned with acb_set_plan and CS16 contexts planned with
                                         acb_set_plan_cs16, K = 160 or 192 (real-input contexts planned with
                                         acb_set_plan_air, K = 200, 240, 400, 480 or 800: the same idea on a real row,
                                         k_channelize_rdft): run the channelizer
                                         as a shared 4-point DFT across the row quarters + K/4 MACs per channel
                                         (5x less FP32 work) when every stream's channels sit on the 12.5 kHz raster
                                         around Fc; otherwise the exact kernel runs.  NOT the reference's operation
                                         order: relative to the total in-band signal the envelope is within 1e-6 of the exact DFT
                                         bin and within the reference's own table rounding (1e-5) of the reference; decoded
                                         messages are the same; without this flag the envelope is bit-identical */
#define ACB_FLAG_REAL_INPUT 2         /* Airspy front-end (air.c): float32 REAL samples at IF = rate/4,
                                         rate = K*12500; use acb_set_plan_air / acb_submit_real_host */

/* One decoded block, after parity/CRC repair: msgblk_t (acarsdec.h:48-57) without the queue
 * link, plus where it came from.  `txt` is parity-stripped (acars.c:200). */
typedef struct {
	int stream;
	int chn;
	int len;
	int err;                /* parity errors repaired (acars.c:156) */
	float lvl;              /* 10*log10(MskLvlSum/MskBitCount), acars.c:351 */
	uint64_t block;         /* index of the 1024-sample block in which the frame completed */
	uint64_t pos;           /* channel sample index (12.5 kS/s) at which the frame completed */
	uint64_t soh_pos;       /* channel sample index of the SOH byte (reference: gettimeofday, acars.c:290) */
	unsigned char txt[ACB_TXTMAX];
	unsigned char crc[2];
} acb_msg_t;

/* Per-channel demodulator + framing state: the persistent part of channel_t (acarsdec.h:76-89). */
typedef struct {
	double MskPhi, MskDf, MskLvlSum;
	float MskClk;
	int MskBitCount;
	unsigned MskS, idx;
	int nbits, Acarsstate;
	unsigned outbits;
	int blk_len, blk_err;
	uint64_t pos, soh_pos;
	float inb_re[11], inb_im[11];   /* msk.c:40 ring, FLEN=11 */
	unsigned char blk_crc[2];
	unsigned char blk_txt[ACB_TXTMAX];
} acb_chan_state_t;

/* ---- message formatting (SURVEY §8 f3): for hosts that take acb_msg_t blocks and do not link the reference's output.c ----
 * outputmsg()'s field split (output.c:486-640), label.c's OOOI fields, and the reference's wire formats, byte for byte
 * (tests/test_outfmt.py diffs them against output.c / label.c / netout.c / cJSON.c compiled in place).  Host only.
 * Not rebuilt: MQTT, libacars decoding, log-file rotation. */
#define ACB_REFERENCE_VERSION "3.7"      /* ACARSDEC_VERSION (acarsdec.h:28): the "app" object of the JSON format carries it */
typedef struct {
	char mode, ack, bid, bs, be;          /* ack: '!' for NAK; bs / be: the text's start and end bytes (STX/ETX/ETB) */
	char addr[8], label[3], no[5], fid[7];
	int downlink;                         /* block id '0'..'9' (output.c:31): message number and flight id are present */
	int txt_off, txt_len;                 /* the message text inside acb_msg_t.txt */
	int has_oooi;                         /* label.c's DecodeLabel matched; fields below are 4 characters or empty */
	char da[5], sa[5], eta[5], gout[5], gin[5], woff[5], won[5];
} acb_fields_t;
/* 1 = split done, 0 = not a block blk_thread would deliver (len < 13) */
int acb_msg_fields(const acb_msg_t *m, acb_fields_t *out);
typedef struct {
	int64_t tv_sec, tv_usec;              /* msgblk_t.tv */
	unsigned freq_hz;                     /* channel[chn].Fr: printed by the full format when inmode >= 3, and by JSON */
	int inmode;                           /* acarsdec.c's input mode: >= 3 shows the frequency, 2 (sound file) shows no date */
	int airflt, emptymsg;                 /* -A: downlinks only; -e: messages with text only */
	const char *labels;                   /* -i "H1:Q0:...": labels to keep; NULL keeps all */
	const char *station_id;               /* idstation; NULL or "" for none */
} acb_fmt_opts_t;
enum { ACB_FMT_ONELINE = 1, ACB_FMT_FULL = 2, ACB_FMT_JSON = 4,          /* -o 1 / 2 / 4 (without the JSON line's "\n") */
       ACB_FMT_NET_PP = 11, ACB_FMT_NET_NATIVE = 12, ACB_FMT_NET_JSON = 13 };   /* -N / -n / -j datagrams */
/* Writes the message in `format` to out (NUL-terminated; the formats may contain NUL bytes themselves where the reference
 * prints one).  Returns the length, 0 when a filter of `opt` drops the message, or a negative ACB_ERR_*. */
int acb_format_msg(const acb_msg_t *m, int format, const acb_fmt_opts_t *opt, char *out, size_t cap);
/* The flight table of output.c:349-426 (one entry per aircraft heard on a downlink; entries silent for `mdly_seconds`,
 * acarsdec's -t, default 600, are dropped) and the two outputs that need it.  Feed every block, in emission order, to ONE
 * of the two calls:
 *   acb_flights_route_json  -o 5: one JSON object per flight, the first time flight id, departure and destination are all
 *                           known (output.c:428-456); returns its length, 0 when this block produces none;
 *   acb_flights_monitor     -o 3: the monitor screen as redrawn after this block (output.c:458-484), `nbch` = channels
 *                           of the receiver (<= 16). */
typedef struct acb_flights acb_flights_t;
acb_flights_t *acb_flights_new(int mdly_seconds);
void acb_flights_free(acb_flights_t *t);
int acb_flights_route_json(acb_flights_t *t, const acb_msg_t *m, const acb_fmt_opts_t *opt, char *out, size_t cap);
int acb_flights_monitor(acb_flights_t *t, const acb_msg_t *m, int nbch, const acb_fmt_opts_t *opt, char *out, size_t cap);

/* ---- front-end planning: host-side, bit-identical to the reference's initRtl ---- */

/* rtl.c:245-247 — "131.525" -> Hz on the 12.5 kHz raster */
int acb_round_freq(double mhz);
/* rtl.c:255 — the value initRtl leaves in channel[].Fr (int <- float <- unsigned) */
int acb_stored_fr(unsigned freq_hz);
/* rtl.c:131-168 chooseFc — 0 when the span does not fit */
unsigned acb_choose_fc(const unsigned *freqs_hz, int n, int K);
/* Channel sets wider than one tuner span (rtl.c:149-152 gives up; scan.sh:1-16 walks the band sequentially): the
 * fewest receiver bands that cover them, each with its chooseFc centre.  group_of[i] = band of freqs_hz[i],
 * fc_out[g] = centre of band g; returns the number of bands (<= max_groups) or a negative error. */
int acb_plan_bands(const unsigned *freqs_hz, int n, int K, int *group_of, unsigned *fc_out, int max_groups);
/* rtl.c:283-286 — wf[ind] = cexpf(-j*AMFreq*ind)/K/127.5 as 2K floats (re,im interleaved) */
void acb_build_wf(int fr_stored, unsigned fc_hz, int K, float *wf);
/* air.c:42-64 (filter == 0) — Airspy tuner centre for the span [min,max] */
unsigned acb_air_choose_fc(unsigned min_hz, unsigned max_hz);
/* air.c:263-285 — wf[i] = cexpf(-j*Ph_i)/AIRMULT with the reference's double phase accumulator */
void acb_air_build_wf(int fr_hz, int fc_hz, unsigned rate, float *wf);
/* soapy.c:159-162 (variant ACB_CS16_SOAPY, with soapy.c:242's /32768.0 folded in) and
 * sdrplay.c:133-137 (ACB_CS16_SDRPLAY, with sdrplay.c:225's /4 folded in): effective mixer tables */
#define ACB_CS16_SOAPY 0
#define ACB_CS16_SDRPLAY 1
void acb_cs16_build_wf(int variant, unsigned freq_hz, unsigned fc_hz, int K, float *wf);
/* Planning step of ACB_FLAG_FAST_CHANNELIZER: returns 1 when every channel's mixer offset (float image
 * of the stored Fr minus float image of Fc, as rtl.c:283 computes it) is a whole, even number k of
 * 12.5 kHz steps with 0 < |k| < K/2; then k_out[ch] = k and tw[(ch*(K/4) + n2)*2 + {0,1}] =
 * exp(-j*2*pi*k*n2/K)/K/127.5.  k_out and tw may be NULL.  Returns 0 otherwise (the exact kernel runs). */
int acb_fast_plan(const unsigned *freqs_hz, int nch, int K, unsigned fc_hz, int *k_out, float *tw);
/* The same for CS16 contexts (soapy.c:159-165 / sdrplay.c:133-137: the offset is (float)Fr - (float)Fc); the twiddles
 * carry the variant's power-of-two scale, exp(-j*2*pi*k*n2/K)/K/32768 (soapy.c:242) or /K/4 (sdrplay.c:225). */
int acb_fast_plan_cs16(int variant, const unsigned *freqs_hz, int nch, int K, unsigned fc_hz, int *k_out, float *tw);
/* The same for real-input contexts (air.c:278-285): k = (Fc - Fr + rate/4)/12500 must be whole, 0 < k < K (any parity: the
 * real form splits the row in quarters only), tw = exp(-j*2*pi*k*n2/K)/K; K a multiple of 8. */
int acb_fast_plan_air(const unsigned *freqs_hz, int nch, int K, unsigned fc_hz, int *k_out, float *tw);
/* msk.c:44-48 — 133-tap oversampled half-cosine matched filter */
void acb_build_h(float *h);

/* ---- context ---- */

int  acb_create(const acb_config_t *cfg, acb_ctx_t **out);
void acb_destroy(acb_ctx_t *ctx);
const char *acb_last_error(void);
const char *acb_version(void);

/* Replaces the channel part of initRtl (rtl.c:243-287) for one stream: freqs in CLI order,
 * chooses Fc, builds and uploads the tables.  fc_out may be NULL. */
int acb_set_plan(acb_ctx_t *ctx, int stream, const unsigned *freqs_hz, int nch, unsigned *fc_out);
/* Same with the centre frequency given (a host that tuned already; a context that serves only SOME of the
 * channels chooseFc planned for — acb_multi_* in channel-split mode, the wide-stream case of SURVEY.md §8e). */
int acb_set_plan_at(acb_ctx_t *ctx, int stream, const unsigned *freqs_hz, int nch, unsigned fc_hz);
/* The channel part of initAirspy (air.c:165-285) for a real-input context. */
int acb_set_plan_air(acb_ctx_t *ctx, int stream, const unsigned *freqs_hz, int nch, unsigned *fc_out);
/* The channel part of initSoapy (soapy.c:112-163) / initSdrplay (sdrplay.c:95-138) for a CS16
 * context; fc_hz = 0 lets chooseFc pick the centre (soapy.c:132-133 honours a user frequency). */
int acb_set_plan_cs16(acb_ctx_t *ctx, int stream, const unsigned *freqs_hz, int nch, int variant, unsigned fc_hz, unsigned *fc_out);
/* Same, with caller-supplied tables (nch x 2K floats), e.g. taken from channel[].wf. */
int acb_set_wf(acb_ctx_t *ctx, int stream, const float *wf, int nch);
/* initMsk + initAcars for every channel of every stream (msk.c:30-51, acars.c:230-234). */
int acb_reset(acb_ctx_t *ctx);

/* ---- processing ---- */

/* Replaces in_callback (rtl.c:314-361) for all streams at once.  Stream s's input is
 * `nblk` consecutive blocks of 1024*K*2 bytes (interleaved u8 I,Q) at iq + s*stream_stride.
 * Asynchronous: host->device copy, channelizer and demod are queued; call acb_sync to
 * collect.  `iq` should come from acb_host_alloc (pinned) for full PCIe overlap. */
int acb_submit_host(acb_ctx_t *ctx, const uint8_t *iq, size_t stream_stride, int nblk);
/* Same with the input already resident in device memory (no copy).
 * Input lifetime, both calls: up to three submits are in flight; when submit N+2 returns, the input of submit N
 * (the host buffer, or the device buffer) has been read and may be overwritten — as it may after an acb_collect /
 * acb_sync that covered submit N. */
int acb_submit_device(acb_ctx_t *ctx, const uint8_t *iq_dev, size_t stream_stride, int nblk);
/* Replaces rx_callback (air.c:291-341): `nsamples` float32 real samples per stream (stream s at
 * x + s*stream_stride_samples), ANY count per call — what does not fill a K-sample output row is
 * carried to the next call, the equivalent of the reference's carried partial sum ch->D / ind.
 * Returns the number of envelope samples produced per channel (>= 0) or a negative error. */
int acb_submit_real_host(acb_ctx_t *ctx, const float *x, size_t stream_stride_samples, size_t nsamples);
/* Replaces the channelizer loops of soapy.c:232-254 (interleaved CS16) and sdrplay.c:215-236
 * (planar xi/xq): `nsamples` complex int16 samples per stream, any count per call, remainder
 * carried (the reference carries ch->D and the tap index).  Returns envelope samples produced. */
int acb_submit_cs16_host(acb_ctx_t *ctx, const int16_t *iq, size_t stream_stride_samples, size_t nsamples);
int acb_submit_cs16_planar_host(acb_ctx_t *ctx, const int16_t *xi, const int16_t *xq, size_t stream_stride_samples, size_t nsamples);
/* Emission order of the streaming front-ends (SURVEY H5).  The reference runs demodMSK channel by channel on
 * whatever a transfer (air.c:336) or a full dm_buffer (soapy.c:247: 1024 outputs; sdrplay.c:229: 512) delivered, so
 * its messages leave in (group, channel, time) order.  A submit may carry many such groups; tell the context how
 * they are cut and acb_sync / acb_collect queue the frames in the reference's order.  A submit boundary always acts
 * as a group boundary too (a submit's frames are queued when it is collected, never held back for the next one), so
 * the order is exactly the reference's when every submit ends on a group boundary; a submit that ends inside a
 * group splits it in two.  A frame belongs to the group holding its completion sample (msg.pos), first and last
 * samples included:
 *   ACB_GROUP_SUBMIT   one group per submit call (default);
 *   ACB_GROUP_OUTPUTS  a group every `period` envelope samples, counted from the start of the stream;
 *   ACB_GROUP_INPUT    a group per transfer of `period` input samples, counted from the start of the stream.
 * (u8 IQ contexts always group per 1024-sample block, rtl.c:357-360.) */
enum { ACB_GROUP_SUBMIT = 0, ACB_GROUP_OUTPUTS = 1, ACB_GROUP_INPUT = 2 };
int acb_set_emission_groups(acb_ctx_t *ctx, int unit, uint64_t period);
/* Replaces demodMSK's input side (msk.c:67; soundfile.c:71-77): 12.5 kS/s envelope samples,
 * dm[(s*nsamp + n)*nch + c], fed straight to the demodulator (no channelizer). */
int acb_submit_dm_host(acb_ctx_t *ctx, const float *dm, int nsamp);
/* Order the next acb_submit_device behind work of ANOTHER CUDA stream: `cuda_event` is a cudaEvent_t recorded there
 * (e.g. behind the NCCL broadcast that fills the input buffer; torch.cuda.Event.cuda_event).  No host sync. */
int acb_wait_event(acb_ctx_t *ctx, void *cuda_event);
/* Wait for the OLDEST submit still in flight only (at most three are), run the block FEC on its
 * frames and queue the survivors; later submits keep running.  This is what lets the H2D copy
 * of step i+1 overlap the kernels of step i.  Returns the number of messages waiting. */
int acb_collect(acb_ctx_t *ctx);
/* Wait for everything queued, run the block FEC (blk_thread, acars.c:93-215) on what the
 * device decoded, and append the survivors to the output queue in the reference's emission
 * order (block-major, then stream, then channel, then time; rtl.c:357-360).
 * Returns the number of messages waiting, or a negative error. */
int acb_sync(acb_ctx_t *ctx);
/* Pop up to `max` messages from the output queue (the outputmsg() feed, acars.c:209). */
int acb_drain(acb_ctx_t *ctx, acb_msg_t *out, int max);
/* Messages currently waiting in the output queue. */
int acb_pending(acb_ctx_t *ctx);

/* Pinned host memory for submit_host callers. */
void *acb_host_alloc(size_t bytes);
void  acb_host_free(void *p);
/* Device memory for submit_device callers (benchmarks keep the input resident in HBM). */
void *acb_device_alloc(acb_ctx_t *ctx, size_t bytes);
void  acb_device_free(acb_ctx_t *ctx, void *p);
int   acb_copy_to_device(acb_ctx_t *ctx, void *dst_dev, const void *src_host, size_t bytes);

/* ---- inspection (parity tests, the compat shim, bench instrumentation) ---- */

/* Tolerance of what these return (default, exact channelizer): envelope samples and messages are bit-identical to the
 * reference's; the demodulator state is bit-identical on every fixture of the test suite, and structurally within 1 ulp of
 * a float ring entry with probability ~2^-29 per sample (the device's VCO sincos is a 1.7-ulp table evaluation, glibc's is
 * 0.52 ulp, and the product is rounded to float, msk.c:90) — far inside the stated bar of 1e-5 relative.  With
 * ACB_FLAG_FAST_CHANNELIZER: messages identical, intermediates as documented in DESIGN.md §2. */
/* Envelope samples the channelizer produced for the last submit: out[(s*nsamp+n)*nch + c]. */
int acb_read_dm(acb_ctx_t *ctx, float *out, size_t nfloats);
int acb_get_state(acb_ctx_t *ctx, int stream, int chn, acb_chan_state_t *out);
int acb_set_state(acb_ctx_t *ctx, int stream, int chn, const acb_chan_state_t *in);

/* CUDA-event stopwatch on the context's compute stream (the stream the kernels run on):
 * acb_mark(ctx,0) ... submits ... acb_mark(ctx,1); acb_elapsed_ms waits for mark 1. */
int acb_mark(acb_ctx_t *ctx, int which);
int acb_elapsed_ms(acb_ctx_t *ctx, float *ms);

typedef struct {
	uint64_t submits;           /* submit calls */
	uint64_t kernel_launches;   /* CUDA kernels launched by this context */
	uint64_t blocks;            /* stream-blocks processed */
	uint64_t raw_frames;        /* frames handed from the device to the FEC */
	uint64_t fec_dropped;       /* frames the FEC rejected */
	double   chan_ms;           /* accumulated device time of the channelizer kernel (CUDA events) */
	double   demod_ms;          /* accumulated device time from a demod kernel's start to the end of its block FEC */
	uint64_t chan_launches, demod_launches;
	uint64_t fast_chan_launches; /* channelizer launches that took the ACB_FLAG_FAST_CHANNELIZER form */
	uint64_t frames_lost;       /* frames that found the device ring full (ACB_ERR_OVERFLOW was returned once per submit) */
	double   host_ms;           /* accumulated wall time the consumer thread spent ordering and queuing frames */
} acb_stats_t;
int acb_get_stats(acb_ctx_t *ctx, acb_stats_t *out, int reset);

/* ---- one process, several GPUs (the C host's way to a whole node; SURVEY.md §8e) ----
 *
 * acb_multi_* fronts one context per device.  Two ways to cut the work, neither with any device-to-device
 * traffic (channels and streams share nothing):
 *   ACB_MULTI_SPLIT_STREAMS   device d serves a contiguous range of the streams (BASELINE config 4);
 *   ACB_MULTI_SPLIT_CHANNELS  every device sees every stream and serves a contiguous range of its channels
 *                             (one wide stream, configs 3/5); each device fetches the block over its own PCIe link.
 * Stream / channel indices in the API and in the messages are global; messages are merged into the reference's
 * emission order (block, stream, channel, time; rtl.c:357-360).  cfg->device is ignored, `devices` names the
 * CUDA ordinals (repeats allowed: two contexts on one GPU). */
typedef struct acb_multi acb_multi_t;
enum { ACB_MULTI_SPLIT_STREAMS = 0, ACB_MULTI_SPLIT_CHANNELS = 1 };
int  acb_multi_create(const acb_config_t *cfg, const int *devices, int ndev, int mode, acb_multi_t **out);
void acb_multi_destroy(acb_multi_t *m);
int  acb_multi_parts(acb_multi_t *m);                        /* number of per-device contexts */
acb_ctx_t *acb_multi_part(acb_multi_t *m, int i);            /* the i-th one (stats, inspection) */
int  acb_multi_set_plan(acb_multi_t *m, int stream, const unsigned *freqs_hz, int nch, unsigned *fc_out);
int  acb_multi_set_wf(acb_multi_t *m, int stream, const float *wf, int nch);
int  acb_multi_reset(acb_multi_t *m);
int  acb_multi_submit_host(acb_multi_t *m, const uint8_t *iq, size_t stream_stride, int nblk);
int  acb_multi_collect(acb_multi_t *m);
int  acb_multi_sync(acb_multi_t *m);
int  acb_multi_drain(acb_multi_t *m, acb_msg_t *out, int max);
int  acb_multi_get_state(acb_multi_t *m, int stream, int chn, acb_chan_state_t *out);
int  acb_multi_set_state(acb_multi_t *m, int stream, int chn, const acb_chan_state_t *in);

/* Block FEC on one frame in place on the HOST (acars.c:123-207): 1 = deliver, 0 = drop.  The
 * processing path runs the same repair on the device (k_block_fec, one thread per frame, right
 * behind the demod); this entry serves the shim's host-side decodeAcars and callers with their own
 * queue. */
int acb_block_fec(acb_msg_t *m);
/* The device block FEC on a batch of raw frames (len, txt with parity bits, crc): repairs msgs[i]
 * in place, keep[i] = 1 where the reference would call outputmsg().  Returns the number kept. */
int acb_block_fec_batch(acb_ctx_t *ctx, acb_msg_t *msgs, int n, int *keep);
/* Tables behind it, generated rather than stored (syndrom.h:4-13, 15-49, 52-295). */
uint16_t acb_crc_update(uint16_t crc, uint8_t c);
uint16_t acb_syndrome(int index);      /* index = bit + 8*bytes_from_end, 0..1935 */

/* The bit/byte frame synchroniser (decodeAcars, acars.c:246-375) as a host call, over caller-owned
 * state: the same definition (csrc/frame_sm.h) the demod kernel runs per channel on the device.
 * Used by the compat shim's decodeAcars(channel_t*).  Integer-only. */
typedef struct {
	int *state, *nbits, *bitcount, *blk_len, *blk_err;
	unsigned *msk_s;
	double *msk_df, *lvlsum;
	unsigned char *txt;                 /* >= 250 bytes */
	unsigned char *crc;                 /* 2 bytes */
	int (*frame_begin)(void *user);     /* SOH seen; return 0 to refuse (no storage) */
	void (*frame_emit)(void *user);     /* frame complete */
	void *user;
} acb_frame_view_t;
void acb_frame_byte(acb_frame_view_t *v, unsigned char r);

#ifdef __cplusplus
}
#endif
#endif
