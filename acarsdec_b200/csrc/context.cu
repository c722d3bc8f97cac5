/*
 * libacars_b200 context: device memory, streams, submit/sync/drain (C ABI in include/acars_b200.h).
 *
 * Replaces, for N streams x C channels at once, what the reference does per RTL block on its
 * input thread (in_callback rtl.c:314-361 -> demodMSK msk.c:67 -> decodeAcars acars.c:246) and
 * on its blk_thread (acars.c:93-215).  Data flow per submit:
 *
 *   host u8 IQ --copy stream--> d_iq[buf] --channelizer stream--> K1 k_channelize -> d_dm[b] (HBM)
 *                                           --demod stream-------> K2 k_demod    -> frame ring[b]
 *                                           --FEC stream---------> K3 k_block_fec on ring[b], frame count -> host
 *   K2 of submit i (latency bound: one serial recurrence per channel) runs concurrently with K1
 *   of submits i+1, i+2; envelope buffers and frame rings come in threes (NPIPE) between them.
 *   acb_collect / acb_sync: D2H of that submit's frames -> consumer thread -> output queue
 *
 * Up to three submits are in flight: input staging is double-buffered, so the H2D copy of submit i+1
 * overlaps the kernels of i, and the read-back of i overlaps the kernels of i+1 and i+2.
 * The frames of a finished submit are sorted into emission order and queued by a CONSUMER THREAD (the role of the
 * reference's blk_thread, acars.c:93-215, minus the FEC, which runs on the device): at a Tsample/s a step carries tens
 * of thousands of messages, and that per-message host work must not sit between two launches.
 */
#include <cuda_runtime.h>
#include <math.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <chrono>
#include <condition_variable>
#include <deque>
#include <memory>
#include <mutex>
#include <system_error>
#include <thread>
#include <vector>

#include "../../include/acars_b200.h"
#include "acb_internal.h"

using namespace acb;

extern "C" void acb_build_sincos_table(double *cos_hi_lo, double *sin_hi_lo);

static thread_local char g_err[512] = "";

static int fail(int code, const char *fmt, ...)
{
	va_list ap;
	va_start(ap, fmt);
	vsnprintf(g_err, sizeof(g_err), fmt, ap);
	va_end(ap);
	return code;
}

#define CU(call)                                                                                   \
	do {                                                                                           \
		cudaError_t e_ = (call);                                                                   \
		if (e_ != cudaSuccess)                                                                     \
			return fail(ACB_ERR_CUDA, "%s: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); \
	} while (0)

extern "C" const char *acb_last_error(void) { return g_err; }
extern "C" const char *acb_version(void) { return "acars_b200 0.1 (sm_100a)"; }

struct EvTriple { cudaEvent_t a, b, b2, c; bool chan; };   /* a..b = K1 on s_comp, b2 = K2 starts on s_dem, c = block FEC done on s_fec */

/* Submits in flight = envelope buffers = frame rings.  Three, not two: with two, the host may queue the channelizer of
 * submit N+2 only once the demod of submit N has finished (it reuses that submit's buffers), so every step ended with the
 * demod running alone and began with both kernels starting together; with three the channelizer of N+2 is already queued
 * behind that of N+1 and both kernels run back to back on their streams (profiles/r2_notes.md: pipeline depth). */
constexpr int NPIPE = 3;

/* one submit in flight: which frame ring it appends to and how its frames are grouped */
struct Ticket {
	EvTriple ev;                                   /* a..b = channelizer, b..c = demod; c = done */
	int ring;
	std::vector<unsigned long long> group_starts;  /* emission-order groups (input blocks / chunks) */
};

struct acb_ctx {
	acb_config_t cfg;
	int ngrp;
	size_t blk_bytes;            /* 1024*K*2 */
	cudaStream_t s_copy, s_comp, s_dem, s_fec;   /* H2D copies | channelizer (K1) | demod (K2) | block FEC (K3) + its count read-back */
	uint8_t *d_iq[2];
	cudaEvent_t ev_copied[2], ev_consumed[2];
	bool buf_used[2];
	int next_buf;
	float *d_wf4;                /* [stream][grp][K][8] float2 (c, d), every input kind */
	bool fast;                   /* ACB_FLAG_FAST_CHANNELIZER and a shape k_channelize_dft takes */
	bool fold8;                  /* fast form: fold the row in half first (8-way split, K/8 MACs per channel) */
	int demod_lanes;             /* lanes per channel in k_demod: 8 for small contexts, else 4 */
	float *d_tw;                 /* fast form: [stream][grp][8 ch][K/4] (Tr, Ti) twiddles */
	unsigned *d_twmeta;          /* fast form: [stream][grp] residues k_c mod 4, 2 bits per channel slot */
	std::vector<unsigned char> fast_ok;   /* per stream: planned on the 12.5 kHz raster (0 after acb_set_wf: caller's own table) */
	float *d_dm[NPIPE];          /* [stream][nsamp][nch], one per submit in flight */
	cudaEvent_t ev_k1_done[NPIPE], ev_dm_free[NPIPE], ev_k2_done[NPIPE], ev_ring_read[NPIPE];
	bool ring_read_pending[NPIPE];
	bool dm_used[NPIPE];
	bool k1_pending[NPIPE];      /* ev_k1_done[b] recorded and not yet waited for by the host */
	int last_dm;
	size_t dm_floats;
	ChainState *d_state;
	cudaStream_t s_d2h;
	RawFrame *d_ring[NPIPE];     /* frame rings, one per submit in flight so that one can be read
	                                back while the next submits' demods append to the others */
	RingCtl *d_ctl[NPIPE];
	unsigned ring_cap;
	RawFrame *h_ring[NPIPE];     /* pinned, one per frame ring: the consumer may still read one while the next lands in another */
	RingCtl *h_ctl[NPIPE];       /* pinned */
	int last_nsamp;
	unsigned long long nsubmit;
	unsigned long long pos;      /* envelope samples submitted so far (all chains move together) */
	std::deque<Ticket> inflight; /* oldest first; at most NPIPE */
	/* output queue: one batch per harvested submit, already in emission order; drained by bulk copies (at a
	 * Tsample/s a step carries tens of thousands of messages: per-message queue operations were the host's
	 * largest cost) */
	struct Batch { std::unique_ptr<acb_msg_t[]> v; size_t n, rd; };
	std::deque<Batch> outq;
	size_t outq_count;
	/* consumer thread: everything from `outq` to `jobs_done`, plus stats.raw_frames / fec_dropped, is guarded by mtx */
	struct Job { std::vector<unsigned long long> group_starts; int ring; unsigned count; };
	std::thread consumer;
	std::mutex mtx;
	std::condition_variable cv_job, cv_done;
	std::deque<Job> jobs;
	bool stop;
	unsigned long long jobs_queued, jobs_done, ring_job[NPIPE];   /* ring_job[b]: sequence number of the last job reading h_ring[b] */
	char consumer_err[256];
	std::vector<EvTriple> ev_free;
	cudaEvent_t mark[2], ev_join;
	bool overflowed;
	acb_stats_t stats;
	bool use_generic;
	int taps;                    /* FIR length actually applied per output row (<= K) */
	int taps_pad;                /* taps rounded up to whole 16-byte units of input (zero weights) */
	int in_kind;                 /* IN_KIND_*: u8 IQ blocks | float32 real (air.c) | CS16 IQ (soapy.c, sdrplay.c) */
	bool real_input;             /* in_kind != u8: 4-byte input elements, arbitrary submit lengths, carried remainder */
	float *d_real[2];            /* per stream: [carry + new samples], alternating per submit */
	size_t real_cap;             /* floats per stream in d_real */
	size_t carry;                /* samples of every stream not yet consumed (< K) */
	int real_buf;
	cudaEvent_t ev_real_copied, ev_real_free[2];   /* H2D of a streaming submit landed | d_real[b] may be overwritten */
	bool real_used[2];
	int16_t *d_planar;           /* CS16 planar input: both planes of one submit, interleaved on the device */
	size_t planar_cap;           /* int16 elements per plane and stream */
	int group_unit;              /* ACB_GROUP_*: how the streaming front-ends' frames are grouped for emission */
	unsigned long long group_period;
};

static void consumer_main(acb_ctx *c);
static void wait_consumer(acb_ctx *c, unsigned long long seq);

static int ctx_use(acb_ctx *c)
{
	CU(cudaSetDevice(c->cfg.device));
	return ACB_OK;
}

/* Host -> device upload that is complete when it returns.  A plain cudaMemcpy from pageable memory may
 * return once the data is staged, before the DMA has landed, and the context's streams are non-blocking
 * (not ordered behind the legacy stream): a kernel launched right after could read the old contents. */
static int upload(acb_ctx *c, void *dst, const void *src, size_t bytes)
{
	CU(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, c->s_copy));
	CU(cudaStreamSynchronize(c->s_copy));
	return ACB_OK;
}

extern "C" void *acb_host_alloc(size_t bytes)
{
	void *p = nullptr;
	if (cudaHostAlloc(&p, bytes, cudaHostAllocDefault) != cudaSuccess) {
		fail(ACB_ERR_CUDA, "cudaHostAlloc(%zu) failed", bytes);
		return nullptr;
	}
	return p;
}
extern "C" void acb_host_free(void *p) { if (p) cudaFreeHost(p); }

extern "C" void *acb_device_alloc(acb_ctx_t *c, size_t bytes)
{
	void *p = nullptr;
	if (!c || ctx_use(c)) return nullptr;
	if (cudaMalloc(&p, bytes) != cudaSuccess) {
		fail(ACB_ERR_NOMEM, "cudaMalloc(%zu) failed", bytes);
		return nullptr;
	}
	return p;
}
extern "C" void acb_device_free(acb_ctx_t *c, void *p) { if (c && p && !ctx_use(c)) cudaFree(p); }

extern "C" int acb_copy_to_device(acb_ctx_t *c, void *dst, const void *src, size_t bytes)
{
	if (!c) return fail(ACB_ERR_ARG, "null context");
	if (int r = ctx_use(c)) return r;
	return upload(c, dst, src, bytes);
}

static int sync_streams(acb_ctx *c)
{
	CU(cudaStreamSynchronize(c->s_comp));
	CU(cudaStreamSynchronize(c->s_dem));
	CU(cudaStreamSynchronize(c->s_fec));
	return ACB_OK;
}

static int reset_states(acb_ctx *c)
{
	const size_t n = (size_t)c->cfg.nstreams * c->cfg.nch;
	std::vector<ChainState> init(n);
	memset(init.data(), 0, n * sizeof(ChainState));
	for (auto &s : init) {       /* initMsk msk.c:34-40 zeroes; initAcars acars.c:230-234 */
		s.nbits = 8;
		s.state = 0;             /* WSYN */
	}
	/* everything stream-ordered on s_copy and complete on return: the context's streams are non-blocking,
	 * so nothing on the legacy stream (plain cudaMemset/cudaMemcpy) is ordered against them */
	if (int r = upload(c, c->d_state, init.data(), n * sizeof(ChainState))) return r;
	for (int i = 0; i < NPIPE; i++) CU(cudaMemsetAsync(c->d_ctl[i], 0, sizeof(RingCtl), c->s_copy));
	CU(cudaStreamSynchronize(c->s_copy));
	c->pos = 0;
	c->carry = 0;
	{
		std::lock_guard<std::mutex> lk(c->mtx);
		c->outq.clear();
		c->outq_count = 0;
	}
	c->overflowed = false;
	return ACB_OK;
}

extern "C" int acb_create(const acb_config_t *cfg, acb_ctx_t **out)
{
	if (!cfg || !out) return fail(ACB_ERR_ARG, "null argument");
	if (cfg->K < 1 || cfg->K > ACB_MAXK) return fail(ACB_ERR_ARG, "K=%d out of range 1..%d", cfg->K, ACB_MAXK);
	if (cfg->nstreams < 1 || cfg->nch < 1 || cfg->max_blocks < 1) return fail(ACB_ERR_ARG, "nstreams/nch/max_blocks must be >= 1");
	if (cfg->taps < 0 || cfg->taps > cfg->K) return fail(ACB_ERR_ARG, "taps=%d must be 0 (= K) or 1..K=%d", cfg->taps, cfg->K);
	if ((cfg->flags & ACB_FLAG_REAL_INPUT) && (cfg->flags & ACB_FLAG_CS16_INPUT)) return fail(ACB_ERR_ARG, "REAL_INPUT and CS16_INPUT are exclusive");
	int ndev = 0;
	if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
		return fail(ACB_ERR_CUDA, "no CUDA device: libacars_b200 has no CPU fallback");
	if (cfg->device < 0 || cfg->device >= ndev) return fail(ACB_ERR_ARG, "device %d of %d", cfg->device, ndev);
	CU(cudaSetDevice(cfg->device));
	cudaDeviceProp prop;
	CU(cudaGetDeviceProperties(&prop, cfg->device));
	if (prop.major != 10)
		return fail(ACB_ERR_CUDA, "device %d is sm_%d%d; this library carries sm_100a code only", cfg->device, prop.major, prop.minor);

	acb_ctx *c = new acb_ctx();
	c->cfg = *cfg;
	c->ngrp = (cfg->nch + CH_GROUP - 1) / CH_GROUP;
	c->blk_bytes = (size_t)OUTBLK * cfg->K * 2;
	c->in_kind = (cfg->flags & ACB_FLAG_REAL_INPUT) ? IN_KIND_F32REAL : (cfg->flags & ACB_FLAG_CS16_INPUT) ? IN_KIND_CS16IQ : IN_KIND_U8IQ;
	c->real_input = c->in_kind != IN_KIND_U8IQ;
	c->use_generic = c->real_input ? (cfg->K % 4) != 0 : (cfg->K % 8) != 0;
	c->taps = cfg->taps ? cfg->taps : cfg->K;
	{
		const int per_unit = c->real_input ? 4 : 8;          /* taps per 16 bytes of input (4-byte vs 2-byte taps) */
		c->taps_pad = c->use_generic ? c->taps : (c->taps + per_unit - 1) / per_unit * per_unit;
		if (c->taps_pad > cfg->K) c->taps_pad = cfg->K;      /* K itself is a multiple of per_unit here */
	}
	c->d_real[0] = c->d_real[1] = nullptr;
	c->d_planar = nullptr;
	c->planar_cap = 0;
	c->ev_real_copied = nullptr;
	c->ev_real_free[0] = c->ev_real_free[1] = nullptr;
	c->carry = 0;
	c->real_buf = 0;
	c->group_unit = ACB_GROUP_SUBMIT;
	c->group_period = 0;
	c->next_buf = 0;
	c->last_nsamp = 0;
	c->nsubmit = 0;
	c->outq_count = 0;
	c->stop = false;
	c->jobs_queued = c->jobs_done = 0;
	c->ring_job[0] = c->ring_job[1] = 0;
	c->consumer_err[0] = 0;
	c->h_ring[0] = c->h_ring[1] = nullptr;
	c->overflowed = false;
	memset(&c->stats, 0, sizeof(c->stats));
	*out = c;

	CU(cudaStreamCreateWithFlags(&c->s_copy, cudaStreamNonBlocking));
	CU(cudaStreamCreateWithFlags(&c->s_comp, cudaStreamNonBlocking));
	CU(cudaStreamCreateWithFlags(&c->s_dem, cudaStreamNonBlocking));
	CU(cudaStreamCreateWithFlags(&c->s_fec, cudaStreamNonBlocking));
	CU(cudaEventCreateWithFlags(&c->ev_join, cudaEventDisableTiming));
	CU(cudaStreamCreateWithFlags(&c->s_d2h, cudaStreamNonBlocking));
	CU(cudaEventCreate(&c->mark[0]));
	CU(cudaEventCreate(&c->mark[1]));
	const size_t in_bytes = (size_t)cfg->nstreams * cfg->max_blocks * c->blk_bytes;
	for (int i = 0; i < 2; i++) {
		c->d_iq[i] = nullptr;
		c->buf_used[i] = false;
		if (!(cfg->flags & ACB_FLAG_NO_INPUT_STAGING) && !c->real_input) CU(cudaMalloc(&c->d_iq[i], in_bytes));
		if (c->real_input) {
			/* room for the carried remainder (< K) plus one submit, rounded so streams stay 32-B aligned */
			c->real_cap = (((size_t)cfg->max_blocks * OUTBLK + 1) * cfg->K + 7) & ~(size_t)7;     /* streams 32-B aligned: whole sectors per chunk */
			/* + 32 rows: the fast CS16 / real-input kernels fetch whole tiles of up to 32 rows, the last one may reach past the last row */
			CU(cudaMalloc(&c->d_real[i], ((size_t)cfg->nstreams * c->real_cap + 32 * (size_t)cfg->K) * sizeof(float)));
			CU(cudaEventCreateWithFlags(&c->ev_real_free[i], cudaEventDisableTiming));
			c->real_used[i] = false;
		}
		CU(cudaEventCreateWithFlags(&c->ev_copied[i], cudaEventDisableTiming));
		CU(cudaEventCreateWithFlags(&c->ev_consumed[i], cudaEventDisableTiming));
	}
	if (c->real_input) CU(cudaEventCreateWithFlags(&c->ev_real_copied, cudaEventDisableTiming));
	const size_t wf_floats = (size_t)cfg->nstreams * c->ngrp * c->taps_pad * CH_GROUP * 2;
	CU(cudaMalloc(&c->d_wf4, wf_floats * sizeof(float)));
	CU(cudaMemsetAsync(c->d_wf4, 0, wf_floats * sizeof(float), c->s_copy));
	CU(cudaStreamSynchronize(c->s_copy));
	c->fast = (cfg->flags & ACB_FLAG_FAST_CHANNELIZER) && c->taps == cfg->K &&
	          (c->in_kind == IN_KIND_F32REAL ? channelize_rdft_supports(cfg->K) : channelize_dft_supports(cfg->K));
	c->fast_ok.assign(cfg->nstreams, 0);
	c->fold8 = true;             /* 0.89 ms vs 0.95 ms for the plain 4-way split at 592 streams x 16 blocks */
	if (const char *e = getenv("ACB_FAST_FOLD8")) c->fold8 = atoi(e) != 0;          /* comparison switch; both are tested */
	{
		/* 8 lanes per channel halve the mixer's share of the serial chain but double the warps: a gain (8 % on
		 * one 8-channel stream) only while there is still at most one demod warp per SM sub-partition;
		 * beyond that the extra warps cost more than they hide (592 streams: 4.54 -> 4.72 ms) */
		c->demod_lanes = demod_pick_lanes((long long)cfg->nstreams * cfg->nch, prop.multiProcessorCount);
		/* comparison switch (tests force every width; tools/ab_demod.py sweeps it): 1, 2, 4, 8 lanes per channel,
		 * +16 = F2F bit-clock rounding, +32 = constants not pinned, -4 / -8 = the round-1 kernel (launch_demod) */
		if (const char *e = getenv("ACB_DEMOD_LANES")) {
			const int v = atoi(e), l = v & 15;
			if (v == -4 || v == -8 || (v > 0 && v < 64 && (l == 1 || l == 2 || l == 4 || l == 8))) c->demod_lanes = v;
		}
	}
	if (c->fast) {
		CU(cudaMalloc(&c->d_tw, (size_t)cfg->nstreams * c->ngrp * CH_GROUP * (cfg->K / 4) * 2 * sizeof(float)));
		CU(cudaMalloc(&c->d_twmeta, (size_t)cfg->nstreams * c->ngrp * sizeof(unsigned)));
	}
	c->dm_floats = (size_t)cfg->nstreams * cfg->max_blocks * OUTBLK * cfg->nch;
	for (int i = 0; i < NPIPE; i++) {
		CU(cudaMalloc(&c->d_dm[i], c->dm_floats * sizeof(float)));
		CU(cudaEventCreateWithFlags(&c->ev_k1_done[i], cudaEventDisableTiming));
		CU(cudaEventCreateWithFlags(&c->ev_dm_free[i], cudaEventDisableTiming));
		CU(cudaEventCreateWithFlags(&c->ev_k2_done[i], cudaEventDisableTiming));
		CU(cudaEventCreateWithFlags(&c->ev_ring_read[i], cudaEventDisableTiming));
		c->ring_read_pending[i] = false;
		c->dm_used[i] = false;
		c->k1_pending[i] = false;
	}
	c->last_dm = 0;
	const size_t nchain = (size_t)cfg->nstreams * cfg->nch;
	CU(cudaMalloc(&c->d_state, nchain * sizeof(ChainState)));
	/* Frames of fewer than 13 text bytes never take a slot (emit_frame drops them like blk_thread does,
	 * acars.c:124-129).  The shortest frame that does is SYN SYN SOH + 13 + BCS(2) + the byte the END
	 * state swallows = 19 bytes = 152 bits = 791 envelope samples (frame_sm.h), so a chain finishes
	 * < 1.3 per 1024-sample block: 2 per block (+4 for the ends of the submit) cannot be overrun */
	size_t cap = nchain * (2 * (size_t)cfg->max_blocks + 4);
	if (cap > (1u << 22)) cap = 1u << 22;
	c->ring_cap = (unsigned)cap;
	for (int i = 0; i < NPIPE; i++) {
		CU(cudaMalloc(&c->d_ring[i], cap * sizeof(RawFrame)));
		CU(cudaMalloc(&c->d_ctl[i], sizeof(RingCtl)));
		CU(cudaHostAlloc(&c->h_ctl[i], sizeof(RingCtl), cudaHostAllocDefault));
	}
	for (int i = 0; i < NPIPE; i++) CU(cudaHostAlloc(&c->h_ring[i], cap * sizeof(RawFrame), cudaHostAllocDefault));
	c->consumer = std::thread(consumer_main, c);

	float h[FLENO];
	acb_build_h(h);
	CU((cudaError_t)upload_matched_filter(h, c->s_copy));
	{
		double tc[128], ts[128];
		acb_build_sincos_table(tc, ts);             /* hostmath.cpp */
		CU((cudaError_t)upload_sincos_table(tc, ts, c->s_copy));
	}
	if (int r = reset_states(c)) return r;
	return ACB_OK;
}

extern "C" void acb_destroy(acb_ctx_t *c)
{
	if (!c) return;
	if (c->consumer.joinable()) {
		{
			std::lock_guard<std::mutex> lk(c->mtx);
			c->stop = true;
		}
		c->cv_job.notify_all();
		c->consumer.join();
	}
	if (ctx_use(c) == ACB_OK) {
		cudaDeviceSynchronize();
		for (int i = 0; i < 2; i++) {
			if (c->d_iq[i]) cudaFree(c->d_iq[i]);
			if (c->d_real[i]) cudaFree(c->d_real[i]);
			if (c->ev_real_free[i]) cudaEventDestroy(c->ev_real_free[i]);
			cudaEventDestroy(c->ev_copied[i]);
			cudaEventDestroy(c->ev_consumed[i]);
		}
		for (auto &t : c->inflight) { cudaEventDestroy(t.ev.a); cudaEventDestroy(t.ev.b); cudaEventDestroy(t.ev.b2); cudaEventDestroy(t.ev.c); }
		for (auto &e : c->ev_free) { cudaEventDestroy(e.a); cudaEventDestroy(e.b); cudaEventDestroy(e.b2); cudaEventDestroy(e.c); }
		if (c->ev_real_copied) cudaEventDestroy(c->ev_real_copied);
		cudaFree(c->d_planar);
		cudaFree(c->d_wf4); cudaFree(c->d_state);
		cudaFree(c->d_tw); cudaFree(c->d_twmeta);
		for (int i = 0; i < NPIPE; i++) {
			cudaFree(c->d_dm[i]); cudaEventDestroy(c->ev_k1_done[i]); cudaEventDestroy(c->ev_dm_free[i]);
			cudaEventDestroy(c->ev_k2_done[i]); cudaEventDestroy(c->ev_ring_read[i]);
			cudaFree(c->d_ring[i]); cudaFree(c->d_ctl[i]); cudaFreeHost(c->h_ctl[i]); cudaFreeHost(c->h_ring[i]);
		}
		cudaEventDestroy(c->mark[0]); cudaEventDestroy(c->mark[1]); cudaEventDestroy(c->ev_join);
		cudaStreamDestroy(c->s_copy); cudaStreamDestroy(c->s_comp); cudaStreamDestroy(c->s_dem); cudaStreamDestroy(c->s_fec); cudaStreamDestroy(c->s_d2h);
	}
	delete c;
}

extern "C" int acb_reset(acb_ctx_t *c)
{
	if (!c) return fail(ACB_ERR_ARG, "null context");
	if (int r = ctx_use(c)) return r;
	CU(cudaDeviceSynchronize());
	wait_consumer(c, c->jobs_queued);
	/* submits still in flight are abandoned with their frames: recycle their events, forget pending reads */
	for (auto &t : c->inflight) c->ev_free.push_back(t.ev);
	c->inflight.clear();
	for (int i = 0; i < NPIPE; i++) c->ring_read_pending[i] = false;
	for (int i = 0; i < NPIPE; i++) c->k1_pending[i] = false;
	return reset_states(c);
}

extern "C" int acb_set_wf(acb_ctx_t *c, int stream, const float *wf, int nch)
{
	if (!c || !wf) return fail(ACB_ERR_ARG, "null argument");
	if (stream < 0 || stream >= c->cfg.nstreams || nch != c->cfg.nch) return fail(ACB_ERR_ARG, "stream/nch mismatch");
	if (int r = ctx_use(c)) return r;
	const int T = c->taps, TP = c->taps_pad;      /* taps beyond T keep zero weights: D + (+0) = D */
	std::vector<float> t((size_t)c->ngrp * TP * CH_GROUP * 2, 0.0f);     /* (c, d) for every input kind */
	for (int ch = 0; ch < nch; ch++) {
		const int g = ch / CH_GROUP, cc = ch % CH_GROUP;
		for (int ind = 0; ind < T; ind++) {
			float *o = &t[(((size_t)g * TP + ind) * CH_GROUP + cc) * 2];
			o[0] = wf[((size_t)ch * T + ind) * 2];
			o[1] = wf[((size_t)ch * T + ind) * 2 + 1];
		}
	}
	if (int r = sync_streams(c)) return r;
	if (int r = upload(c, c->d_wf4 + (size_t)stream * t.size(), t.data(), t.size() * sizeof(float))) return r;
	c->fast_ok[stream] = 0;                     /* a caller's table has no known structure: exact kernel */
	return ACB_OK;
}

/* fast form: group the per-channel twiddles and bin residues the way k_channelize_dft* reads them and upload them;
 * `ok` false (a channel off the raster) leaves the stream on the exact kernel */
static int upload_fast_plan(acb_ctx *c, int stream, bool ok, const std::vector<int> &kbin, const std::vector<float> &tw1)
{
	if (!ok) return ACB_OK;
	const int nch = c->cfg.nch, N2 = c->cfg.K / 4;
	std::vector<float> tw((size_t)c->ngrp * CH_GROUP * N2 * 2, 0.0f);
	std::vector<unsigned> meta(c->ngrp, 0u);
	for (int ch = 0; ch < nch; ch++) {
		const int g = ch / CH_GROUP, cc = ch % CH_GROUP;
		meta[g] |= (unsigned)(((kbin[ch] % 4) + 4) % 4) << (2 * cc);      /* k mod 4: the 4-way split (u8: 0 or 2; real input: any) */
		meta[g] |= (unsigned)((((kbin[ch] / 2) % 4) + 4) % 4) << (16 + 2 * cc);   /* k even: residue of k/2, for the folded form */
		memcpy(&tw[((size_t)g * CH_GROUP + cc) * N2 * 2], &tw1[(size_t)ch * N2 * 2], (size_t)N2 * 2 * sizeof(float));
	}
	if (int r = upload(c, c->d_tw + (size_t)stream * tw.size(), tw.data(), tw.size() * sizeof(float))) return r;
	if (int r = upload(c, c->d_twmeta + (size_t)stream * meta.size(), meta.data(), meta.size() * sizeof(unsigned))) return r;
	c->fast_ok[stream] = 1;
	return ACB_OK;
}

extern "C" int acb_set_plan(acb_ctx_t *c, int stream, const unsigned *freqs_hz, int nch, unsigned *fc_out)
{
	if (!c || !freqs_hz) return fail(ACB_ERR_ARG, "null argument");
	const unsigned fc = acb_choose_fc(freqs_hz, nch, c->cfg.K);
	if (fc == 0) return fail(ACB_ERR_PLAN, "Frequencies too far apart");    /* rtl.c:149-152 */
	if (fc_out) *fc_out = fc;
	return acb_set_plan_at(c, stream, freqs_hz, nch, fc);
}

extern "C" int acb_set_plan_at(acb_ctx_t *c, int stream, const unsigned *freqs_hz, int nch, unsigned fc)
{
	if (!c || !freqs_hz) return fail(ACB_ERR_ARG, "null argument");
	if (nch != c->cfg.nch) return fail(ACB_ERR_ARG, "nch mismatch");
	if (c->real_input) return fail(ACB_ERR_ARG, "not a u8-IQ context: use acb_set_plan_air / acb_set_plan_cs16");
	if (c->taps != c->cfg.K) return fail(ACB_ERR_ARG, "taps != K: the reference planner builds K-tap tables; supply yours with acb_set_wf");
	if (fc == 0) return fail(ACB_ERR_PLAN, "centre frequency 0");
	std::vector<float> wf((size_t)nch * c->cfg.K * 2);
	for (int ch = 0; ch < nch; ch++)
		acb_build_wf(acb_stored_fr(freqs_hz[ch]), fc, c->cfg.K, &wf[(size_t)ch * c->cfg.K * 2]);
	if (int r = acb_set_wf(c, stream, wf.data(), nch)) return r;
	if (!c->fast) return ACB_OK;
	/* Fast form: per-channel bin numbers and twiddles, when every channel sits on the raster */
	const int K = c->cfg.K, N2 = K / 4;
	std::vector<int> kbin(nch);
	std::vector<float> tw1((size_t)nch * N2 * 2);
	const bool ok = acb_fast_plan(freqs_hz, nch, K, fc, kbin.data(), tw1.data()) == 1;
	return upload_fast_plan(c, stream, ok, kbin, tw1);
}

static EvTriple get_events(acb_ctx *c)
{
	EvTriple e;
	if (!c->ev_free.empty()) {
		e = c->ev_free.back();
		c->ev_free.pop_back();
	} else {
		cudaEventCreate(&e.a); cudaEventCreate(&e.b); cudaEventCreate(&e.b2); cudaEventCreate(&e.c);
	}
	return e;
}

/* Collecting a submit has a device half and a host half:
 *   harvest_begin  (submitting thread) waits until its demod kernel is done, reads the frame count, queues the D2H
 *                  copy of its frames (copy stream s_d2h, event ev_ring_read[ring]) and hands the rest to the consumer;
 *   consumer_main  (consumer thread) waits for that copy and queues the frames the device block FEC (k_block_fec, the
 *                  blk_thread role, acars.c:93-215) kept, in the reference's emission order: per input block, channel by
 *                  channel, then time (rtl.c:357-360; soundfile.c:71-77); streams are interleaved as
 *                  if the reference served them in turn.
 * So the host-side sort/copy of submit i-1 never delays the launches of submit i+1; acb_collect / acb_sync wait for the
 * consumer to have caught up with what they collected. */
static void consume(acb_ctx *c, const acb_ctx::Job &job)
{
	const unsigned count = job.count;
	const auto &gs = job.group_starts;
	const RawFrame *ring = c->h_ring[job.ring];
	/* emission order = (group, stream, channel, time).  A chain's frames reach the ring in time order (one thread
	 * appends them as it decodes), so a STABLE bucket pass over (group, chain) is the whole sort: O(frames + buckets)
	 * instead of a comparison sort (at a Tsample/s a step carries ~40 000 frames; std::sort on them was half of the
	 * consumer's time, and the consumer, not the GPU, set the step time of the fast pipeline).  Contexts whose
	 * (groups x chains) table would be unreasonable take the comparison sort. */
	const auto t_begin = std::chrono::steady_clock::now();
	const size_t nchain = (size_t)c->cfg.nstreams * c->cfg.nch, nbucket = (gs.size() + 1) * nchain;
	std::vector<unsigned> order(count);
	std::vector<unsigned char> keep(count);             /* 1 = repaired and parity-stripped on the device (k_block_fec) */
	/* test hooks (tests/test_gpu_parity.py): ACB_CONSUMER_SORT=1 forces the comparison sort, ACB_CONSUMER_HELPERS_MIN=n the
	 * helper threads from n frames on */
	const bool force_sort = getenv("ACB_CONSUMER_SORT") && atoi(getenv("ACB_CONSUMER_SORT")) != 0;
	if (!force_sort && nbucket <= ((size_t)1 << 24)) {
		std::vector<unsigned> start(nbucket + 1, 0u), bucket(count);
		for (unsigned i = 0; i < count; i++) {          /* the one pass in ring order: sequential reads */
			const RawFrame &f = ring[i];
			keep[i] = f.pad0 == 1;
			const size_t g = gs.size() == 1 ? (f.pos >= gs[0]) : (size_t)(std::upper_bound(gs.begin(), gs.end(), f.pos) - gs.begin());
			const size_t bk = g * nchain + (size_t)f.stream * c->cfg.nch + f.chn;
			bucket[i] = (unsigned)bk;
			start[bk + 1]++;
		}
		for (size_t k = 0; k < nbucket; k++) start[k + 1] += start[k];
		for (unsigned i = 0; i < count; i++) order[start[bucket[i]]++] = i;
	} else {
		for (unsigned i = 0; i < count; i++) { order[i] = i; keep[i] = ring[i].pad0 == 1; }
		std::stable_sort(order.begin(), order.end(), [ring, &gs](unsigned ia, unsigned ib) {
			const RawFrame &x = ring[ia], &y = ring[ib];
			const size_t gx = (size_t)(std::upper_bound(gs.begin(), gs.end(), x.pos) - gs.begin());
			const size_t gy = (size_t)(std::upper_bound(gs.begin(), gs.end(), y.pos) - gs.begin());
			if (gx != gy) return gx < gy;
			if (x.stream != y.stream) return x.stream < y.stream;
			if (x.chn != y.chn) return x.chn < y.chn;
			return x.pos < y.pos;
		});
	}
	/* The records.  Frames are read in emission order, i.e. at random from an 11 MB ring when a step carries 40 000 of
	 * them: a cache-miss-bound copy (5 ms on one core, more than the GPU needs for the step).  Output slots are fixed
	 * first (a frame the block FEC rejected takes none), then the copy is cut into contiguous ranges of the output,
	 * one helper thread each for large jobs. */
	std::vector<unsigned> slot(count);
	unsigned kept = 0;
	for (unsigned j = 0; j < count; j++) {
		slot[j] = kept;
		kept += keep[order[j]];
	}
	acb_ctx::Batch b;
	b.v.reset(new acb_msg_t[kept ? kept : 1]);
	b.n = kept;
	b.rd = 0;
	const unsigned dropped = count - kept;
	acb_msg_t *out = b.v.get();
	auto fill = [ring, out, &order, &slot, &keep](unsigned j0, unsigned j1) {
		for (unsigned j = j0; j < j1; j++) {
			if (!keep[order[j]]) continue;
			const RawFrame &f = ring[order[j]];
			acb_msg_t &m = out[slot[j]];
			memset(&m, 0, sizeof(m));
			m.stream = f.stream; m.chn = f.chn; m.len = f.len; m.err = f.err;
			m.lvl = (float)(10 * log10(f.lvlsum / f.bitcount));          /* acars.c:351 */
			m.block = f.pos / OUTBLK; m.pos = f.pos; m.soh_pos = f.soh_pos;
			memcpy(m.txt, f.txt, ACB_TXTMAX);
			m.crc[0] = f.crc[0]; m.crc[1] = f.crc[1];
		}
	};
	const unsigned helpers_min = getenv("ACB_CONSUMER_HELPERS_MIN") ? (unsigned)atoi(getenv("ACB_CONSUMER_HELPERS_MIN")) : 8192u;
	const unsigned helpers = count >= helpers_min ? std::min(3u, std::max(1u, std::thread::hardware_concurrency()) - 1u) : 0u;
	if (helpers == 0) {
		fill(0, count);
	} else {
		std::vector<std::thread> pool;
		const unsigned parts = helpers + 1, per = (count + parts - 1) / parts;
		for (unsigned t = 1; t < parts; t++) {
			const unsigned j0 = std::min(count, t * per), j1 = std::min(count, (t + 1) * per);
			try {
				pool.emplace_back(fill, j0, j1);
			} catch (const std::system_error &) {        /* no thread to be had: this one does the range itself */
				fill(j0, j1);
			}
		}
		fill(0, std::min(count, per));
		for (auto &th : pool) th.join();
	}
	const double ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_begin).count();
	std::lock_guard<std::mutex> lk(c->mtx);
	c->stats.raw_frames += count;
	c->stats.fec_dropped += dropped;
	c->stats.host_ms += ms;
	if (b.n) {
		c->outq_count += b.n;
		c->outq.push_back(std::move(b));
	}
}

static void consumer_main(acb_ctx *c)
{
	cudaSetDevice(c->cfg.device);
	for (;;) {
		acb_ctx::Job job;
		{
			std::unique_lock<std::mutex> lk(c->mtx);
			c->cv_job.wait(lk, [c] { return c->stop || !c->jobs.empty(); });
			if (c->jobs.empty()) return;             /* stop requested and nothing left */
			job = std::move(c->jobs.front());
			c->jobs.pop_front();
		}
		const cudaError_t e = job.count ? cudaEventSynchronize(c->ev_ring_read[job.ring]) : cudaSuccess;
		if (e == cudaSuccess) consume(c, job);
		{
			std::lock_guard<std::mutex> lk(c->mtx);
			if (e != cudaSuccess && !c->consumer_err[0]) snprintf(c->consumer_err, sizeof(c->consumer_err), "frame read-back: %s", cudaGetErrorString(e));
			c->jobs_done++;
		}
		c->cv_done.notify_all();
	}
}

/* block until the consumer has finished job number `seq` (1-based count of jobs queued so far) */
static void wait_consumer(acb_ctx *c, unsigned long long seq)
{
	std::unique_lock<std::mutex> lk(c->mtx);
	c->cv_done.wait(lk, [c, seq] { return c->jobs_done >= seq; });
}

static int harvest_begin(acb_ctx *c)
{
	if (c->inflight.empty()) return ACB_OK;
	Ticket t = std::move(c->inflight.front());
	c->inflight.pop_front();
	CU(cudaEventSynchronize(t.ev.c));           /* the RingCtl read-back was queued before ev.c */
	float ms = 0;
	if (t.ev.chan && cudaEventElapsedTime(&ms, t.ev.a, t.ev.b) == cudaSuccess) c->stats.chan_ms += ms;
	if (cudaEventElapsedTime(&ms, t.ev.b2, t.ev.c) == cudaSuccess) c->stats.demod_ms += ms;
	c->ev_free.push_back(t.ev);
	unsigned count = c->h_ctl[t.ring]->count;
	const unsigned shortf = c->h_ctl[t.ring]->short_frames;     /* dropped on the device like acars.c:124-129 */
	/* h_ring[ring] was last filled two submits ago: the consumer must be done with it */
	wait_consumer(c, c->ring_job[t.ring]);
	{
		std::lock_guard<std::mutex> lk(c->mtx);
		c->stats.raw_frames += shortf;
		c->stats.fec_dropped += shortf;
		if (count > c->ring_cap) {                   /* reported once by the collecting call; decoding goes on */
			c->overflowed = true;
			c->stats.frames_lost += count - c->ring_cap;
			count = c->ring_cap;
		}
	}
	if (count)
		CU(cudaMemcpyAsync(c->h_ring[t.ring], c->d_ring[t.ring], (size_t)count * sizeof(RawFrame), cudaMemcpyDeviceToHost, c->s_d2h));
	CU(cudaEventRecord(c->ev_ring_read[t.ring], c->s_d2h));
	c->ring_read_pending[t.ring] = true;
	{
		std::lock_guard<std::mutex> lk(c->mtx);
		c->jobs.push_back(acb_ctx::Job{ std::move(t.group_starts), t.ring, count });
		c->ring_job[t.ring] = ++c->jobs_queued;
	}
	c->cv_job.notify_one();
	return ACB_OK;
}

/* oldest submit in flight -> output queue, complete on return */
static int collect_oldest(acb_ctx *c)
{
	if (int r = harvest_begin(c)) return r;
	wait_consumer(c, c->jobs_queued);
	if (c->consumer_err[0]) return fail(ACB_ERR_CUDA, "%s", c->consumer_err);
	return ACB_OK;
}

/* queue K1+K2 (or K2 only) on the compute stream for `nblk` blocks / `nsamp` envelope samples */
static int run_kernels(acb_ctx *c, const uint8_t *d_iq, size_t stride, int nblk, int nsamp, const float *dm_host,
                       std::vector<unsigned long long> &&groups)
{
	/* the ring this submit appends to was last used NPIPE submits ago: its frames must be on their
	 * way back before the new demod may clear it — but the host-side work on those frames waits
	 * until the new kernels have been launched */
	while (c->inflight.size() > (size_t)NPIPE)
		if (int r = collect_oldest(c)) return r;
	if (c->inflight.size() == (size_t)NPIPE)
		if (int r = harvest_begin(c)) return r;      /* its frames are the consumer's from here on, whatever happens below */
	/* Input lifetime: when submit N+2 returns, the channelizer of submit N has read its input (host buffer copied,
	 * device buffer consumed) — callers rotating three input buffers, or two with a collect in between, rely on it */
	if (c->nsubmit >= 2) {
		const int b2 = (int)((c->nsubmit - 2) % NPIPE);
		if (c->k1_pending[b2]) {
			CU(cudaEventSynchronize(c->ev_k1_done[b2]));
			c->k1_pending[b2] = false;
		}
	}
	Ticket t;
	t.ring = (int)(c->nsubmit % NPIPE);
	t.group_starts = std::move(groups);
	t.ev = get_events(c);
	t.ev.chan = d_iq != nullptr;
	const int b = t.ring;                          /* envelope buffer and frame ring of this submit */
	float *dmbuf = c->d_dm[b];
	if (d_iq) {
		/* K1 may overwrite d_dm[b] only after the demod of NPIPE submits ago has read it */
		if (c->dm_used[b]) CU(cudaStreamWaitEvent(c->s_comp, c->ev_dm_free[b], 0));
		CU(cudaEventRecord(t.ev.a, c->s_comp));
		int r = 0;
		/* whole 1024-row blocks through the pipeline kernel, the remaining rows (submits of 4-byte
		 * samples may carry any count) and unaligned K through the generic one */
		const int fast = c->use_generic ? 0 : nsamp / OUTBLK;
		bool dft = c->fast;                         /* every stream planned on the raster? */
		for (int s = 0; dft && s < c->cfg.nstreams; s++) dft = c->fast_ok[s] != 0;
		bool all_rows = false;                       /* the fast CS16 kernel takes partial blocks too */
		if (dft && c->in_kind == IN_KIND_F32REAL && !c->use_generic) {
			r = launch_channelize_rdft(d_iq, stride, c->d_tw, c->d_twmeta, dmbuf, c->cfg.K, c->cfg.nch, c->cfg.nstreams, (size_t)nsamp, c->s_comp);
			c->stats.kernel_launches++;
			c->stats.fast_chan_launches++;
			all_rows = true;
		} else if (dft && c->in_kind == IN_KIND_CS16IQ && !c->use_generic) {
			r = launch_channelize_dft_cs16(d_iq, stride, c->d_tw, c->d_twmeta, dmbuf, c->cfg.K, c->cfg.nch, c->cfg.nstreams, (size_t)nsamp, c->s_comp);
			c->stats.kernel_launches++;
			c->stats.fast_chan_launches++;
			all_rows = true;
		} else if (fast && dft) {
			r = launch_channelize_dft(d_iq, stride, c->d_tw, c->d_twmeta, dmbuf, c->cfg.K, c->cfg.nch, c->cfg.nstreams, fast, (size_t)nsamp, c->fold8, c->s_comp);
			c->stats.kernel_launches++;
			c->stats.fast_chan_launches++;
		} else if (fast) {
			r = launch_channelize(c->in_kind, d_iq, stride, c->d_wf4, dmbuf, c->cfg.K, c->taps_pad, c->cfg.nch, c->cfg.nstreams, fast, (size_t)nsamp, c->s_comp);
			c->stats.kernel_launches++;
		}
		if (!r && !all_rows && nsamp > fast * OUTBLK) {
			r = launch_channelize_generic(c->in_kind, d_iq, stride, c->d_wf4, dmbuf, c->cfg.K, c->taps_pad, c->cfg.nch, c->cfg.nstreams,
			                              (size_t)fast * OUTBLK, (size_t)nsamp - (size_t)fast * OUTBLK, (size_t)nsamp, c->s_comp);
			c->stats.kernel_launches++;
		}
		if (r) return fail(ACB_ERR_CUDA, "channelizer launch: %s", cudaGetErrorString((cudaError_t)r));
		c->stats.chan_launches++;
		CU(cudaEventRecord(t.ev.b, c->s_comp));
		CU(cudaEventRecord(c->ev_k1_done[b], c->s_comp));
		c->k1_pending[b] = true;
		CU(cudaStreamWaitEvent(c->s_dem, c->ev_k1_done[b], 0));
	} else if (dm_host) {
		/* envelope input: the copy is ordered behind the previous demod on the same stream, and
		 * behind any channelizer launch that still targets the other buffer only */
		CU(cudaMemcpyAsync(dmbuf, dm_host, (size_t)c->cfg.nstreams * nsamp * c->cfg.nch * sizeof(float), cudaMemcpyHostToDevice, c->s_dem));
	}
	if (c->ring_read_pending[b]) {
		CU(cudaStreamWaitEvent(c->s_dem, c->ev_ring_read[b], 0));
		c->ring_read_pending[b] = false;
	}
	CU(cudaMemsetAsync(c->d_ctl[b], 0, sizeof(RingCtl), c->s_dem));
	CU(cudaEventRecord(t.ev.b2, c->s_dem));
	int r = launch_demod(c->d_state, dmbuf, nsamp, c->cfg.nch, c->cfg.nstreams, c->d_ring[b], c->d_ctl[b], c->ring_cap, c->demod_lanes, c->s_dem);
	if (r) return fail(ACB_ERR_CUDA, "demod launch: %s", cudaGetErrorString((cudaError_t)r));
	c->stats.kernel_launches++;
	c->stats.demod_launches++;
	CU(cudaEventRecord(c->ev_dm_free[b], c->s_dem));       /* the envelope buffer is the next-but-two channelizer's from here */
	CU(cudaEventRecord(c->ev_k2_done[b], c->s_dem));
	/* block FEC on the frames this submit appended (blk_thread's job, acars.c:93-215), in place — on its own stream:
	 * it touches this submit's ring only, and the next demod need not wait behind it */
	CU(cudaStreamWaitEvent(c->s_fec, c->ev_k2_done[b], 0));
	r = launch_block_fec(c->d_ring[b], c->d_ctl[b], c->ring_cap, c->s_fec);
	if (r) return fail(ACB_ERR_CUDA, "block FEC launch: %s", cudaGetErrorString((cudaError_t)r));
	c->stats.kernel_launches++;
	CU(cudaMemcpyAsync(c->h_ctl[b], c->d_ctl[b], sizeof(RingCtl), cudaMemcpyDeviceToHost, c->s_fec));
	CU(cudaEventRecord(t.ev.c, c->s_fec));
	c->dm_used[b] = true;
	c->last_dm = b;
	c->inflight.push_back(std::move(t));
	c->nsubmit++;
	c->stats.submits++;
	c->last_nsamp = nsamp;
	return ACB_OK;
}

static int check_blocks(acb_ctx *c, const void *p, size_t stride, int nblk)
{
	if (!c || !p) return fail(ACB_ERR_ARG, "null argument");
	if (c->real_input) return fail(ACB_ERR_ARG, "not a u8-IQ context: use acb_submit_real_host / acb_submit_cs16_host");
	if (nblk < 1 || nblk > c->cfg.max_blocks) return fail(ACB_ERR_ARG, "nblk=%d outside 1..%d", nblk, c->cfg.max_blocks);
	if (c->cfg.nstreams > 1 && stride < (size_t)nblk * c->blk_bytes) return fail(ACB_ERR_ARG, "stream_stride smaller than one stream's input");
	if (stride % 16) return fail(ACB_ERR_ARG, "stream_stride must be a multiple of 16 bytes");
	return ACB_OK;
}

static std::vector<unsigned long long> block_groups(const acb_ctx *c, int nblk)
{
	std::vector<unsigned long long> g(nblk);
	for (int b = 0; b < nblk; b++) g[b] = c->pos + (unsigned long long)b * OUTBLK;
	return g;
}

extern "C" int acb_submit_device(acb_ctx_t *c, const uint8_t *iq_dev, size_t stride, int nblk)
{
	if (int r = check_blocks(c, iq_dev, stride, nblk)) return r;
	if (int r = ctx_use(c)) return r;
	if (((uintptr_t)iq_dev) % 16) return fail(ACB_ERR_ARG, "device input must be 16-byte aligned");
	if (int r = run_kernels(c, iq_dev, stride, nblk, nblk * OUTBLK, nullptr, block_groups(c, nblk))) return r;
	c->pos += (unsigned long long)nblk * OUTBLK;
	c->stats.blocks += (uint64_t)nblk * c->cfg.nstreams;
	return ACB_OK;
}

extern "C" int acb_submit_host(acb_ctx_t *c, const uint8_t *iq, size_t stride, int nblk)
{
	if (int r = check_blocks(c, iq, stride, nblk)) return r;
	if (int r = ctx_use(c)) return r;
	if (!c->d_iq[0]) return fail(ACB_ERR_ARG, "context created with ACB_FLAG_NO_INPUT_STAGING");
	const int b = c->next_buf;
	c->next_buf ^= 1;
	const size_t per_stream = (size_t)nblk * c->blk_bytes;
	/* the kernels that last read this staging buffer must be done before it is overwritten */
	if (c->buf_used[b]) CU(cudaStreamWaitEvent(c->s_copy, c->ev_consumed[b], 0));
	if (stride == per_stream || c->cfg.nstreams == 1) {
		CU(cudaMemcpyAsync(c->d_iq[b], iq, per_stream * c->cfg.nstreams, cudaMemcpyHostToDevice, c->s_copy));
	} else {
		CU(cudaMemcpy2DAsync(c->d_iq[b], per_stream, iq, stride, per_stream, c->cfg.nstreams, cudaMemcpyHostToDevice, c->s_copy));
	}
	CU(cudaEventRecord(c->ev_copied[b], c->s_copy));
	CU(cudaStreamWaitEvent(c->s_comp, c->ev_copied[b], 0));
	if (int r = run_kernels(c, c->d_iq[b], per_stream, nblk, nblk * OUTBLK, nullptr, block_groups(c, nblk))) return r;
	CU(cudaEventRecord(c->ev_consumed[b], c->s_comp));      /* staging buffer is free once K1 has read it */
	c->buf_used[b] = true;
	c->pos += (unsigned long long)nblk * OUTBLK;
	c->stats.blocks += (uint64_t)nblk * c->cfg.nstreams;
	return ACB_OK;
}

extern "C" int acb_set_emission_groups(acb_ctx_t *c, int unit, uint64_t period)
{
	if (!c) return fail(ACB_ERR_ARG, "null context");
	if (unit != ACB_GROUP_SUBMIT && unit != ACB_GROUP_OUTPUTS && unit != ACB_GROUP_INPUT) return fail(ACB_ERR_ARG, "unknown group unit");
	if (unit != ACB_GROUP_SUBMIT && period == 0) return fail(ACB_ERR_ARG, "period must be > 0");
	c->group_unit = unit;
	c->group_period = period;
	return ACB_OK;
}

/* Emission groups of one streaming submit covering envelope samples [pos, pos + nout): the reference hands a
 * channel's new samples to demodMSK per transfer (air.c:336: output m completes with input sample (m+1)K - 1, so
 * transfer g of T samples starts at output floor(g*T/K)) or per full dm_buffer (soapy.c:247 every 1024 outputs,
 * sdrplay.c:229 every 512), channel by channel: frames leave in (group, channel, time) order. */
static std::vector<unsigned long long> stream_groups(const acb_ctx *c, size_t nout)
{
	std::vector<unsigned long long> g{ c->pos };
	const unsigned long long lo = c->pos, hi = c->pos + nout, K = (unsigned long long)c->cfg.K;
	if (c->group_unit == ACB_GROUP_OUTPUTS) {
		for (unsigned long long b = (lo / c->group_period + 1) * c->group_period; b < hi; b += c->group_period) g.push_back(b);
	} else if (c->group_unit == ACB_GROUP_INPUT) {
		const unsigned long long T = c->group_period;
		for (unsigned long long t = (lo * K) / T + 1;; t++) {        /* transfers that start after output `lo` began */
			const unsigned long long b = t * T / K;                  /* first output completed inside transfer t */
			if (b >= hi) break;
			if (b > g.back()) g.push_back(b);
		}
	}
	return g;
}

/* 4-byte samples (float32 real or int16 I,Q) of arbitrary count: appended behind the carried
 * remainder in d_real[b]; `x2` != NULL means planar int16 input (x = I plane, x2 = Q plane), which
 * two strided copies interleave on the way to the device */
static int submit4(acb_ctx *c, const void *x, const void *x2, size_t stride_samples, size_t nsamples)
{
	if (int r = ctx_use(c)) return r;
	const size_t K = (size_t)c->cfg.K, total = c->carry + nsamples;
	const size_t nout = total / K;
	if (nsamples == 0 || total > c->real_cap || nout > (size_t)c->cfg.max_blocks * OUTBLK)
		return fail(ACB_ERR_ARG, "nsamples=%zu exceeds max_blocks*1024*K", nsamples);
	if (c->cfg.nstreams > 1 && stride_samples < nsamples) return fail(ACB_ERR_ARG, "stream stride smaller than one stream's input");
	const int b = c->real_buf;
	/* The copy runs on the copy stream, so the H2D of submit i+1 overlaps the channelizer of submit i.
	 * d_real[b] was last read by the channelizer two submits ago and by the copy that moved its tail on. */
	float *buf = c->d_real[b];
	if (c->real_used[b]) CU(cudaStreamWaitEvent(c->s_copy, c->ev_real_free[b], 0));
	if (!x2) {
		CU(cudaMemcpy2DAsync(buf + c->carry, c->real_cap * sizeof(float), x, stride_samples * sizeof(float),
		                     nsamples * sizeof(float), c->cfg.nstreams, cudaMemcpyHostToDevice, c->s_copy));
	} else {
		/* planar int16 (the SDRplay callback's xi / xq): both planes go over as they are (two dense copies),
		 * a small kernel interleaves them behind the carried remainder */
		if (nsamples > c->planar_cap) {
			CU(cudaStreamSynchronize(c->s_copy));
			cudaFree(c->d_planar);
			c->d_planar = nullptr;
			c->planar_cap = std::max(nsamples, (size_t)c->cfg.max_blocks * OUTBLK * K);
			CU(cudaMalloc(&c->d_planar, 2 * (size_t)c->cfg.nstreams * c->planar_cap * sizeof(int16_t)));
		}
		int16_t *pi = c->d_planar, *pq = c->d_planar + (size_t)c->cfg.nstreams * c->planar_cap;
		CU(cudaMemcpy2DAsync(pi, c->planar_cap * 2, x, stride_samples * 2, nsamples * 2, c->cfg.nstreams, cudaMemcpyHostToDevice, c->s_copy));
		CU(cudaMemcpy2DAsync(pq, c->planar_cap * 2, x2, stride_samples * 2, nsamples * 2, c->cfg.nstreams, cudaMemcpyHostToDevice, c->s_copy));
		int r = launch_interleave_cs16(pi, pq, c->planar_cap, reinterpret_cast<uint32_t *>(buf + c->carry), c->real_cap, nsamples, c->cfg.nstreams, c->s_copy);
		if (r) return fail(ACB_ERR_CUDA, "interleave launch: %s", cudaGetErrorString((cudaError_t)r));
		c->stats.kernel_launches++;
	}
	CU(cudaEventRecord(c->ev_real_copied, c->s_copy));
	CU(cudaStreamWaitEvent(c->s_comp, c->ev_real_copied, 0));
	const size_t rem = total - nout * K;
	if (nout) {
		if (int r = run_kernels(c, (const uint8_t *)buf, c->real_cap * sizeof(float), 0, (int)nout, nullptr, stream_groups(c, nout)))
			return r;
		c->pos += nout;
		/* the unconsumed tail (air.c:329-334 / soapy.c:238-252 keep a partial sum instead: same
		 * arithmetic order) moves to the front of the other buffer */
		if (rem) {
			if (c->real_used[b ^ 1]) CU(cudaStreamWaitEvent(c->s_comp, c->ev_real_free[b ^ 1], 0));
			CU(cudaMemcpy2DAsync(c->d_real[b ^ 1], c->real_cap * sizeof(float), buf + nout * K, c->real_cap * sizeof(float),
			                     rem * sizeof(float), c->cfg.nstreams, cudaMemcpyDeviceToDevice, c->s_comp));
		}
		CU(cudaEventRecord(c->ev_real_free[b], c->s_comp));
		c->real_used[b] = true;
		c->real_buf = b ^ 1;
	}
	c->carry = rem;          /* nout == 0: the samples simply stay behind the previous carry */
	return (int)nout;
}

extern "C" int acb_submit_real_host(acb_ctx_t *c, const float *x, size_t stride_samples, size_t nsamples)
{
	if (!c || !x) return fail(ACB_ERR_ARG, "null argument");
	if (c->in_kind != IN_KIND_F32REAL) return fail(ACB_ERR_ARG, "context was not created with ACB_FLAG_REAL_INPUT");
	return submit4(c, x, nullptr, stride_samples, nsamples);
}

extern "C" int acb_submit_cs16_host(acb_ctx_t *c, const int16_t *iq, size_t stride_samples, size_t nsamples)
{
	if (!c || !iq) return fail(ACB_ERR_ARG, "null argument");
	if (c->in_kind != IN_KIND_CS16IQ) return fail(ACB_ERR_ARG, "context was not created with ACB_FLAG_CS16_INPUT");
	return submit4(c, iq, nullptr, stride_samples, nsamples);
}

extern "C" int acb_submit_cs16_planar_host(acb_ctx_t *c, const int16_t *xi, const int16_t *xq, size_t stride_samples, size_t nsamples)
{
	if (!c || !xi || !xq) return fail(ACB_ERR_ARG, "null argument");
	if (c->in_kind != IN_KIND_CS16IQ) return fail(ACB_ERR_ARG, "context was not created with ACB_FLAG_CS16_INPUT");
	return submit4(c, xi, xq, stride_samples, nsamples);
}

extern "C" int acb_set_plan_cs16(acb_ctx_t *c, int stream, const unsigned *freqs_hz, int nch, int variant, unsigned fc_hz, unsigned *fc_out)
{
	if (!c || !freqs_hz) return fail(ACB_ERR_ARG, "null argument");
	if (c->in_kind != IN_KIND_CS16IQ || nch != c->cfg.nch) return fail(ACB_ERR_ARG, "not a CS16 context / nch mismatch");
	if (c->taps != c->cfg.K) return fail(ACB_ERR_ARG, "taps != K: supply the tables with acb_set_wf");
	if (variant != ACB_CS16_SOAPY && variant != ACB_CS16_SDRPLAY) return fail(ACB_ERR_ARG, "unknown CS16 variant");
	const unsigned fc = fc_hz ? fc_hz : acb_choose_fc(freqs_hz, nch, c->cfg.K);      /* soapy.c:132-136, sdrplay.c:124 */
	if (fc == 0) return fail(ACB_ERR_PLAN, "Frequencies too far apart");
	std::vector<float> wf((size_t)nch * c->cfg.K * 2);
	for (int ch = 0; ch < nch; ch++) acb_cs16_build_wf(variant, freqs_hz[ch], fc, c->cfg.K, &wf[(size_t)ch * c->cfg.K * 2]);
	if (fc_out) *fc_out = fc;
	if (int r = acb_set_wf(c, stream, wf.data(), nch)) return r;
	if (!c->fast) return ACB_OK;
	std::vector<int> kbin(nch);
	std::vector<float> tw1((size_t)nch * (c->cfg.K / 4) * 2);
	const bool ok = acb_fast_plan_cs16(variant, freqs_hz, nch, c->cfg.K, fc, kbin.data(), tw1.data()) == 1;
	return upload_fast_plan(c, stream, ok, kbin, tw1);
}

extern "C" int acb_set_plan_air(acb_ctx_t *c, int stream, const unsigned *freqs_hz, int nch, unsigned *fc_out)
{
	if (!c || !freqs_hz) return fail(ACB_ERR_ARG, "null argument");
	if (c->in_kind != IN_KIND_F32REAL || nch != c->cfg.nch) return fail(ACB_ERR_ARG, "not a real-input context / nch mismatch");
	if (c->taps != c->cfg.K) return fail(ACB_ERR_ARG, "taps != K: supply the tables with acb_set_wf");
	unsigned lo = freqs_hz[0], hi = freqs_hz[0];
	for (int i = 1; i < nch; i++) { lo = std::min(lo, freqs_hz[i]); hi = std::max(hi, freqs_hz[i]); }
	const unsigned rate = (unsigned)c->cfg.K * ACB_INTRATE;
	const unsigned fc = acb_air_choose_fc(lo, hi);
	std::vector<float> wf((size_t)nch * c->cfg.K * 2);
	for (int ch = 0; ch < nch; ch++) acb_air_build_wf((int)freqs_hz[ch], (int)fc, rate, &wf[(size_t)ch * c->cfg.K * 2]);
	if (fc_out) *fc_out = fc;
	if (int r = acb_set_wf(c, stream, wf.data(), nch)) return r;
	if (!c->fast) return ACB_OK;
	std::vector<int> kbin(nch);
	std::vector<float> tw1((size_t)nch * (c->cfg.K / 4) * 2);
	const bool ok = acb_fast_plan_air(freqs_hz, nch, c->cfg.K, fc, kbin.data(), tw1.data()) == 1;
	return upload_fast_plan(c, stream, ok, kbin, tw1);
}

extern "C" int acb_submit_dm_host(acb_ctx_t *c, const float *dm, int nsamp)
{
	if (!c || !dm) return fail(ACB_ERR_ARG, "null argument");
	if (int r = ctx_use(c)) return r;
	const size_t n = (size_t)c->cfg.nstreams * nsamp * c->cfg.nch;
	if (nsamp < 1 || n > c->dm_floats) return fail(ACB_ERR_ARG, "nsamp=%d exceeds max_blocks*1024", nsamp);
	/* A pageable source has been staged when the call returns; a pinned one must stay untouched
	 * until the submit is collected. */
	if (int r = run_kernels(c, nullptr, 0, 0, nsamp, dm, std::vector<unsigned long long>{ c->pos })) return r;
	c->pos += (unsigned long long)nsamp;
	return ACB_OK;
}

extern "C" int acb_wait_event(acb_ctx_t *c, void *cuda_event)
{
	if (!c || !cuda_event) return fail(ACB_ERR_ARG, "null argument");
	if (int r = ctx_use(c)) return r;
	CU(cudaStreamWaitEvent(c->s_comp, (cudaEvent_t)cuda_event, 0));
	return ACB_OK;
}

extern "C" int acb_collect(acb_ctx_t *c)
{
	if (!c) return fail(ACB_ERR_ARG, "null context");
	if (int r = ctx_use(c)) return r;
	if (int r = collect_oldest(c)) return r;
	wait_consumer(c, c->jobs_queued);
	if (c->overflowed) {
		c->overflowed = false;
		return fail(ACB_ERR_OVERFLOW, "device frame ring overflowed (%u slots): %llu frames lost so far", c->ring_cap, (unsigned long long)c->stats.frames_lost);
	}
	std::lock_guard<std::mutex> lk(c->mtx);
	return (int)c->outq_count;
}

extern "C" int acb_sync(acb_ctx_t *c)
{
	if (!c) return fail(ACB_ERR_ARG, "null context");
	if (int r = ctx_use(c)) return r;
	while (!c->inflight.empty())
		if (int r = collect_oldest(c)) return r;
	CU(cudaStreamSynchronize(c->s_comp));
	CU(cudaStreamSynchronize(c->s_dem));
	CU(cudaStreamSynchronize(c->s_fec));
	wait_consumer(c, c->jobs_queued);
	if (c->consumer_err[0]) return fail(ACB_ERR_CUDA, "%s", c->consumer_err);
	if (c->overflowed) {
		c->overflowed = false;
		return fail(ACB_ERR_OVERFLOW, "device frame ring overflowed (%u slots): %llu frames lost so far", c->ring_cap, (unsigned long long)c->stats.frames_lost);
	}
	std::lock_guard<std::mutex> lk(c->mtx);
	return (int)c->outq_count;
}

extern "C" int acb_mark(acb_ctx_t *c, int which)
{
	if (!c || which < 0 || which > 1) return fail(ACB_ERR_ARG, "bad argument");
	if (int r = ctx_use(c)) return r;
	/* a timed region starts on the channelizer stream and ends behind the last demod and the last block FEC */
	if (which == 0) {
		CU(cudaEventRecord(c->mark[0], c->s_comp));
	} else {
		CU(cudaEventRecord(c->ev_join, c->s_dem));
		CU(cudaStreamWaitEvent(c->s_fec, c->ev_join, 0));
		CU(cudaEventRecord(c->mark[1], c->s_fec));
	}
	return ACB_OK;
}

extern "C" int acb_elapsed_ms(acb_ctx_t *c, float *ms)
{
	if (!c || !ms) return fail(ACB_ERR_ARG, "null argument");
	if (int r = ctx_use(c)) return r;
	CU(cudaEventSynchronize(c->mark[1]));
	CU(cudaEventElapsedTime(ms, c->mark[0], c->mark[1]));
	return ACB_OK;
}

extern "C" int acb_drain(acb_ctx_t *c, acb_msg_t *out, int max)
{
	if (!c || (!out && max > 0)) return fail(ACB_ERR_ARG, "null argument");
	int n = 0;
	std::lock_guard<std::mutex> lk(c->mtx);
	while (n < max && !c->outq.empty()) {
		acb_ctx::Batch &b = c->outq.front();
		const size_t take = std::min((size_t)(max - n), b.n - b.rd);
		memcpy(out + n, b.v.get() + b.rd, take * sizeof(acb_msg_t));
		n += (int)take;
		b.rd += take;
		if (b.rd == b.n) c->outq.pop_front();
	}
	c->outq_count -= (size_t)n;
	return n;
}

extern "C" int acb_block_fec_batch(acb_ctx_t *c, acb_msg_t *msgs, int n, int *keep)
{
	if (!c || !msgs || !keep || n < 0) return fail(ACB_ERR_ARG, "bad argument");
	if (int r = ctx_use(c)) return r;
	if (n == 0) return 0;
	std::vector<RawFrame> raw(n);
	memset(raw.data(), 0, (size_t)n * sizeof(RawFrame));
	for (int i = 0; i < n; i++) {
		raw[i].len = msgs[i].len; raw[i].err = msgs[i].err; raw[i].chn = msgs[i].chn;
		memcpy(raw[i].txt, msgs[i].txt, ACB_TXTMAX);
		raw[i].crc[0] = msgs[i].crc[0]; raw[i].crc[1] = msgs[i].crc[1];
	}
	RawFrame *d = nullptr;
	RingCtl *dc = nullptr, hc;
	memset(&hc, 0, sizeof(hc));
	hc.count = (unsigned)n;
	cudaError_t e = cudaMalloc(&d, (size_t)n * sizeof(RawFrame));
	if (e == cudaSuccess) e = cudaMalloc(&dc, sizeof(RingCtl));
	if (e == cudaSuccess) e = cudaMemcpyAsync(d, raw.data(), (size_t)n * sizeof(RawFrame), cudaMemcpyHostToDevice, c->s_d2h);   /* same stream as the kernel */
	if (e == cudaSuccess) e = cudaMemcpyAsync(dc, &hc, sizeof(hc), cudaMemcpyHostToDevice, c->s_d2h);
	if (e == cudaSuccess) e = (cudaError_t)launch_block_fec(d, dc, (unsigned)n, c->s_d2h);
	if (e == cudaSuccess) e = cudaMemcpyAsync(raw.data(), d, (size_t)n * sizeof(RawFrame), cudaMemcpyDeviceToHost, c->s_d2h);
	if (e == cudaSuccess) e = cudaStreamSynchronize(c->s_d2h);
	cudaFree(d);
	cudaFree(dc);
	if (e != cudaSuccess) return fail(ACB_ERR_CUDA, "block FEC batch: %s", cudaGetErrorString(e));
	int kept = 0;
	for (int i = 0; i < n; i++) {
		keep[i] = raw[i].pad0 == 1;
		kept += keep[i];
		if (keep[i]) {
			msgs[i].err = raw[i].err;
			memcpy(msgs[i].txt, raw[i].txt, ACB_TXTMAX);
		}
	}
	return kept;
}

extern "C" int acb_pending(acb_ctx_t *c)
{
	if (!c) return fail(ACB_ERR_ARG, "null context");
	std::lock_guard<std::mutex> lk(c->mtx);
	return (int)c->outq_count;
}

extern "C" int acb_read_dm(acb_ctx_t *c, float *out, size_t nfloats)
{
	if (!c || !out) return fail(ACB_ERR_ARG, "null argument");
	if (int r = ctx_use(c)) return r;
	const size_t have = (size_t)c->cfg.nstreams * c->last_nsamp * c->cfg.nch;
	if (nfloats > have) return fail(ACB_ERR_ARG, "asked for %zu floats, last submit produced %zu", nfloats, have);
	CU(cudaStreamSynchronize(c->s_comp));
	CU(cudaStreamSynchronize(c->s_dem));
	CU(cudaMemcpyAsync(out, c->d_dm[c->last_dm], nfloats * sizeof(float), cudaMemcpyDeviceToHost, c->s_copy));
	CU(cudaStreamSynchronize(c->s_copy));
	return ACB_OK;
}

static void to_api(const ChainState &s, acb_chan_state_t *o)
{
	memset(o, 0, sizeof(*o));
	o->MskPhi = s.phi; o->MskDf = s.df; o->MskLvlSum = s.lvlsum; o->MskClk = s.clk;
	o->MskBitCount = s.bitcount; o->MskS = s.S; o->idx = s.idx; o->nbits = s.nbits;
	o->Acarsstate = s.state; o->outbits = s.outbits; o->blk_len = s.blk_len; o->blk_err = s.blk_err;
	o->pos = s.pos; o->soh_pos = s.soh_pos;
	memcpy(o->inb_re, s.inb_re, sizeof(o->inb_re));
	memcpy(o->inb_im, s.inb_im, sizeof(o->inb_im));
	o->blk_crc[0] = s.crc[0]; o->blk_crc[1] = s.crc[1];
	memcpy(o->blk_txt, s.txt, ACB_TXTMAX);
}

static void from_api(const acb_chan_state_t *i, ChainState &s)
{
	memset(&s, 0, sizeof(s));
	s.phi = i->MskPhi; s.df = i->MskDf; s.lvlsum = i->MskLvlSum; s.clk = i->MskClk;
	s.bitcount = i->MskBitCount; s.S = i->MskS; s.idx = i->idx % FLEN; s.nbits = i->nbits;
	s.state = i->Acarsstate; s.outbits = i->outbits & 0xffu; s.blk_len = i->blk_len; s.blk_err = i->blk_err;
	s.pos = i->pos; s.soh_pos = i->soh_pos;
	memcpy(s.inb_re, i->inb_re, sizeof(s.inb_re));
	memcpy(s.inb_im, i->inb_im, sizeof(s.inb_im));
	s.crc[0] = i->blk_crc[0]; s.crc[1] = i->blk_crc[1];
	memcpy(s.txt, i->blk_txt, ACB_TXTMAX);
}

extern "C" int acb_get_state(acb_ctx_t *c, int stream, int chn, acb_chan_state_t *out)
{
	if (!c || !out) return fail(ACB_ERR_ARG, "null argument");
	if (stream < 0 || stream >= c->cfg.nstreams || chn < 0 || chn >= c->cfg.nch) return fail(ACB_ERR_ARG, "stream/chn out of range");
	if (int r = ctx_use(c)) return r;
	ChainState s;
	if (int r = sync_streams(c)) return r;
	CU(cudaMemcpyAsync(&s, c->d_state + (size_t)stream * c->cfg.nch + chn, sizeof(s), cudaMemcpyDeviceToHost, c->s_copy));
	CU(cudaStreamSynchronize(c->s_copy));
	to_api(s, out);
	return ACB_OK;
}

extern "C" int acb_set_state(acb_ctx_t *c, int stream, int chn, const acb_chan_state_t *in)
{
	if (!c || !in) return fail(ACB_ERR_ARG, "null argument");
	if (stream < 0 || stream >= c->cfg.nstreams || chn < 0 || chn >= c->cfg.nch) return fail(ACB_ERR_ARG, "stream/chn out of range");
	if (in->blk_len < 0 || in->blk_len > 248) return fail(ACB_ERR_ARG, "blk_len out of range");
	if (int r = ctx_use(c)) return r;
	ChainState s;
	from_api(in, s);
	if (int r = sync_streams(c)) return r;
	if (int r = upload(c, c->d_state + (size_t)stream * c->cfg.nch + chn, &s, sizeof(s))) return r;
	return ACB_OK;
}

extern "C" int acb_get_stats(acb_ctx_t *c, acb_stats_t *out, int reset)
{
	if (!c || !out) return fail(ACB_ERR_ARG, "null argument");
	std::lock_guard<std::mutex> lk(c->mtx);
	*out = c->stats;
	if (reset) memset(&c->stats, 0, sizeof(c->stats));
	return ACB_OK;
}
