#!/usr/bin/env python
"""bench.py — IQ Msamples/s through channelize + demodMSK + frame sync on B200 (BASELINE.json metric).

  python bench.py [--gpus N] [--steps K] [--warmup W]            # this repo's CUDA path
  python bench.py --impl reference [...]                         # the reference's own CPU path

Headline workload: BASELINE configs[1] (synthetic 2 MS/s uint8 IQ, K=160, 8 ACARS channels per stream) x S
independent streams per GPU.  One "step" = one pass of the hot path over B blocks of 1024*K complex samples of
every stream.  S is the stream count at which a B200 saturates: the demodulator is a serial recurrence per
channel (msk.c:67-137), so one stream alone is latency bound; the bench sweeps S in {592, 1184, 2368, 4736}
(4..32 streams per SM) on the device and quotes `value` at the best one, naming it in config.workload.
Per-GPU work is fixed as N grows (weak scaling): N GPUs serve N*S streams, sharded by stream index with no
collective on the data path (SURVEY.md §8e).

Printed JSON (rank 0, one line):
  value        device-resident throughput: inputs already in HBM, CUDA events on the library's streams around
               exactly K steps, max over ranks
  e2e          same metric through the C ABI with HOST buffers: pinned H2D copy of every step's input and D2H
               read-back of the decoded frames inside the timed region
  roofline     channelizer kernel (the dominant kernel) of --channelizer: algorithmic bytes / CUDA-event duration
               vs measured HBM peak, in the pipeline (demod running underneath) and isolated
  alt_channelizer  the other channelizer form at the same S, same treatment (its own roofline object)
  checked      every frame of the timed steps (and the passes before them) of the distinct pool streams against the
               CPU port of the reference (oracle/), which the tests pin to the unmodified reference
  cpu_baseline the unmodified reference (oracle/_ref, -Ofast) on all host threads, bounded sample
  configs      the literal BASELINE configs 2..5 (one stream x 8 ch; K=192 x 64 ch x 165 taps; 128 streams total,
               strong-scaled; 20 MS/s x 256 ch tap sweep) with the wide-stream broadcast inside the timed region at N>1
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tests"))

METRIC = "IQ Msamples/s through channelize+demodMSK (msgs bit-exact)"
UNIT = "Msamples/s"
SWEEP = (592, 1184, 2368, 4736)          # 4, 8, 16, 32 streams per SM
FRAME_BYTES = 304                        # RawFrame record read back per decoded frame


STEP_CAP = 37888                         # stream-blocks per step: 12.4 GB of input (halved if the host cannot pin that much)


def blocks_for(S: int, want: int, cap: int = STEP_CAP) -> int:
    """Blocks per step: `want` (16 = 1.31 s of signal) while a step's input stays <= 12.4 GB, so that the
    e2e leg's pinned host buffer and the two device staging buffers stay bounded at large S."""
    return max(1, min(want, cap // S))


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--streams", type=int, default=0, help="IQ streams per GPU; 0 = sweep %s and take the best" % (SWEEP,))
    ap.add_argument("--blocks", type=int, default=16, help="1024-sample output blocks per stream per step (capped so a step's input stays <= 12.4 GB)")
    ap.add_argument("--K", type=int, default=160, help="rtlMult (160 = 2.0 MS/s)")
    ap.add_argument("--channelizer", default="exact", choices=["exact", "fast"],
                    help="exact: the reference's rounding sequence, envelope bit-identical; fast: ACB_FLAG_FAST_CHANNELIZER "
                         "(shared DFT factorisation; messages identical, envelope within its stated tolerance)")
    ap.add_argument("--pool", type=int, default=4, help="distinct synthetic streams generated (tiled over S)")
    ap.add_argument("--cpu-seconds", type=float, default=10.0)
    ap.add_argument("--config", default="all", help="BASELINE configs to add to the line: all | none | comma list of 2,3,4,5")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-alt", action="store_true", help="skip the measurement of the other channelizer form")
    ap.add_argument("--no-check", action="store_true", help="skip the oracle check of the timed frames")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one computed for the distinct pool streams as DIR/*.npy "
                         "(envelope, decoded frames); the stream count is then --streams, or %d without the sweep, so that "
                         "the same arguments give the same inputs" % SWEEP[-1])
    ap.add_argument("--cpu-worker", action="store_true", help=argparse.SUPPRESS)
    ap.add_argument("--variant", default="", help=argparse.SUPPRESS)
    ap.add_argument("--worker-blocks", type=int, default=256, help=argparse.SUPPRESS)
    ap.add_argument("--worker-seed", type=int, default=0, help=argparse.SUPPRESS)
    return ap.parse_args()


# ----------------------------------------------------------------------------- synthetic input

def make_pool(K: int, nblk: int, pool: int, fc: int, seed0: int = 1000):
    """`pool` distinct streams of `nblk` blocks with injected ACARS frames (synth.py)."""
    from acarsdec_b200 import synth
    secs = nblk * 1024 / 12500.0
    out = []
    for i in range(pool):
        plan = synth.make_plan(K, synth.DEFAULT_FREQS_MHZ, fc, seconds=secs, seed=seed0 + i)
        out.append(synth.render_blocks(plan, 0, nblk).reshape(-1))
    return out


# ----------------------------------------------------------------------------- CPU reference arm

def effective_cpus() -> int:
    """Host threads this process may actually use: affinity mask capped by the cgroup CPU quota
    (the GPU boxes show 128 CPUs but run the container under a 16-CPU quota)."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()
        if quota != "max":
            n = min(n, max(1, -(-int(quota) // int(period))))
    except (OSError, ValueError):
        pass
    return n


def cpu_worker(args) -> None:
    """Child process: the reference's in_callback + demodMSK + decodeAcars + blk_thread loop
    (oracle/_ref, unmodified sources) over a small ring of synthetic blocks."""
    import refs
    from acarsdec_b200 import synth
    ref = refs.RefLib(args.variant)
    sys.stderr = open(os.devnull, "w")
    devnull = os.open(os.devnull, os.O_WRONLY)
    os.dup2(devnull, 2)                       # the reference prints its sample rate on stderr
    ref.open_rtl(args.K, synth.DEFAULT_FREQS_MHZ)
    bufs = np.stack(make_pool(args.K, 4, 1, ref.fc, seed0=5000 + args.worker_seed)).reshape(4, -1)
    ref.run(bufs, 4)
    print("READY", flush=True)
    sys.stdin.readline()
    t = []
    for s in range(args.warmup + args.steps):
        t.append(time.perf_counter())
        ref.run(bufs, args.worker_blocks)
    t.append(time.perf_counter())
    nmsg = len(ref.msgs())
    print(json.dumps({"timed_s": t[-1] - t[args.warmup], "msgs": nmsg}), flush=True)


def run_cpu_reference(K: int, steps: int, warmup: int, blocks_per_step: int, nproc: int | None = None):
    """All host threads, one reference instance (= one stream) per process.  Returns dict."""
    import refs
    variant = refs.best_fast_variant()
    kind = "reference"
    if not refs.ref_available(variant):
        variant = "v3" if refs.ref_available("v3") else ("O2" if refs.ref_available("O2") else "")
    if not variant:
        return run_cpu_port(K, steps, warmup, blocks_per_step, nproc)
    nproc = nproc or effective_cpus()
    cmd = [sys.executable, str(ROOT / "bench.py"), "--cpu-worker", "--variant", variant, "--K", str(K),
           "--steps", str(steps), "--warmup", str(warmup), "--worker-blocks", str(blocks_per_step)]
    procs = [subprocess.Popen(cmd + ["--worker-seed", str(i)], stdin=subprocess.PIPE, stdout=subprocess.PIPE, text=True)
             for i in range(nproc)]
    for p in procs:
        assert p.stdout.readline().strip() == "READY"
    for p in procs:
        p.stdin.write("go\n")
        p.stdin.flush()
    res = [json.loads(p.stdout.readline()) for p in procs]
    for p in procs:
        p.wait()
    slowest = max(r["timed_s"] for r in res)
    samples = nproc * steps * blocks_per_step * 1024 * K
    return {"value": samples / slowest / 1e6, "unit": UNIT, "cores": nproc, "kind": kind,
            "sample": f"{nproc} processes (= usable host threads; {os.cpu_count()} visible) x 1 stream x 8 ch, "
                      f"{steps} steps x {blocks_per_step} blocks "
                      f"({samples / 1e6:.0f} Msamples), oracle/_ref libacarsref_{variant}.so "
                      f"(unmodified rtl.c/msk.c/acars.c, -Ofast -march=x86-64-{variant})",
            "ms_per_step": slowest / steps * 1e3, "single_thread_value": None}


def run_cpu_port(K, steps, warmup, blocks_per_step, nproc=None):
    """Fallback when oracle/_ref is absent: the C restatement on all threads."""
    import refs
    refs.ensure_built()
    orc = refs.OracleLib()
    nproc = nproc or effective_cpus()
    from acarsdec_b200 import synth
    wf = orc.wf(K, synth.DEFAULT_FREQS_MHZ)
    _, _, fc = orc.plan(K, synth.DEFAULT_FREQS_MHZ)
    bufs = np.stack(make_pool(K, 4, 1, fc)).reshape(-1)
    orc.lib.orc_bench_streams(nproc, K, 8, wf.ctypes.data, bufs.ctypes.data, 4, warmup * blocks_per_step)
    secs = orc.lib.orc_bench_streams(nproc, K, 8, wf.ctypes.data, bufs.ctypes.data, 4, steps * blocks_per_step)
    samples = nproc * steps * blocks_per_step * 1024 * K
    return {"value": samples / secs / 1e6, "unit": UNIT, "cores": nproc, "kind": "port",
            "sample": f"{nproc} threads x 1 stream x 8 ch, {steps * blocks_per_step} blocks each, oracle/acars_oracle.c -O2",
            "ms_per_step": secs / steps * 1e3}


# ----------------------------------------------------------------------------- the checker (oracle/)

def oracle_frames(K: int, streams, reps: int):
    """The CPU port of the reference (oracle/acars_oracle.c, pinned against the unmodified reference by the
    tests) over each stream's blocks fed `reps` times in a row (state carried, like the bench's repeated
    submits of the same device buffer).  One thread per stream (ctypes releases the GIL)."""
    import refs
    from common import msg_tuple
    from acarsdec_b200 import synth
    refs.ensure_built()
    orc = refs.OracleLib()
    wf = orc.wf(K, synth.DEFAULT_FREQS_MHZ)
    out = [None] * len(streams)

    def work(i):
        o = refs.OracleStream(orc, K, wf)
        for _ in range(reps):
            o.blocks(streams[i])
        out[i] = [msg_tuple(m) for m in o.msgs()]
        o.close()

    th = [threading.Thread(target=work, args=(i,)) for i in range(len(streams))]
    for t in th:
        t.start()
    for t in th:
        t.join()
    return out


def check_frames(K: int, pool, reps: int, recs, exact: bool, nstreams: int, per_stream=None):
    """recs: numpy records (api.MSG_DTYPE) of everything the context decoded since reset for the first len(pool)
    streams, in emission order; per_stream: frames decoded per stream, all streams (default: counted from recs).
    Streams s and s + len(pool) carry the same bytes: the first len(pool) streams must equal the CPU port frame
    for frame (text, BCS, err, lvl bits; order), and every replica must have decoded the same number of frames."""
    want = oracle_frames(K, pool, reps)
    ok, frames = True, 0
    for i in range(len(pool)):
        mine = [rec_tuple(m) for m in recs[recs["stream"] == i]]
        if exact:
            ok = ok and mine == want[i]
        else:
            ok = ok and [t[:-1] for t in mine] == [t[:-1] for t in want[i]]
            la = np.array([t[-1] for t in mine], dtype=np.uint32).view(np.float32)
            lb = np.array([t[-1] for t in want[i]], dtype=np.uint32).view(np.float32)
            ok = ok and la.shape == lb.shape and bool(np.all(np.abs(la - lb) <= 0.05))
        frames += len(want[i])
    if per_stream is None:
        per_stream = np.bincount(recs["stream"], minlength=nstreams)
    replicas_ok = all(len(set(per_stream[i::len(pool)].tolist())) == 1 for i in range(len(pool)))
    out = {"streams_vs_cpu_port": len(pool), "passes_checked": reps, "frames": frames, "bit_exact": bool(ok),
           "replicas_identical_counts": bool(replicas_ok), "frames_all_streams": int(per_stream.sum())}
    if not exact:
        out["note"] = "messages (chn, len, err, text, BCS) identical; lvl within 0.05 dB (fast channelizer)"
    return out


def dump_outputs(d: str, m: dict, B: int) -> None:
    """The timed path's results in its last step (pass m["passes"]) for the distinct pool streams, which every other
    stream repeats: envelope.npy float32 (stream, sample, channel); frames.npy float64, one row per decoded frame in
    emission order (stream, chn, len, err, lvl, block, pos, soh_pos, crc[0], crc[1]); frames_txt.npy float32, the
    frames' text bytes, zero past len."""
    d = Path(d)
    d.mkdir(parents=True, exist_ok=True)
    recs = m["recs"][m["recs"]["block"] >= (m["passes"] - 1) * B]
    cols = [recs[f].astype(np.float64) for f in ("stream", "chn", "len", "err", "lvl", "block", "pos", "soh_pos")]
    np.save(d / "envelope.npy", m["dm_last"])
    np.save(d / "frames.npy", np.stack(cols + [recs["crc"][:, 0].astype(np.float64), recs["crc"][:, 1].astype(np.float64)], axis=1))
    txt = recs["txt"].astype(np.float32)
    txt[np.arange(txt.shape[1])[None, :] >= recs["len"][:, None]] = 0
    np.save(d / "frames_txt.npy", txt)


def rec_tuple(m):
    return (int(m["chn"]), int(m["len"]), int(m["err"]), bytes(m["txt"][:int(m["len"])]), bytes(m["crc"]), int(np.float32(m["lvl"]).view(np.uint32)))


# ----------------------------------------------------------------------------- clocks

class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.idx = gpu_index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.idx}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), [x.strip() for x in line.split(",")]))

    def stop(self):
        if self.proc:
            self.proc.terminate()

    def summary(self, t0: float, t1: float):
        rows = [r for (t, r) in self.rows if t0 <= t <= t1 + 0.15 and len(r) >= 8] or [r for (_, r) in self.rows[-3:] if len(r) >= 8]
        if not rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        sm = sorted(float(r[1]) for r in rows)
        reasons = set()
        for r in rows:
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": float(rows[0][2]), "reasons": sorted(reasons),
                "power_w_max": max(float(r[3]) for r in rows), "samples": len(rows)}


# ----------------------------------------------------------------------------- GPU arm helpers

def pin_to_gpu_numa_node(gpu_index: int):
    """Run this rank on the CPUs of the NUMA node its GPU hangs off (the e2e leg streams 55 GB/s per GPU out of
    pinned host memory; across the socket link that costs a few percent at N=8).  Best effort: returns the node or None."""
    try:
        bus = subprocess.run(["nvidia-smi", f"--id={gpu_index}", "--query-gpu=pci.bus_id", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=20).stdout.strip().lower()
        if bus.startswith("0000"):
            bus = bus[4:]                     # nvidia-smi prints an 8-digit domain, sysfs a 4-digit one
        node = int(open(f"/sys/bus/pci/devices/{bus}/numa_node").read())
        if node < 0:
            return None
        cpus = set()
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
            return node
    except Exception:
        pass
    return None


def measured_peak():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def traffic_per_launch(channelizer: str, S: int, B: int, K: int):
    """dram__bytes_read + dram__bytes_write of the channelizer kernel from the committed ncu capture
    (profiles/k1_traffic.json, written by tools/summarize_ncu.py).  The kernel's grid is one CTA per (block, stream,
    channel group) and every CTA reads its own rows once, so a capture at S0 x B0 scales by S*B/(S0*B0); the
    entry says which shape was captured."""
    tp = ROOT / "profiles" / "k1_traffic.json"
    try:
        tj = json.load(open(tp)).get(channelizer)
        if tj and tj.get("K") == K:
            return tj["dram_bytes_per_launch"] * (S * B) / (tj["streams"] * tj["blocks"]), f"ncu capture at {tj['streams']} x {tj['blocks']}, scaled by stream-blocks"
    except Exception:
        pass
    return None, None


class DeviceInput:
    """The pool tiled over S streams, resident in HBM (streams s and s + len(pool) carry the same bytes)."""

    def __init__(self, ctx, pool, S: int, stride: int):
        self.ctx, self.ptr = ctx, ctx.device_alloc(S * stride)
        for s in range(S):
            ctx.copy_to_device(self.ptr + s * stride, pool[s % len(pool)][:stride])

    def free(self):
        self.ctx.device_free(self.ptr)


def roofline_obj(channelizer: str, fast_ran: bool, k1_ms: float, k1_iso_ms, S: int, B: int, K: int, nch: int, sm_mhz: float):
    peak, peak_src = measured_peak()
    blk_bytes = 2048 * K
    alg = S * B * (blk_bytes + 1024 * nch * 4)            # u8 IQ read once + dm written once (K1 and K2 are separate kernels)
    achieved = alg / (k1_ms * 1e-3) / 1e9
    traffic, tsrc = traffic_per_launch(channelizer, S, B, K)
    cmacs = S * B * 1024 * K * nch
    # FP32 lane-ops per complex MAC-equivalent: exact = 8 rounded ops; fast (folded) = (3.25 + C/2) per input sample over C channels
    ops_per_cmac = (3.25 + nch / 2) / nch if fast_ran else 8.0
    fp32_peak_cmac = 148 * 128 * sm_mhz * 1e6 / ops_per_cmac
    o = {"kernel": "k_channelize_dft" if fast_ran else "k_channelize", "channelizer": channelizer, "bound": "hbm",
         "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic, "traffic_source": tsrc,
         "peak_source": peak_src, "algorithmic_bytes_per_launch": alg, "launch_ms": k1_ms,
         "timing": "CUDA events around the kernel on its own stream, averaged over the timed steps, demod of the previous step running underneath",
         "fp32_issue_frac": (cmacs / (k1_ms * 1e-3)) / fp32_peak_cmac,
         "note": ("fast form: K-point DFT bins via an exact fold + 4-point split shared by the channels, K/8 MACs per channel"
                  if fast_ran else
                  "FP32-issue bound: the reference's rounding sequence costs 8 rounded FP32 ops per complex "
                  "MAC per channel (4*C flop/B, C=8); ceiling 17.7 % of HBM peak, see DESIGN.md")}
    if k1_iso_ms:
        o["isolated"] = {"launch_ms": k1_iso_ms, "achieved": alg / (k1_iso_ms * 1e-3) / 1e9, "frac": alg / (k1_iso_ms * 1e-3) / 1e9 / peak,
                         "timing": "same kernel, nothing else on the GPU (sync between steps)"}
    return o


def main():
    args = parse_args()
    if args.cpu_worker:
        cpu_worker(args)
        return

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    K = args.K
    nch = 8

    if args.impl == "reference":
        if rank != 0:
            return
        blocks = 256
        r = run_cpu_reference(K, args.steps, args.warmup, blocks)
        line = {"impl": "reference", "metric": METRIC, "value": r["value"], "unit": UNIT, "n_gpus": args.gpus,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": r["ms_per_step"], "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": {"workload": f"configs[1]: synthetic 2 MS/s uint8 IQ, 8 ACARS channels per stream (K={K}); "
                                       f"one reference process per host thread, {blocks} blocks per step each",
                           "K": K, "channels_per_stream": nch},
                "cpu_baseline": {k: r[k] for k in ("value", "unit", "cores", "kind", "sample")},
                "e2e": {"value": r["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "gpu_launches": 0}
        print(json.dumps(line))
        return

    from acarsdec_b200 import sharding
    numa = pin_to_gpu_numa_node(local) if world > 1 else None      # before any pinned allocation: first touch lands on the GPU's node
    dist, rank, world, local = sharding.init_process_group()      # NCCL: rendezvous, timing reductions, the wide-stream broadcast
    dev = f"cuda:{local}" if dist is not None else None

    def barrier():
        if dist is not None:
            dist.barrier()

    def max_over_ranks(x: float) -> float:
        return sharding.reduce_scalar(dist, x, "max", dev)

    def sum_over_ranks(x: float) -> float:
        return sharding.reduce_scalar(dist, x, "sum", dev)

    # the CPU baseline runs first (rank 0, N=1 only), before this process touches CUDA
    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        blocks = 256
        steps = max(2, int(args.cpu_seconds / 0.4))
        cpu = run_cpu_reference(K, steps, 1, blocks)

    from acarsdec_b200 import api, build, synth
    build.build()

    fd, _, fc = api.plan(K, synth.DEFAULT_FREQS_MHZ)
    blk_bytes = 2048 * K
    pool = make_pool(K, min(args.blocks, 16), args.pool, fc, seed0=1000 + 17 * rank)
    do_check = (not args.no_check) and rank == 0
    fastflag = {"exact": 0, "fast": 8}                    # ACB_FLAG_FAST_CHANNELIZER

    # how much input one step may carry: the e2e leg pins a step's worth of host memory; if this host cannot pin
    # 12.4 GB the whole run uses half of that (all ranks agree through the min over ranks)
    cap = STEP_CAP
    pinned_pool = None                                    # allocated once, kept for the e2e leg
    if not args.no_e2e:
        for cap in (STEP_CAP, STEP_CAP // 2, STEP_CAP // 4):
            try:
                pinned_pool = api.PinnedBuffer(cap * blk_bytes)
                break
            except Exception:
                pinned_pool = None
        if pinned_pool is None:
            raise SystemExit("bench: cannot pin %d bytes of host memory for the e2e leg" % (STEP_CAP // 4 * blk_bytes))
    cap = int(-max_over_ranks(-float(cap)))

    # ---- stream-count sweep (device-resident, short): where does this GPU saturate?
    sweep = None
    if args.streams > 0:
        S = args.streams
    elif args.dump_outputs:
        S = SWEEP[-1]
    else:
        sweep = []
        for Ssw in SWEEP:
            Bsw = blocks_for(Ssw, args.blocks, cap)
            st_b = Bsw * blk_bytes
            with api.Context(K, Ssw, nch, Bsw, device=local, flags=1 | fastflag[args.channelizer]) as c:
                for s in range(Ssw):
                    c.set_plan(s, fd)
                din = DeviceInput(c, pool, Ssw, st_b)
                for _ in range(2):
                    c.submit_device(din.ptr, Bsw, st_b)
                c.sync(); c.drain_records()
                barrier()
                c.mark(0)
                for _ in range(4):
                    c.submit_device(din.ptr, Bsw, st_b)
                    c.drain_records()
                c.mark(1)
                c.sync(); c.drain_records()
                ms = max_over_ranks(c.elapsed_ms()) / 4
                din.free()
            sweep.append({"streams_per_gpu": Ssw, "blocks_per_step": Bsw, "ms_per_step": ms,
                          "value": Ssw * Bsw * 1024 * K * world / ms / 1e3})
        S = max(sweep, key=lambda r: r["value"])["streams_per_gpu"]
    B = blocks_for(S, args.blocks, cap)
    stride = B * blk_bytes
    pool_b = [p[:stride] for p in pool]
    samples_per_step_rank = S * B * 1024 * K

    def measure(channelizer: str, steps: int, warmup: int, with_e2e: bool, clk=None, dump: bool = False):
        """One context at (S, B): first pass through the host API from reset state, `warmup` + `steps` device-resident
        submits (timed with the library's CUDA events), an isolated-kernel pass, optionally the host-buffer leg."""
        out = {}
        kept, per_stream, nframes = [], np.zeros(S, dtype=np.int64), []

        take_s = [0.0]

        def take():
            # what the checker needs: every record of the distinct pool streams, and a per-stream count of the rest
            # (a step carries tens of thousands of messages at this rate: nothing else is kept)
            t_in = time.perf_counter()
            r = ctx.drain_records()
            if len(r):
                per_stream[:] += np.bincount(r["stream"], minlength=S)
                kept.append(r[r["stream"] < len(pool_b)].copy())
            nframes.append(len(r))
            take_s[0] += time.perf_counter() - t_in

        flags = fastflag[channelizer] | (0 if with_e2e else 1)
        ctx = api.Context(K, S, nch, B, device=local, flags=flags)
        for s in range(S):
            ctx.set_plan(s, fd)
        din = DeviceInput(ctx, pool_b, S, stride)
        pinned = host = None
        if with_e2e:
            pinned = pinned_pool
            host = pinned.array[:S * stride].reshape(S, stride)
            for s in range(S):
                host[s] = pool_b[s % len(pool_b)]
        # first pass from reset state (through the host path when this context has one)
        if with_e2e:
            ctx.submit_host(host, B)
        else:
            ctx.submit_device(din.ptr, B, stride)
        for _ in range(warmup):
            ctx.submit_device(din.ptr, B, stride)
            take()
        ctx.sync()
        take()
        ctx.stats(reset=True)
        n_before = len(nframes)
        if clk is not None:
            clk.start()
            time.sleep(0.3)
        barrier()
        t0 = time.perf_counter()
        ctx.mark(0)
        take_s[0] = 0.0
        for _ in range(steps):
            ctx.submit_device(din.ptr, B, stride)
            take()
        ctx.mark(1)
        ctx.sync()
        take()
        t1 = time.perf_counter()
        out["drain_ms_per_step"] = take_s[0] * 1e3 / steps      # this process draining the output queue (bench's own host work)
        ev_ms = ctx.elapsed_ms()
        barrier()
        st = ctx.stats(reset=True)
        out["ev_ms"] = max_over_ranks(ev_ms)
        out["wall_ms"] = max_over_ranks((t1 - t0) * 1e3)
        out["t0"], out["t1"] = t0, t1
        out["st"] = st
        out["recs"] = np.concatenate(kept) if kept else np.empty(0, dtype=api.MSG_DTYPE)
        out["per_stream"] = per_stream
        out["passes"] = 1 + warmup + steps
        out["frames_timed"] = int(sum(nframes[n_before:]))
        if dump:
            out["dm_last"] = ctx.read_dm(B * 1024, streams=len(pool_b))
        # isolated kernels: sync between steps, so nothing overlaps
        for _ in range(3):
            ctx.submit_device(din.ptr, B, stride)
            ctx.sync()
        ctx.drain_records()
        iso = ctx.stats(reset=True)
        out["k1_iso_ms"] = iso.chan_ms / max(1, iso.chan_launches)
        out["k2_iso_ms"] = iso.demod_ms / max(1, iso.demod_launches)
        if with_e2e:
            for _ in range(2):
                ctx.submit_host(host, B)
            ctx.sync()
            ctx.drain_records()
            ctx.stats(reset=True)
            barrier()
            e0 = time.perf_counter()
            frames_e2e = 0
            for _ in range(steps):
                ctx.submit_host(host, B)          # queues H2D + kernels; collects the submit two back
                frames_e2e += len(ctx.drain_records())    # decoded frames of completed steps, on the host
            ctx.sync()
            frames_e2e += len(ctx.drain_records())
            e1 = time.perf_counter()
            barrier()
            st2 = ctx.stats(reset=True)
            e_ms = max_over_ranks((e1 - e0) * 1e3)
            tot = sum_over_ranks(float(samples_per_step_rank * steps))
            out["e2e"] = {"value": tot / (e_ms * 1e-3) / 1e6, "unit": UNIT,
                          "h2d_bytes_per_step": S * stride * world,
                          "d2h_bytes_per_step": int((st2.raw_frames * FRAME_BYTES + 16 * st2.submits) / max(1, steps)) * world,
                          "ms_per_step": e_ms / steps, "frames_per_step": frames_e2e / steps,
                          "timing": "host wall clock between full device syncs, max over ranks"}
        din.free()
        ctx.close()
        return out

    clk = ClockSampler(local)
    main_m = measure(args.channelizer, args.steps, args.warmup, not args.no_e2e, clk, dump=bool(args.dump_outputs) and rank == 0)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, main_m, B)
    clocks = clk.summary(main_m["t0"], main_m["t1"])
    clk.stop()
    total_samples = sum_over_ranks(float(samples_per_step_rank * args.steps))
    value = total_samples / (main_m["ev_ms"] * 1e-3) / 1e6
    st = main_m["st"]
    checked = {"skipped": "rank != 0 or --no-check"}
    if do_check:
        checked = check_frames(K, pool_b, main_m["passes"], main_m["recs"], args.channelizer == "exact", S, main_m["per_stream"])
        if not (checked["bit_exact"] and checked["replicas_identical_counts"]):
            raise SystemExit("bench: GPU frames of the timed region differ from the CPU reference port")
    checked["frames_per_step_device"] = main_m["frames_timed"] / args.steps

    # ---- the other channelizer form at the same S, same treatment (its own roofline object)
    other = None
    sm_mhz = clocks.get("sm_mhz") or 1965.0
    if not args.no_alt:
        alt = "fast" if args.channelizer == "exact" else "exact"
        nst = max(3, min(args.steps, 10))
        am = measure(alt, nst, 2, False)
        k1b = am["st"].chan_ms / max(1, am["st"].chan_launches)
        chk2 = {"skipped": "rank != 0 or --no-check"}
        if do_check:
            chk2 = check_frames(K, pool_b, am["passes"], am["recs"], alt == "exact", S, am["per_stream"])
            if not chk2["bit_exact"]:
                # reported, not fatal: the line's own numbers belong to --channelizer, checked above
                print(f"bench: GPU frames ({alt} channelizer) differ from the CPU reference port", file=sys.stderr)
        other = {"channelizer": alt, "value": sum_over_ranks(float(samples_per_step_rank * nst)) / (am["ev_ms"] * 1e-3) / 1e6, "unit": UNIT,
                 "steps": nst, "ms_per_step": am["ev_ms"] / nst, "k_channelize_ms": k1b,
                 "k_demod_and_fec_ms": am["st"].demod_ms / max(1, am["st"].demod_launches),
                 "host_consumer_ms_per_step": am["st"].host_ms / max(1, am["st"].submits),
                 "fast_launches": int(am["st"].fast_chan_launches), "checked": chk2,
                 "roofline": roofline_obj(alt, am["st"].fast_chan_launches > 0, k1b, am["k1_iso_ms"], S, B, K, nch, sm_mhz)}

    # ---- the literal BASELINE configs
    configs = None
    if args.config != "none":
        import bench_configs
        want = {"2", "3", "4", "5"} if args.config == "all" else set(args.config.split(","))
        configs = bench_configs.run(want, dist, rank, world, local, dev, fastflag[args.channelizer], do_check)

    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return

    k1_ms = st.chan_ms / max(1, st.chan_launches)
    k2_ms = st.demod_ms / max(1, st.demod_launches)
    fast_ran = st.fast_chan_launches > 0
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": main_m["ev_ms"] / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": f"synthetic ({args.pool} distinct seeded streams per rank, tiled over {S})",
        "config": {"workload": f"configs[1] x {S} streams per GPU (the saturating stream count of the sweep): synthetic 2 MS/s uint8 IQ "
                               f"(K={K}), 8 ACARS channels per stream, {B} blocks of 1024*K samples per stream per step",
                   "K": K, "streams_per_gpu": S, "channels_per_stream": nch, "blocks_per_step": B, "channelizer": args.channelizer,
                   "channels_total": S * nch * world, "input_bytes_per_step_per_gpu": S * stride,
                   "l2": "inputs larger than L2 (no flush needed)" if S * stride > 200e6 else "input smaller than L2",
                   "sharding": "streams by index, no data-path collective", "timing": "CUDA events on the library's streams, max over ranks",
                   "numa_node_of_rank0": numa},
        "streams_sweep": sweep,
        "clocks": clocks,
        "e2e": main_m.get("e2e"),
        "gpu_launches": int(st.kernel_launches),
        "wall_ms_per_step": main_m["wall_ms"] / args.steps,
        "kernels": {"k_channelize_ms": k1_ms, "k_demod_and_fec_ms": k2_ms, "k_channelize_isolated_ms": main_m["k1_iso_ms"],
                    "k_demod_and_fec_isolated_ms": main_m["k2_iso_ms"], "launches_per_step": st.kernel_launches / args.steps,
                    # the library's consumer thread (frames of a finished submit -> emission order -> output queue), wall time
                    "host_consumer_ms_per_step": st.host_ms / args.steps, "host_drain_ms_per_step": main_m["drain_ms_per_step"]},
        "alt_channelizer": other,
        "configs": configs,
        "real_time_receivers": {"device_resident": value / (K * 12500 / 1e6),
                                "e2e": (main_m["e2e"]["value"] / (K * 12500 / 1e6)) if main_m.get("e2e") else None,
                                "note": "2 MS/s receivers this rate serves in real time"},
        "roofline": roofline_obj(args.channelizer, fast_ran, k1_ms, main_m["k1_iso_ms"], S, B, K, nch, sm_mhz),
        "checked": checked,
    }
    if cpu is not None:
        line["cpu_baseline"] = {k: cpu[k] for k in ("value", "unit", "cores", "kind", "sample")}
    print(json.dumps(line))
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
