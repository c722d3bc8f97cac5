"""ctypes binding of the C ABI in include/acars_b200.h.

This is host-side convenience for the tests and bench.py; the product is the shared library.
There is no CPU fallback: importing works anywhere (so the symbol tests can run on a CPU-only
box), but creating a Context without a B200 raises, and a missing libacars_b200.so raises at
import of this module.
"""
from __future__ import annotations

import ctypes as C
from pathlib import Path

import numpy as np

PKG = Path(__file__).resolve().parent
LIB_PATH = PKG / "libacars_b200.so"

OUTBLK = 1024
TXTMAX = 250


class Config(C.Structure):
    _fields_ = [("device", C.c_int), ("K", C.c_int), ("nstreams", C.c_int), ("nch", C.c_int),
                ("max_blocks", C.c_int), ("flags", C.c_int), ("taps", C.c_int)]


class Msg(C.Structure):
    _fields_ = [("stream", C.c_int), ("chn", C.c_int), ("len", C.c_int), ("err", C.c_int), ("lvl", C.c_float),
                ("block", C.c_uint64), ("pos", C.c_uint64), ("soh_pos", C.c_uint64),
                ("txt", C.c_ubyte * TXTMAX), ("crc", C.c_ubyte * 2)]

    def as_tuple(self):
        """(chn, len, err, txt, crc) — the fields the reference's msgblk_t carries."""
        return (self.chn, self.len, self.err, bytes(self.txt[:self.len]), bytes(self.crc))

    def key(self):
        return self.as_tuple() + (np.float32(self.lvl).tobytes(),)


# acb_msg_t as a numpy record (same layout as the ctypes Msg above; checked at import)
MSG_DTYPE = np.dtype([("stream", "<i4"), ("chn", "<i4"), ("len", "<i4"), ("err", "<i4"), ("lvl", "<f4"),
                      ("block", "<u8"), ("pos", "<u8"), ("soh_pos", "<u8"), ("txt", "u1", (TXTMAX,)), ("crc", "u1", (2,))],
                     align=True)
assert MSG_DTYPE.itemsize == C.sizeof(Msg)


class Fields(C.Structure):
    """acb_fields_t: outputmsg's field split + label.c's OOOI fields (include/acars_b200.h)."""
    _fields_ = [("mode", C.c_char), ("ack", C.c_char), ("bid", C.c_char), ("bs", C.c_char), ("be", C.c_char),
                ("addr", C.c_char * 8), ("label", C.c_char * 3), ("no", C.c_char * 5), ("fid", C.c_char * 7),
                ("downlink", C.c_int), ("txt_off", C.c_int), ("txt_len", C.c_int), ("has_oooi", C.c_int),
                ("da", C.c_char * 5), ("sa", C.c_char * 5), ("eta", C.c_char * 5), ("gout", C.c_char * 5),
                ("gin", C.c_char * 5), ("woff", C.c_char * 5), ("won", C.c_char * 5)]


class FmtOpts(C.Structure):
    """acb_fmt_opts_t"""
    _fields_ = [("tv_sec", C.c_int64), ("tv_usec", C.c_int64), ("freq_hz", C.c_uint), ("inmode", C.c_int),
                ("airflt", C.c_int), ("emptymsg", C.c_int), ("labels", C.c_char_p), ("station_id", C.c_char_p)]


FMT_ONELINE, FMT_FULL, FMT_JSON, FMT_NET_PP, FMT_NET_NATIVE, FMT_NET_JSON = 1, 2, 4, 11, 12, 13


class ChanState(C.Structure):
    _fields_ = [("MskPhi", C.c_double), ("MskDf", C.c_double), ("MskLvlSum", C.c_double), ("MskClk", C.c_float),
                ("MskBitCount", C.c_int), ("MskS", C.c_uint), ("idx", C.c_uint), ("nbits", C.c_int),
                ("Acarsstate", C.c_int), ("outbits", C.c_uint), ("blk_len", C.c_int), ("blk_err", C.c_int),
                ("pos", C.c_uint64), ("soh_pos", C.c_uint64), ("inb_re", C.c_float * 11), ("inb_im", C.c_float * 11),
                ("blk_crc", C.c_ubyte * 2), ("blk_txt", C.c_ubyte * TXTMAX)]

    def vec(self):
        """Same tuple shape as tests/refs.py RefState.vec() / OrcChan.vec()."""
        inb = []
        for i in range(11):
            inb += [self.inb_re[i], self.inb_im[i]]
        return (self.MskPhi, self.MskDf, self.MskLvlSum, self.MskClk, self.MskBitCount, self.MskS, self.idx,
                self.nbits, self.Acarsstate, self.outbits & 0xFF, tuple(inb))


class Stats(C.Structure):
    _fields_ = [("submits", C.c_uint64), ("kernel_launches", C.c_uint64), ("blocks", C.c_uint64),
                ("raw_frames", C.c_uint64), ("fec_dropped", C.c_uint64), ("chan_ms", C.c_double),
                ("demod_ms", C.c_double), ("chan_launches", C.c_uint64), ("demod_launches", C.c_uint64),
                ("fast_chan_launches", C.c_uint64), ("frames_lost", C.c_uint64), ("host_ms", C.c_double)]


# every symbol include/acars_b200.h declares: (name, restype, argtypes)
ABI = [
    ("acb_round_freq", C.c_int, [C.c_double]),
    ("acb_stored_fr", C.c_int, [C.c_uint]),
    ("acb_choose_fc", C.c_uint, [C.c_void_p, C.c_int, C.c_int]),
    ("acb_plan_bands", C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_int]),
    ("acb_build_wf", None, [C.c_int, C.c_uint, C.c_int, C.c_void_p]),
    ("acb_air_choose_fc", C.c_uint, [C.c_uint, C.c_uint]),
    ("acb_air_build_wf", None, [C.c_int, C.c_int, C.c_uint, C.c_void_p]),
    ("acb_cs16_build_wf", None, [C.c_int, C.c_uint, C.c_uint, C.c_int, C.c_void_p]),
    ("acb_fast_plan", C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_uint, C.c_void_p, C.c_void_p]),
    ("acb_fast_plan_cs16", C.c_int, [C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_uint, C.c_void_p, C.c_void_p]),
    ("acb_fast_plan_air", C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_uint, C.c_void_p, C.c_void_p]),
    ("acb_build_h", None, [C.c_void_p]),
    ("acb_create", C.c_int, [C.POINTER(Config), C.POINTER(C.c_void_p)]),
    ("acb_destroy", None, [C.c_void_p]),
    ("acb_last_error", C.c_char_p, []),
    ("acb_version", C.c_char_p, []),
    ("acb_set_plan", C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.POINTER(C.c_uint)]),
    ("acb_set_plan_air", C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.POINTER(C.c_uint)]),
    ("acb_set_plan_cs16", C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_uint, C.POINTER(C.c_uint)]),
    ("acb_set_plan_at", C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_uint]),
    ("acb_set_wf", C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_int]),
    ("acb_reset", C.c_int, [C.c_void_p]),
    ("acb_submit_host", C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t, C.c_int]),
    ("acb_submit_device", C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t, C.c_int]),
    ("acb_submit_real_host", C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t, C.c_size_t]),
    ("acb_submit_cs16_host", C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t, C.c_size_t]),
    ("acb_submit_cs16_planar_host", C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_size_t]),
    ("acb_set_emission_groups", C.c_int, [C.c_void_p, C.c_int, C.c_uint64]),
    ("acb_submit_dm_host", C.c_int, [C.c_void_p, C.c_void_p, C.c_int]),
    ("acb_sync", C.c_int, [C.c_void_p]),
    ("acb_collect", C.c_int, [C.c_void_p]),
    ("acb_wait_event", C.c_int, [C.c_void_p, C.c_void_p]),
    ("acb_multi_create", C.c_int, [C.POINTER(Config), C.c_void_p, C.c_int, C.c_int, C.POINTER(C.c_void_p)]),
    ("acb_multi_destroy", None, [C.c_void_p]),
    ("acb_multi_parts", C.c_int, [C.c_void_p]),
    ("acb_multi_part", C.c_void_p, [C.c_void_p, C.c_int]),
    ("acb_multi_set_plan", C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.POINTER(C.c_uint)]),
    ("acb_multi_set_wf", C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_int]),
    ("acb_multi_reset", C.c_int, [C.c_void_p]),
    ("acb_multi_submit_host", C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t, C.c_int]),
    ("acb_multi_collect", C.c_int, [C.c_void_p]),
    ("acb_multi_sync", C.c_int, [C.c_void_p]),
    ("acb_multi_drain", C.c_int, [C.c_void_p, C.POINTER(Msg), C.c_int]),
    ("acb_multi_get_state", C.c_int, [C.c_void_p, C.c_int, C.c_int, C.POINTER(ChanState)]),
    ("acb_multi_set_state", C.c_int, [C.c_void_p, C.c_int, C.c_int, C.POINTER(ChanState)]),
    ("acb_mark", C.c_int, [C.c_void_p, C.c_int]),
    ("acb_elapsed_ms", C.c_int, [C.c_void_p, C.POINTER(C.c_float)]),
    ("acb_msg_fields", C.c_int, [C.POINTER(Msg), C.POINTER(Fields)]),
    ("acb_format_msg", C.c_int, [C.POINTER(Msg), C.c_int, C.POINTER(FmtOpts), C.c_char_p, C.c_size_t]),
    ("acb_flights_new", C.c_void_p, [C.c_int]),
    ("acb_flights_free", None, [C.c_void_p]),
    ("acb_flights_route_json", C.c_int, [C.c_void_p, C.POINTER(Msg), C.POINTER(FmtOpts), C.c_char_p, C.c_size_t]),
    ("acb_flights_monitor", C.c_int, [C.c_void_p, C.POINTER(Msg), C.c_int, C.POINTER(FmtOpts), C.c_char_p, C.c_size_t]),
    ("acb_drain", C.c_int, [C.c_void_p, C.POINTER(Msg), C.c_int]),
    ("acb_pending", C.c_int, [C.c_void_p]),
    ("acb_host_alloc", C.c_void_p, [C.c_size_t]),
    ("acb_host_free", None, [C.c_void_p]),
    ("acb_device_alloc", C.c_void_p, [C.c_void_p, C.c_size_t]),
    ("acb_device_free", None, [C.c_void_p, C.c_void_p]),
    ("acb_copy_to_device", C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t]),
    ("acb_read_dm", C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t]),
    ("acb_get_state", C.c_int, [C.c_void_p, C.c_int, C.c_int, C.POINTER(ChanState)]),
    ("acb_set_state", C.c_int, [C.c_void_p, C.c_int, C.c_int, C.POINTER(ChanState)]),
    ("acb_get_stats", C.c_int, [C.c_void_p, C.POINTER(Stats), C.c_int]),
    ("acb_block_fec", C.c_int, [C.POINTER(Msg)]),
    ("acb_block_fec_batch", C.c_int, [C.c_void_p, C.POINTER(Msg), C.c_int, C.POINTER(C.c_int)]),
    ("acb_crc_update", C.c_uint16, [C.c_uint16, C.c_uint8]),
    ("acb_syndrome", C.c_uint16, [C.c_int]),
    ("acb_frame_byte", None, [C.c_void_p, C.c_ubyte]),
]

_lib = None


def load():
    """Load libacars_b200.so (built in-tree by acarsdec_b200.build); raises if it is missing."""
    global _lib
    if _lib is None:
        if not LIB_PATH.exists():
            raise ImportError(f"{LIB_PATH} is missing: run `python -m acarsdec_b200.build` (needs nvcc). "
                              "There is no CPU fallback.")
        lib = C.CDLL(str(LIB_PATH))
        for name, res, args in ABI:
            fn = getattr(lib, name)     # AttributeError if the library does not export it
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib


class AcbError(RuntimeError):
    pass


def _check(lib, rc: int) -> int:
    if rc < 0:
        raise AcbError(f"acars_b200 error {rc}: {lib.acb_last_error().decode()}")
    return rc


# ---- front-end planning (host; same results as initRtl) ----

def plan(K: int, freqs_mhz):
    """(freqs_hz, stored Fr, Fc) as initRtl derives them (rtl.c:243-268)."""
    lib = load()
    fd = np.array([lib.acb_round_freq(float(f)) for f in freqs_mhz], dtype=np.uint32)
    fc = lib.acb_choose_fc(fd.ctypes.data, len(fd), K)
    return [int(f) for f in fd], [lib.acb_stored_fr(int(f)) for f in fd], int(fc)


def plan_bands(K: int, freqs_hz, max_groups: int = 64):
    """Fewest receiver bands covering `freqs_hz` (any span): (band index per channel, centre per band)."""
    lib = load()
    f = np.asarray(freqs_hz, dtype=np.uint32)
    grp = np.zeros(len(f), dtype=np.int32)
    fc = np.zeros(max_groups, dtype=np.uint32)
    n = lib.acb_plan_bands(f.ctypes.data, len(f), K, grp.ctypes.data, fc.ctypes.data, max_groups)
    if n < 0:
        raise AcbError(f"acb_plan_bands failed ({n})")
    return grp, fc[:n]


def build_wf(K: int, freqs_mhz) -> np.ndarray:
    lib = load()
    _, fr, fc = plan(K, freqs_mhz)
    out = np.empty((len(fr), 2 * K), dtype=np.float32)
    for i, f in enumerate(fr):
        lib.acb_build_wf(f, fc, K, out[i].ctypes.data)
    return out


def fast_plan(K: int, freqs_hz, fc: int):
    """Planning step of the fast channelizer: (k per channel, twiddles (nch, K/4) complex64), or None when
    some channel is off the 12.5 kHz raster around Fc (the exact kernel runs then)."""
    lib = load()
    f = np.asarray(freqs_hz, dtype=np.uint32)
    k = np.zeros(len(f), dtype=np.int32)
    tw = np.zeros((len(f), K // 4, 2), dtype=np.float32)
    if lib.acb_fast_plan(f.ctypes.data, len(f), K, fc, k.ctypes.data, tw.ctypes.data) != 1:
        return None
    return k, tw[..., 0] + 1j * tw[..., 1]


def msg_fields(m: Msg) -> Fields | None:
    f = Fields()
    return f if load().acb_msg_fields(C.byref(m), C.byref(f)) == 1 else None


def format_msg(m: Msg, fmt: int, *, tv_sec: int = 0, tv_usec: int = 0, freq_hz: int = 0, inmode: int = 0, airflt: bool = False,
               emptymsg: bool = False, labels: str | None = None, station_id: str | None = None) -> bytes | None:
    """One decoded block in one of the reference's wire formats (FMT_*), byte for byte; None when a filter drops it."""
    o = FmtOpts(tv_sec, tv_usec, freq_hz, inmode, int(airflt), int(emptymsg),
                labels.encode() if labels else None, station_id.encode() if station_id else None)
    buf = C.create_string_buffer(8192)
    n = load().acb_format_msg(C.byref(m), fmt, C.byref(o), buf, len(buf))
    if n < 0:
        raise AcbError(f"acb_format_msg: error {n} (bad block, unknown format or buffer too small)")
    return buf.raw[:n] if n else None


class Flights:
    """The flight table behind acarsdec's route JSON (-o 5) and monitor screen (-o 3): feed every block in emission order."""

    def __init__(self, mdly_seconds: int = 600):
        self.lib = load()
        self.h = C.c_void_p(self.lib.acb_flights_new(mdly_seconds))
        if not self.h:
            raise AcbError("acb_flights_new failed")

    @staticmethod
    def _opts(kw):
        lab, sta = kw.get("labels"), kw.get("station_id")
        return FmtOpts(kw.get("tv_sec", 0), kw.get("tv_usec", 0), kw.get("freq_hz", 0), kw.get("inmode", 0), int(kw.get("airflt", False)),
                       int(kw.get("emptymsg", False)), lab.encode() if lab else None, sta.encode() if sta else None)

    def _call(self, fn, *args):
        buf = C.create_string_buffer(16384)
        n = fn(*args, buf, len(buf))
        if n < 0:
            raise AcbError(f"flight table: error {n}")
        return buf.raw[:n] if n else None

    def route_json(self, m: Msg, **kw) -> bytes | None:
        o = self._opts(kw)
        return self._call(self.lib.acb_flights_route_json, self.h, C.byref(m), C.byref(o))

    def monitor(self, m: Msg, nbch: int, **kw) -> bytes | None:
        o = self._opts(kw)
        return self._call(self.lib.acb_flights_monitor, self.h, C.byref(m), nbch, C.byref(o))

    def close(self):
        if self.h:
            self.lib.acb_flights_free(self.h)
            self.h = None

    def __del__(self):
        self.close()


def air_plan(rate: int, freqs_mhz):
    """(freqs_hz, Fc, K) as initAirspy derives them (air.c:165-242, no-filter rates)."""
    lib = load()
    fd = [lib.acb_round_freq(float(f)) for f in freqs_mhz]
    return fd, int(lib.acb_air_choose_fc(min(fd), max(fd))), rate // 12500


def build_wf_air(rate: int, freqs_mhz) -> np.ndarray:
    lib = load()
    fd, fc, K = air_plan(rate, freqs_mhz)
    out = np.empty((len(fd), 2 * K), dtype=np.float32)
    for i, f in enumerate(fd):
        lib.acb_air_build_wf(f, fc, rate, out[i].ctypes.data)
    return out


def build_wf_cs16(variant: int, K: int, freqs_hz, fc_hz: int) -> np.ndarray:
    lib = load()
    out = np.empty((len(freqs_hz), 2 * K), dtype=np.float32)
    for i, f in enumerate(freqs_hz):
        lib.acb_cs16_build_wf(variant, int(f), int(fc_hz), K, out[i].ctypes.data)
    return out


def build_h() -> np.ndarray:
    h = np.empty(133, dtype=np.float32)
    load().acb_build_h(h.ctypes.data)
    return h


def block_fec(msg: Msg):
    out = Msg()
    C.memmove(C.byref(out), C.byref(msg), C.sizeof(Msg))
    return out if load().acb_block_fec(C.byref(out)) else None


class PinnedBuffer:
    """uint8 numpy view over cudaHostAlloc memory (acb_host_alloc)."""

    def __init__(self, nbytes: int):
        self.lib = load()
        self.ptr = self.lib.acb_host_alloc(nbytes)
        if not self.ptr:
            raise AcbError(self.lib.acb_last_error().decode())
        self.nbytes = nbytes
        self.array = np.ctypeslib.as_array((C.c_uint8 * nbytes).from_address(self.ptr))

    def close(self):
        if self.ptr:
            self.lib.acb_host_free(self.ptr)
            self.ptr = None

    def __del__(self):
        self.close()


class Context:
    """N streams x C channels on one GPU (acb_ctx_t)."""

    def __init__(self, K: int, nstreams: int, nch: int, max_blocks: int, device: int = 0, flags: int = 0, taps: int = 0):
        self.lib = load()
        self.K, self.nstreams, self.nch, self.max_blocks = K, nstreams, nch, max_blocks
        self.block_bytes = OUTBLK * K * 2
        cfg = Config(device, K, nstreams, nch, max_blocks, flags, taps)
        h = C.c_void_p()
        rc = self.lib.acb_create(C.byref(cfg), C.byref(h))
        if rc < 0:
            msg = self.lib.acb_last_error().decode()
            if h:
                self.lib.acb_destroy(h)
            raise AcbError(f"acb_create failed ({rc}): {msg}")
        self.h = h

    def close(self):
        if getattr(self, "h", None):
            self.lib.acb_destroy(self.h)
            self.h = None

    def __del__(self):
        self.close()

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def set_plan(self, stream: int, freqs_hz) -> int:
        f = np.asarray(freqs_hz, dtype=np.uint32)
        fc = C.c_uint()
        _check(self.lib, self.lib.acb_set_plan(self.h, stream, f.ctypes.data, len(f), C.byref(fc)))
        return fc.value

    def set_wf(self, stream: int, wf: np.ndarray) -> None:
        wf = np.ascontiguousarray(wf, dtype=np.float32)
        _check(self.lib, self.lib.acb_set_wf(self.h, stream, wf.ctypes.data, wf.shape[0]))

    def reset(self) -> None:
        _check(self.lib, self.lib.acb_reset(self.h))

    def submit_host(self, iq, nblk: int, stream_stride: int | None = None) -> None:
        """iq: uint8 array (nstreams, nblk*block_bytes) or a raw pointer + stride."""
        if isinstance(iq, np.ndarray):
            assert iq.dtype == np.uint8 and iq.flags.c_contiguous
            ptr = iq.ctypes.data
            if stream_stride is None:
                stream_stride = iq.strides[0] if iq.ndim == 2 else nblk * self.block_bytes
        else:
            ptr = iq
        _check(self.lib, self.lib.acb_submit_host(self.h, ptr, stream_stride, nblk))

    def submit_device(self, dev_ptr: int, nblk: int, stream_stride: int) -> None:
        _check(self.lib, self.lib.acb_submit_device(self.h, dev_ptr, stream_stride, nblk))

    def set_plan_air(self, stream: int, freqs_hz) -> int:
        f = np.asarray(freqs_hz, dtype=np.uint32)
        fc = C.c_uint()
        _check(self.lib, self.lib.acb_set_plan_air(self.h, stream, f.ctypes.data, len(f), C.byref(fc)))
        return fc.value

    def submit_real(self, x: np.ndarray) -> int:
        """x: float32 (nstreams, nsamples) real samples; returns envelope samples produced per channel."""
        assert x.dtype == np.float32 and x.ndim == 2 and x.shape[0] == self.nstreams and x.strides[1] == 4
        return _check(self.lib, self.lib.acb_submit_real_host(self.h, x.ctypes.data, x.strides[0] // 4, x.shape[1]))

    def set_plan_cs16(self, stream: int, freqs_hz, variant: int, fc_hz: int = 0) -> int:
        f = np.asarray(freqs_hz, dtype=np.uint32)
        fc = C.c_uint()
        _check(self.lib, self.lib.acb_set_plan_cs16(self.h, stream, f.ctypes.data, len(f), variant, fc_hz, C.byref(fc)))
        return fc.value

    def submit_cs16(self, iq: np.ndarray) -> int:
        """iq: int16 (nstreams, nsamples, 2) interleaved I,Q."""
        assert iq.dtype == np.int16 and iq.ndim == 3 and iq.shape[0] == self.nstreams and iq.shape[2] == 2 and iq.flags.c_contiguous
        return _check(self.lib, self.lib.acb_submit_cs16_host(self.h, iq.ctypes.data, iq.shape[1], iq.shape[1]))

    def submit_cs16_planar(self, xi: np.ndarray, xq: np.ndarray) -> int:
        """xi, xq: int16 (nstreams, nsamples) separate I and Q planes (the SDRplay callback's layout)."""
        assert xi.dtype == np.int16 and xq.dtype == np.int16 and xi.shape == xq.shape and xi.flags.c_contiguous and xq.flags.c_contiguous
        return _check(self.lib, self.lib.acb_submit_cs16_planar_host(self.h, xi.ctypes.data, xq.ctypes.data, xi.shape[1], xi.shape[1]))

    def set_emission_groups(self, unit: int, period: int = 0) -> None:
        """unit: 0 per submit, 1 every `period` envelope samples, 2 per transfer of `period` input samples."""
        _check(self.lib, self.lib.acb_set_emission_groups(self.h, unit, period))

    def submit_dm(self, dm: np.ndarray) -> None:
        """dm: float32 (nstreams, nsamp, nch)."""
        dm = np.ascontiguousarray(dm, dtype=np.float32)
        assert dm.shape[0] == self.nstreams and dm.shape[2] == self.nch
        _check(self.lib, self.lib.acb_submit_dm_host(self.h, dm.ctypes.data, dm.shape[1]))

    def sync(self) -> int:
        return _check(self.lib, self.lib.acb_sync(self.h))

    def collect(self) -> int:
        return _check(self.lib, self.lib.acb_collect(self.h))

    def mark(self, which: int) -> None:
        _check(self.lib, self.lib.acb_mark(self.h, which))

    def elapsed_ms(self) -> float:
        ms = C.c_float()
        _check(self.lib, self.lib.acb_elapsed_ms(self.h, C.byref(ms)))
        return ms.value

    def drain(self):
        out = []
        buf = (Msg * 256)()
        while True:
            n = self.lib.acb_drain(self.h, buf, 256)
            for i in range(n):
                m = Msg()
                C.memmove(C.byref(m), C.byref(buf[i]), C.sizeof(Msg))
                out.append(m)
            if n < 256:
                return out

    def pending(self) -> int:
        return self.lib.acb_pending(self.h)

    def drain_records(self) -> np.ndarray:
        """All queued messages as one numpy record array (MSG_DTYPE), one C call."""
        n = self.lib.acb_pending(self.h)
        buf = np.empty(n, dtype=MSG_DTYPE)
        if n:
            got = self.lib.acb_drain(self.h, buf.ctypes.data_as(C.POINTER(Msg)), n)
            buf = buf[:got]
        return buf

    def block_fec_batch(self, msgs):
        """Device block FEC over a list of raw Msg (parity-bearing txt): returns [fixed Msg or None]."""
        n = len(msgs)
        arr = (Msg * n)()
        for i, m in enumerate(msgs):
            C.memmove(C.byref(arr[i]), C.byref(m), C.sizeof(Msg))
        keep = (C.c_int * n)()
        _check(self.lib, self.lib.acb_block_fec_batch(self.h, arr, n, keep))
        out = []
        for i in range(n):
            if keep[i]:
                m = Msg()
                C.memmove(C.byref(m), C.byref(arr[i]), C.sizeof(Msg))
                out.append(m)
            else:
                out.append(None)
        return out

    def read_dm(self, nsamp: int, streams: int | None = None) -> np.ndarray:
        """Envelope of the last submit, (streams, nsamp, nch): all streams, or the first `streams`."""
        out = np.empty((self.nstreams if streams is None else streams, nsamp, self.nch), dtype=np.float32)
        _check(self.lib, self.lib.acb_read_dm(self.h, out.ctypes.data, out.size))
        return out

    def get_state(self, stream: int, chn: int) -> ChanState:
        s = ChanState()
        _check(self.lib, self.lib.acb_get_state(self.h, stream, chn, C.byref(s)))
        return s

    def set_state(self, stream: int, chn: int, s: ChanState) -> None:
        _check(self.lib, self.lib.acb_set_state(self.h, stream, chn, C.byref(s)))

    def stats(self, reset: bool = False) -> Stats:
        s = Stats()
        _check(self.lib, self.lib.acb_get_stats(self.h, C.byref(s), int(reset)))
        return s

    def device_alloc(self, nbytes: int) -> int:
        p = self.lib.acb_device_alloc(self.h, nbytes)
        if not p:
            raise AcbError(self.lib.acb_last_error().decode())
        return p

    def device_free(self, p: int) -> None:
        self.lib.acb_device_free(self.h, p)

    def copy_to_device(self, dst: int, src: np.ndarray) -> None:
        src = np.ascontiguousarray(src)
        _check(self.lib, self.lib.acb_copy_to_device(self.h, dst, src.ctypes.data, src.nbytes))

    def set_plan_at(self, stream: int, freqs_hz, fc_hz: int) -> None:
        f = np.asarray(freqs_hz, dtype=np.uint32)
        _check(self.lib, self.lib.acb_set_plan_at(self.h, stream, f.ctypes.data, len(f), int(fc_hz)))

    def wait_event(self, cuda_event: int) -> None:
        """Order the next submit_device behind a cudaEvent_t of another stream (torch.cuda.Event.cuda_event)."""
        _check(self.lib, self.lib.acb_wait_event(self.h, cuda_event))


class MultiContext:
    """acb_multi_t: one process, several GPUs; streams (mode 0) or channels (mode 1) split among them."""

    def __init__(self, K: int, nstreams: int, nch: int, max_blocks: int, devices, mode: int = 0, flags: int = 0, taps: int = 0):
        self.lib = load()
        self.K, self.nstreams, self.nch = K, nstreams, nch
        cfg = Config(0, K, nstreams, nch, max_blocks, flags, taps)
        dev = np.asarray(list(devices), dtype=np.int32)
        h = C.c_void_p()
        rc = self.lib.acb_multi_create(C.byref(cfg), dev.ctypes.data, len(dev), mode, C.byref(h))
        if rc < 0:
            msg = self.lib.acb_last_error().decode()
            if h:
                self.lib.acb_multi_destroy(h)
            raise AcbError(f"acb_multi_create failed ({rc}): {msg}")
        self.h = h

    def close(self):
        if getattr(self, "h", None):
            self.lib.acb_multi_destroy(self.h)
            self.h = None

    __del__ = close

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def parts(self) -> int:
        return self.lib.acb_multi_parts(self.h)

    def set_plan(self, stream: int, freqs_hz) -> int:
        f = np.asarray(freqs_hz, dtype=np.uint32)
        fc = C.c_uint()
        _check(self.lib, self.lib.acb_multi_set_plan(self.h, stream, f.ctypes.data, len(f), C.byref(fc)))
        return fc.value

    def set_wf(self, stream: int, wf: np.ndarray) -> None:
        wf = np.ascontiguousarray(wf, dtype=np.float32)
        _check(self.lib, self.lib.acb_multi_set_wf(self.h, stream, wf.ctypes.data, wf.shape[0]))

    def submit_host(self, iq: np.ndarray, nblk: int) -> None:
        assert iq.dtype == np.uint8 and iq.flags.c_contiguous
        stride = iq.strides[0] if iq.ndim == 2 else nblk * OUTBLK * self.K * 2
        _check(self.lib, self.lib.acb_multi_submit_host(self.h, iq.ctypes.data, stride, nblk))

    def sync(self) -> int:
        return _check(self.lib, self.lib.acb_multi_sync(self.h))

    def collect(self) -> int:
        return _check(self.lib, self.lib.acb_multi_collect(self.h))

    def drain(self):
        out = []
        buf = (Msg * 256)()
        while True:
            n = self.lib.acb_multi_drain(self.h, buf, 256)
            for i in range(n):
                m = Msg()
                C.memmove(C.byref(m), C.byref(buf[i]), C.sizeof(Msg))
                out.append(m)
            if n < 256:
                return out

    def get_state(self, stream: int, chn: int) -> ChanState:
        s = ChanState()
        _check(self.lib, self.lib.acb_multi_get_state(self.h, stream, chn, C.byref(s)))
        return s
