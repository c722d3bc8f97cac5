"""ctypes front-ends for the two CPU checkers under oracle/ (TEST INFRASTRUCTURE).

RefLib    — oracle/_ref/libacarsref_*.so: the unmodified reference compiled in place.
            It is process-global (the reference keeps its state in globals), so one
            instance at a time per process.
OracleLib — oracle/libacars_oracle.so: the re-entrant C restatement.
Recorded  — what the reference returned in one test, replayed from tests/golden/reference/.
"""
from __future__ import annotations

import contextlib
import ctypes as C
import gzip
import hashlib
import json
import os
import re
import subprocess
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
ORACLE_DIR = ROOT / "oracle"
RECORDINGS = ROOT / "tests" / "golden" / "reference"
RECORD = os.environ.get("ACB_RECORD_REFERENCE") == "1"


def ensure_built() -> None:
    """Build oracle/ (and oracle/_ref when /root/reference exists); no-op when up to date."""
    subprocess.run(["make", "-s", "-C", str(ORACLE_DIR), "all"], check=True,
                   stdout=subprocess.DEVNULL)


class Msg(C.Structure):
    _fields_ = [("chn", C.c_int), ("len", C.c_int), ("err", C.c_int), ("lvl", C.c_float),
                ("txt", C.c_ubyte * 250), ("crc", C.c_ubyte * 2)]

    def as_tuple(self):
        return (self.chn, self.len, self.err, bytes(self.txt[:self.len]), bytes(self.crc))

    def key(self):
        return self.as_tuple() + (np.float32(self.lvl).tobytes(),)


class RefState(C.Structure):
    _fields_ = [("MskPhi", C.c_double), ("MskDf", C.c_double), ("MskLvlSum", C.c_double),
                ("MskClk", C.c_float), ("MskBitCount", C.c_int), ("MskS", C.c_uint), ("idx", C.c_uint),
                ("nbits", C.c_int), ("state", C.c_int), ("outbits", C.c_ubyte), ("inb", C.c_float * 22)]

    def vec(self):
        return (self.MskPhi, self.MskDf, self.MskLvlSum, self.MskClk, self.MskBitCount, self.MskS,
                self.idx, self.nbits, self.state, self.outbits, tuple(self.inb))


class OrcChan(C.Structure):
    _fields_ = [("chn", C.c_int), ("MskPhi", C.c_double), ("MskDf", C.c_double), ("MskLvlSum", C.c_double),
                ("MskClk", C.c_float), ("MskBitCount", C.c_int), ("MskS", C.c_uint), ("idx", C.c_uint),
                ("inb_re", C.c_float * 11), ("inb_im", C.c_float * 11), ("outbits", C.c_ubyte),
                ("nbits", C.c_int), ("state", C.c_int), ("have_blk", C.c_int), ("blk", Msg),
                ("nbit_total", C.c_uint64)]

    def vec(self):
        inb = []
        for i in range(11):
            inb += [self.inb_re[i], self.inb_im[i]]
        return (self.MskPhi, self.MskDf, self.MskLvlSum, self.MskClk, self.MskBitCount, self.MskS,
                self.idx, self.nbits, self.state, self.outbits, tuple(inb))


class OrcSink(C.Structure):
    _fields_ = [("msgs", C.POINTER(Msg)), ("nmsg", C.c_int), ("capmsg", C.c_int),
                ("bits", C.POINTER(C.c_uint8)), ("nbits", C.c_int64), ("capbits", C.c_int64)]


def ref_available(variant: str = "O2") -> bool:
    return (ORACLE_DIR / "_ref" / f"libacarsref_{variant}.so").exists()


def best_fast_variant() -> str:
    """-Ofast build matching the host: AVX-512 when the CPU has it, else AVX2+FMA."""
    try:
        flags = open("/proc/cpuinfo").read()
    except OSError:
        flags = ""
    return "v4" if " avx512f" in flags and " avx512vl" in flags and " avx512bw" in flags else "v3"


class RefLib:
    def __init__(self, variant: str = "O2"):
        self.lib = C.CDLL(str(ORACLE_DIR / "_ref" / f"libacarsref_{variant}.so"))
        L = self.lib
        L.ref_open_rtl.argtypes = [C.c_int, C.c_int, C.POINTER(C.c_char_p)]
        L.ref_rtl_block.argtypes = [C.c_void_p, C.c_uint]
        L.ref_rtl_run.argtypes = [C.c_void_p, C.c_uint, C.c_int, C.c_int]
        L.ref_get_wf.argtypes = [C.c_int, C.c_void_p]
        L.ref_get_dm.argtypes = [C.c_int, C.c_void_p, C.c_int]
        L.ref_audio_chunk.argtypes = [C.c_int, C.c_void_p, C.c_int]
        L.ref_state.argtypes = [C.c_int, C.POINTER(RefState)]
        L.ref_msgs.argtypes = [C.POINTER(Msg), C.c_int]
        L.ref_center_freq.restype = C.c_uint
        L.ref_tab_syndrom.argtypes = [C.c_void_p, C.c_int]
        L.ref_tab_crc.argtypes = [C.c_void_p]
        L.ref_tab_numbits.argtypes = [C.c_void_p]
        L.ref_tap_push_block.argtypes = [C.c_int, C.c_int, C.c_char_p, C.c_char_p]
        self.K = None

    def open_rtl(self, K: int, freqs_mhz) -> None:
        strs = [("%.4f" % f).encode() for f in freqs_mhz]
        arr = (C.c_char_p * len(strs))(*strs)
        r = self.lib.ref_open_rtl(K, len(strs), arr)
        if r:
            raise RuntimeError(f"ref_open_rtl -> {r}")
        self.K = K

    def open_audio(self, nch: int) -> None:
        if self.lib.ref_open_audio(nch):
            raise RuntimeError("ref_open_audio failed")

    @property
    def nbch(self) -> int:
        return self.lib.ref_nbch()

    @property
    def fc(self) -> int:
        return self.lib.ref_center_freq()

    def chan_freq(self, ch: int) -> int:
        return self.lib.ref_chan_freq(ch)

    def wf(self, ch: int) -> np.ndarray:
        out = np.empty(2 * self.K, dtype=np.float32)
        self.lib.ref_get_wf(ch, out.ctypes.data)
        return out

    def block(self, buf: np.ndarray) -> None:
        assert buf.dtype == np.uint8 and buf.flags.c_contiguous
        self.lib.ref_rtl_block(buf.ctypes.data, buf.size)

    def run(self, bufs: np.ndarray, nblk: int) -> None:
        assert bufs.dtype == np.uint8 and bufs.flags.c_contiguous and bufs.ndim == 2
        self.lib.ref_rtl_run(bufs.ctypes.data, bufs.shape[1], bufs.shape[0], nblk)

    def dm(self, ch: int, n: int = 1024) -> np.ndarray:
        out = np.empty(n, dtype=np.float32)
        self.lib.ref_get_dm(ch, out.ctypes.data, n)
        return out

    def audio(self, ch: int, x: np.ndarray) -> None:
        x = np.ascontiguousarray(x, dtype=np.float32)
        self.lib.ref_audio_chunk(ch, x.ctypes.data, len(x))

    def state(self, ch: int) -> RefState:
        s = RefState()
        self.lib.ref_state(ch, C.byref(s))
        return s

    def msgs(self, flush: bool = True):
        if flush:
            self.lib.ref_flush()
        out = []
        buf = (Msg * 256)()
        while True:
            n = self.lib.ref_msgs(buf, 256)
            for i in range(n):
                m = Msg()
                C.memmove(C.byref(m), C.byref(buf[i]), C.sizeof(Msg))
                out.append(m)
            if n < 256:
                return out

    def push_block(self, chn: int, txt: bytes, crc: bytes) -> None:
        """Feed one pre-FEC block straight into the reference's blk_thread queue."""
        self.lib.ref_tap_push_block(chn, len(txt), bytes(txt), bytes(crc))

    def tables(self):
        n = self.lib.ref_tab_syndrom(None, 0)
        syn = np.empty(n, dtype=np.uint16)
        self.lib.ref_tab_syndrom(syn.ctypes.data, n)
        crc = np.empty(256, dtype=np.uint16)
        self.lib.ref_tab_crc(crc.ctypes.data)
        nb = np.empty(256, dtype=np.uint8)
        self.lib.ref_tab_numbits(nb.ctypes.data)
        return syn, crc, nb

    def close(self) -> None:
        self.lib.ref_close()


class RefAirLib:
    """oracle/_ref/libacarsref_air_O2.so: the reference's air.c front-end compiled in place."""

    def __init__(self):
        self.lib = C.CDLL(str(ORACLE_DIR / "_ref" / "libacarsref_air_O2.so"))
        L = self.lib
        L.ref_air_open.argtypes = [C.c_uint, C.c_int, C.POINTER(C.c_char_p)]
        L.ref_air_transfer.argtypes = [C.c_void_p, C.c_int]
        L.ref_get_wf.argtypes = [C.c_int, C.c_void_p]
        L.ref_get_dm.argtypes = [C.c_int, C.c_void_p, C.c_int]
        L.ref_state.argtypes = [C.c_int, C.POINTER(RefState)]
        L.ref_msgs.argtypes = [C.POINTER(Msg), C.c_int]
        L.ref_air_fc.restype = C.c_uint
        L.ref_air_mult.restype = C.c_uint

    def open(self, rate: int, freqs_mhz) -> None:
        strs = [("%.4f" % f).encode() for f in freqs_mhz]
        arr = (C.c_char_p * len(strs))(*strs)
        if self.lib.ref_air_open(rate, len(strs), arr):
            raise RuntimeError("ref_air_open failed")
        self.K = self.lib.ref_air_mult()

    @property
    def fc(self) -> int:
        return self.lib.ref_air_fc()

    def wf(self, ch: int) -> np.ndarray:
        out = np.empty(2 * self.K, dtype=np.float32)
        self.lib.ref_get_wf(ch, out.ctypes.data)
        return out

    def transfer(self, x: np.ndarray) -> int:
        x = np.ascontiguousarray(x, dtype=np.float32)
        return self.lib.ref_air_transfer(x.ctypes.data, len(x))

    def dm(self, ch: int, n: int) -> np.ndarray:
        out = np.empty(n, dtype=np.float32)
        self.lib.ref_get_dm(ch, out.ctypes.data, n)
        return out

    def state(self, ch: int) -> RefState:
        s = RefState()
        self.lib.ref_state(ch, C.byref(s))
        return s

    def msgs(self):
        self.lib.ref_flush()
        out = []
        buf = (Msg * 256)()
        while True:
            n = self.lib.ref_msgs(buf, 256)
            for i in range(n):
                m = Msg()
                C.memmove(C.byref(m), C.byref(buf[i]), C.sizeof(Msg))
                out.append(m)
            if n < 256:
                return out

    def close(self) -> None:
        self.lib.ref_close()


class RefCs16Lib:
    """oracle/_ref/libacarsref_{soapy,sdrplay}_O2.so: the reference's CS16 front-ends in place."""

    def __init__(self, which: str):
        self.which = which
        self.lib = C.CDLL(str(ORACLE_DIR / "_ref" / f"libacarsref_{which}_O2.so"))
        L = self.lib
        L.ref_get_osc.argtypes = [C.c_int, C.c_void_p, C.c_int]
        L.ref_get_dm.argtypes = [C.c_int, C.c_void_p, C.c_int]
        L.ref_get_carry.argtypes = [C.c_int, C.c_void_p]
        L.ref_state.argtypes = [C.c_int, C.POINTER(RefState)]
        L.ref_msgs.argtypes = [C.POINTER(Msg), C.c_int]
        if which == "soapy":
            L.ref_soapy_open.argtypes = [C.c_int, C.c_int, C.c_int, C.POINTER(C.c_char_p)]
            L.ref_soapy_feed.argtypes = [C.c_void_p, C.c_size_t, C.c_void_p, C.c_int]
        else:
            L.ref_sdrplay_open.argtypes = [C.c_int, C.POINTER(C.c_char_p)]
            L.ref_sdrplay_packet.argtypes = [C.c_void_p, C.c_void_p, C.c_uint]
            L.ref_sdrplay_fc.restype = C.c_uint

    def open(self, freqs_mhz, K: int = 160, user_freq: int = 0) -> None:
        strs = [("%.4f" % f).encode() for f in freqs_mhz]
        arr = (C.c_char_p * len(strs))(*strs)
        r = self.lib.ref_soapy_open(K, user_freq, len(strs), arr) if self.which == "soapy" else self.lib.ref_sdrplay_open(len(strs), arr)
        if r:
            raise RuntimeError(f"open failed: {r}")
        self.K = K if self.which == "soapy" else 160

    @property
    def fc(self) -> int:
        return self.lib.ref_soapy_fc() if self.which == "soapy" else self.lib.ref_sdrplay_fc()

    def osc(self, ch: int) -> np.ndarray:
        out = np.empty(2 * self.K, dtype=np.float32)
        self.lib.ref_get_osc(ch, out.ctypes.data, self.K)
        return out

    def feed(self, iq: np.ndarray, sizes) -> None:
        """iq: int16 (n, 2).  soapy: one run of the read loop with the given read sizes (cycled);
        sdrplay: one callback per size, planar xi/xq."""
        iq = np.ascontiguousarray(iq, dtype=np.int16)
        if self.which == "soapy":
            sz = np.asarray(sizes, dtype=np.int32)
            self.lib.ref_soapy_feed(iq.ctypes.data, len(iq), sz.ctypes.data, len(sz))
        else:
            pos, i = 0, 0
            while pos < len(iq):
                n = min(int(sizes[i % len(sizes)]), len(iq) - pos)
                xi = np.ascontiguousarray(iq[pos:pos + n, 0])
                xq = np.ascontiguousarray(iq[pos:pos + n, 1])
                self.lib.ref_sdrplay_packet(xi.ctypes.data, xq.ctypes.data, n)
                pos += n
                i += 1

    def counter(self, ch: int) -> int:
        return self.lib.ref_counter(ch)

    def dm(self, ch: int, n: int) -> np.ndarray:
        out = np.empty(n, dtype=np.float32)
        self.lib.ref_get_dm(ch, out.ctypes.data, n)
        return out

    def carry(self, ch: int) -> np.ndarray:
        out = np.empty(2, dtype=np.float32)
        self.lib.ref_get_carry(ch, out.ctypes.data)
        return out

    def state(self, ch: int) -> RefState:
        s = RefState()
        self.lib.ref_state(ch, C.byref(s))
        return s

    def msgs(self):
        self.lib.ref_flush()
        out = []
        buf = (Msg * 256)()
        while True:
            n = self.lib.ref_msgs(buf, 256)
            for i in range(n):
                m = Msg()
                C.memmove(C.byref(m), C.byref(buf[i]), C.sizeof(Msg))
                out.append(m)
            if n < 256:
                return out

    def close(self) -> None:
        self.lib.ref_close()


class OracleLib:
    def __init__(self):
        self.lib = C.CDLL(str(ORACLE_DIR / "libacars_oracle.so"))
        L = self.lib
        L.orc_build_h.argtypes = [C.c_void_p]
        L.orc_crc_step.argtypes = [C.c_uint16, C.c_uint8]
        L.orc_crc_step.restype = C.c_uint16
        L.orc_syndrome.argtypes = [C.c_int, C.c_int]
        L.orc_syndrome.restype = C.c_uint16
        L.orc_odd_parity.argtypes = [C.c_uint8]
        L.orc_choose_fc.argtypes = [C.c_void_p, C.c_int, C.c_int]
        L.orc_choose_fc.restype = C.c_uint
        L.orc_round_freq.argtypes = [C.c_double]
        L.orc_stored_fr.argtypes = [C.c_uint]
        L.orc_build_wf.argtypes = [C.c_int, C.c_uint, C.c_int, C.c_void_p]
        L.orc_channelize.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p]
        L.orc_air_choose_fc.argtypes = [C.c_uint, C.c_uint]
        L.orc_air_choose_fc.restype = C.c_uint
        L.orc_air_build_wf.argtypes = [C.c_int, C.c_int, C.c_uint, C.c_void_p]
        L.orc_channelize_real.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p]
        L.orc_channelize_fir.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p]
        L.orc_fast_plan.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_uint, C.c_void_p, C.c_void_p]
        L.orc_channelize_dft.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]
        L.orc_channelize_dft8.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]
        L.orc_fast_plan_air.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p]
        L.orc_channelize_rdft.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]
        L.orc_fast_plan_cs16.argtypes = [C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_uint, C.c_void_p, C.c_void_p]
        L.orc_channelize_dft8_cs16.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]
        L.orc_cs16_build_osc.argtypes = [C.c_int, C.c_uint, C.c_uint, C.c_int, C.c_void_p]
        L.orc_channelize_cs16.argtypes = [C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p]
        L.orc_channelize_cs16_table.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p]
        L.orc_chan_init.argtypes = [C.POINTER(OrcChan), C.c_int]
        L.orc_demod.argtypes = [C.POINTER(OrcChan), C.c_void_p, C.c_void_p, C.c_int, C.POINTER(OrcSink)]
        L.orc_block_fec.argtypes = [C.POINTER(Msg)]
        L.orc_stream_new.argtypes = [C.c_int, C.c_int, C.c_void_p]
        L.orc_stream_new.restype = C.c_void_p
        L.orc_stream_free.argtypes = [C.c_void_p]
        L.orc_stream_blocks.argtypes = [C.c_void_p, C.c_void_p, C.c_int]
        L.orc_stream_msgs.argtypes = [C.c_void_p, C.POINTER(Msg), C.c_int]
        L.orc_stream_chan.argtypes = [C.c_void_p, C.c_int]
        L.orc_stream_chan.restype = C.POINTER(OrcChan)
        L.orc_stream_dm.argtypes = [C.c_void_p, C.c_int]
        L.orc_stream_dm.restype = C.POINTER(C.c_float)
        L.orc_bench_streams.argtypes = [C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_int]
        L.orc_bench_streams.restype = C.c_double
        self._h = np.empty(133, dtype=np.float32)
        L.orc_build_h(self._h.ctypes.data)

    @property
    def h(self) -> np.ndarray:
        return self._h

    def plan(self, K: int, freqs_mhz):
        """(freqs_hz, stored Fr per channel, Fc) the way initRtl derives them (rtl.c:243-268)."""
        fd = np.array([self.lib.orc_round_freq(float(f)) for f in freqs_mhz], dtype=np.uint32)
        fc = self.lib.orc_choose_fc(fd.ctypes.data, len(fd), K)
        fr = [self.lib.orc_stored_fr(int(f)) for f in fd]
        return [int(f) for f in fd], fr, int(fc)

    def wf(self, K: int, freqs_mhz) -> np.ndarray:
        _, fr, fc = self.plan(K, freqs_mhz)
        out = np.empty((len(fr), 2 * K), dtype=np.float32)
        for i, f in enumerate(fr):
            self.lib.orc_build_wf(f, fc, K, out[i].ctypes.data)
        return out

    def channelize(self, iq: np.ndarray, K: int, wf: np.ndarray) -> np.ndarray:
        iq = np.ascontiguousarray(iq, dtype=np.uint8).reshape(-1)
        nout = iq.size // (2 * K)
        nch = wf.shape[0]
        dm = np.empty((nch, nout), dtype=np.float32)
        wf = np.ascontiguousarray(wf, dtype=np.float32)
        self.lib.orc_channelize(iq.ctypes.data, nout, K, nch, wf.ctypes.data, dm.ctypes.data)
        return dm

    def air_plan(self, rate: int, freqs_mhz):
        """(freqs_hz, Fc, K) the way initAirspy derives them (air.c:165-242, no-filter rates)."""
        fd = [self.lib.orc_round_freq(float(f)) for f in freqs_mhz]
        return fd, int(self.lib.orc_air_choose_fc(min(fd), max(fd))), rate // 12500

    def air_wf(self, rate: int, freqs_mhz) -> np.ndarray:
        fd, fc, K = self.air_plan(rate, freqs_mhz)
        out = np.empty((len(fd), 2 * K), dtype=np.float32)
        for i, f in enumerate(fd):
            self.lib.orc_air_build_wf(f, fc, rate, out[i].ctypes.data)
        return out

    def channelize_real(self, x: np.ndarray, K: int, wf: np.ndarray) -> np.ndarray:
        x = np.ascontiguousarray(x, dtype=np.float32).reshape(-1)
        nout = x.size // K
        dm = np.empty((wf.shape[0], nout), dtype=np.float32)
        wf = np.ascontiguousarray(wf, dtype=np.float32)
        self.lib.orc_channelize_real(x.ctypes.data, nout, K, wf.shape[0], wf.ctypes.data, dm.ctypes.data)
        return dm

    def channelize_fir(self, iq: np.ndarray, K: int, taps: int, wf: np.ndarray) -> np.ndarray:
        iq = np.ascontiguousarray(iq, dtype=np.uint8).reshape(-1)
        nout = iq.size // (2 * K)
        dm = np.empty((wf.shape[0], nout), dtype=np.float32)
        wf = np.ascontiguousarray(wf, dtype=np.float32)
        assert wf.shape[1] == 2 * taps
        self.lib.orc_channelize_fir(iq.ctypes.data, nout, K, taps, wf.shape[0], wf.ctypes.data, dm.ctypes.data)
        return dm

    def fast_plan(self, K: int, freqs_hz, fc: int):
        """(k per channel, twiddles (nch, K/4, 2) float32) of the fast channelizer's restatement, or None."""
        f = np.asarray(freqs_hz, dtype=np.uint32)
        k = np.zeros(len(f), dtype=np.int32)
        tw = np.zeros((len(f), K // 4, 2), dtype=np.float32)
        if self.lib.orc_fast_plan(f.ctypes.data, len(f), K, int(fc), k.ctypes.data, tw.ctypes.data) != 1:
            return None
        return k, tw

    def channelize_dft(self, iq: np.ndarray, K: int, k: np.ndarray, tw: np.ndarray, fold8: bool = False) -> np.ndarray:
        iq = np.ascontiguousarray(iq, dtype=np.uint8).reshape(-1)
        nout = iq.size // (2 * K)
        dm = np.empty((len(k), nout), dtype=np.float32)
        k = np.ascontiguousarray(k, dtype=np.int32)
        tw = np.ascontiguousarray(tw, dtype=np.float32)
        fn = self.lib.orc_channelize_dft8 if fold8 else self.lib.orc_channelize_dft
        fn(iq.ctypes.data, nout, K, len(k), k.ctypes.data, tw.ctypes.data, dm.ctypes.data)
        return dm

    def fast_plan_air(self, K: int, freqs_hz, fc: int):
        """(k per channel, twiddles (nch, K/4, 2) float32) of the fast real-input channelizer's restatement, or None."""
        f = np.asarray(freqs_hz, dtype=np.int32)
        k = np.zeros(len(f), dtype=np.int32)
        tw = np.zeros((len(f), K // 4, 2), dtype=np.float32)
        if self.lib.orc_fast_plan_air(f.ctypes.data, len(f), K, int(fc), k.ctypes.data, tw.ctypes.data) != 1:
            return None
        return k, tw

    def channelize_rdft(self, x: np.ndarray, K: int, k: np.ndarray, tw: np.ndarray) -> np.ndarray:
        x = np.ascontiguousarray(x, dtype=np.float32).reshape(-1)
        nout = x.size // K
        dm = np.empty((len(k), nout), dtype=np.float32)
        k = np.ascontiguousarray(k, dtype=np.int32)
        tw = np.ascontiguousarray(tw, dtype=np.float32)
        self.lib.orc_channelize_rdft(x.ctypes.data, nout, K, len(k), k.ctypes.data, tw.ctypes.data, dm.ctypes.data)
        return dm

    def fast_plan_cs16(self, variant: int, K: int, freqs_hz, fc: int):
        """(k per channel, twiddles (nch, K/4, 2) float32) of the fast CS16 channelizer's restatement, or None."""
        f = np.asarray(freqs_hz, dtype=np.uint32)
        k = np.zeros(len(f), dtype=np.int32)
        tw = np.zeros((len(f), K // 4, 2), dtype=np.float32)
        if self.lib.orc_fast_plan_cs16(variant, f.ctypes.data, len(f), K, int(fc), k.ctypes.data, tw.ctypes.data) != 1:
            return None
        return k, tw

    def channelize_dft8_cs16(self, iq: np.ndarray, K: int, k: np.ndarray, tw: np.ndarray) -> np.ndarray:
        iq = np.ascontiguousarray(iq, dtype=np.int16).reshape(-1)
        nout = iq.size // (2 * K)
        dm = np.empty((len(k), nout), dtype=np.float32)
        k = np.ascontiguousarray(k, dtype=np.int32)
        tw = np.ascontiguousarray(tw, dtype=np.float32)
        self.lib.orc_channelize_dft8_cs16(iq.ctypes.data, nout, K, len(k), k.ctypes.data, tw.ctypes.data, dm.ctypes.data)
        return dm

    def cs16_osc(self, variant: int, K: int, freqs_hz, fc: int) -> np.ndarray:
        out = np.empty((len(freqs_hz), 2 * K), dtype=np.float32)
        for i, f in enumerate(freqs_hz):
            self.lib.orc_cs16_build_osc(variant, int(f), int(fc), K, out[i].ctypes.data)
        return out

    def channelize_cs16(self, variant: int, iq: np.ndarray, K: int, osc: np.ndarray) -> np.ndarray:
        iq = np.ascontiguousarray(iq, dtype=np.int16).reshape(-1)
        nout = iq.size // (2 * K)
        dm = np.empty((osc.shape[0], nout), dtype=np.float32)
        osc = np.ascontiguousarray(osc, dtype=np.float32)
        self.lib.orc_channelize_cs16(variant, iq.ctypes.data, nout, K, osc.shape[0], osc.ctypes.data, dm.ctypes.data)
        return dm

    def channelize_cs16_table(self, iq: np.ndarray, K: int, taps: int, wf: np.ndarray) -> np.ndarray:
        """A CS16 context with the caller's table: |sum of the first `taps` (float)int16 samples x wf| per K-sample row."""
        iq = np.ascontiguousarray(iq, dtype=np.int16).reshape(-1)
        nout = iq.size // (2 * K)
        dm = np.empty((wf.shape[0], nout), dtype=np.float32)
        wf = np.ascontiguousarray(wf, dtype=np.float32)
        assert wf.shape[1] == 2 * taps
        self.lib.orc_channelize_cs16_table(iq.ctypes.data, nout, K, taps, wf.shape[0], wf.ctypes.data, dm.ctypes.data)
        return dm

    def new_chan(self, chn: int) -> OrcChan:
        c = OrcChan()
        self.lib.orc_chan_init(C.byref(c), chn)
        return c

    def demod(self, chan: OrcChan, dm: np.ndarray, sink: "Sink | None" = None) -> None:
        dm = np.ascontiguousarray(dm, dtype=np.float32)
        self.lib.orc_demod(C.byref(chan), self._h.ctypes.data, dm.ctypes.data, len(dm),
                           C.byref(sink.c) if sink else None)

    def fec(self, m: Msg):
        """Returns a fixed copy, or None when the reference would drop the block."""
        out = Msg()
        C.memmove(C.byref(out), C.byref(m), C.sizeof(Msg))
        return out if self.lib.orc_block_fec(C.byref(out)) else None


def mask_time(out: bytes) -> bytes:
    """The program's output with its wall-clock time stamps (text formats, JSON "timestamp") replaced by <time>."""
    out = re.sub(rb'"timestamp":[0-9.e+]+', b'"timestamp":<time>', out)
    return re.sub(rb"\d\d/\d\d/\d{4} \d\d:\d\d:\d\d\.\d{3}", b"<time>", out)


class RefPrograms:
    """The programs oracle/Makefile builds from the unmodified reference under oracle/_ref."""

    def outfmt(self, raw: bytes, *argv: str):
        """ref_outfmt: the reference's output.c / label.c / netout.c fed the records `raw`; one entry per record,
        what the reference printed (net == "-") or the one datagram it sent, None for nothing."""
        net = argv[1]
        r = subprocess.run([str(ORACLE_DIR / "_ref" / "ref_outfmt"), *argv], input=raw, capture_output=True, timeout=120)
        assert r.returncode == 0, r.stderr
        out = []
        for chunk in r.stdout.split(b"\x1e")[1:]:
            if net == "-":
                out.append(chunk or None)
            else:
                grams = chunk.split(b"\x1d")[1:]
                assert len(grams) <= 1
                out.append(grams[0] if grams else None)
        return out

    def acarsdec_rtl(self, iq: np.ndarray, *argv: str) -> bytes:
        """stdout of the whole reference program (acarsdec_ref) on the u8 IQ capture `iq` (file-replay librtlsdr),
        wall-clock time stamps masked (mask_time)."""
        import tempfile
        with tempfile.TemporaryDirectory() as d:
            cap = Path(d) / "cap.iq"
            iq.tofile(cap)
            r = subprocess.run([str(ORACLE_DIR / "_ref" / "acarsdec_ref"), *argv], env=dict(os.environ, ACARSDEC_STUB_IQ=str(cap)),
                               capture_output=True, timeout=120)
        assert r.returncode == 0, r.stderr
        return mask_time(r.stdout)

    def abi_layout(self) -> str:
        """channel_t / msgblk_t offsets and constants as the reference's acarsdec.h defines them (oracle/abi_layout.c)."""
        return subprocess.run([str(ORACLE_DIR / "_ref" / "abi_layout")], capture_output=True, text=True, check=True).stdout

    def close(self):
        pass


def _canon(v) -> bytes:
    """The bytes that identify a value the way the tests compare it: float arrays by shape and float32 bit
    pattern (common.bits_equal), floats exactly with -0.0 folded into 0.0 (== does not tell them apart)."""
    if isinstance(v, np.ndarray):
        if v.dtype.kind == "f":
            return repr(v.shape).encode() + np.ascontiguousarray(v, dtype=np.float32).tobytes()
        return v.dtype.str.encode() + repr(v.shape).encode() + np.ascontiguousarray(v).tobytes()
    if isinstance(v, (bytes, bytearray)):
        return b"b" + bytes(v)
    if isinstance(v, (float, np.floating)):
        return (float(v) + 0.0).hex().encode()
    if isinstance(v, (tuple, list)):
        return b"(" + b",".join(_canon(x) for x in v) + b")"
    if isinstance(v, Path):
        raise TypeError("a path is not an input of the reference: pass the data")
    return repr(v).encode()


def _digest(v) -> str:
    return hashlib.sha256(_canon(v)).hexdigest()[:8]


class Digest:
    """A recorded value too large to store: equal to any value with the same _canon bytes (32-bit digest)."""
    __hash__ = None

    def __init__(self, h: str):
        self.h = h

    def __eq__(self, other):
        return self.h == (other.h if isinstance(other, Digest) else _digest(other))

    def __repr__(self):
        return f"<reference value, digest {self.h}>"


class _State:
    def __init__(self, h: str):
        self._vec = Digest(h)

    def vec(self):
        return self._vec


def _encode(v):
    if v is None or isinstance(v, (bool, int, str)):
        return v
    if isinstance(v, np.integer):
        return int(v)
    if isinstance(v, float):
        return {"f": v.hex()}
    if isinstance(v, np.ndarray) and v.dtype.kind in "iu":
        return {"a": v.dtype.str, "v": v.tolist()}
    if isinstance(v, (RefState, _State)):
        return {"state": _digest(v.vec()) if isinstance(v, RefState) else v.vec().h}
    if isinstance(v, Msg):
        return {"msg": [v.chn, v.len, v.err, int(np.float32(v.lvl).view(np.uint32)), bytes(v.txt[:v.len]).hex(), bytes(v.crc).hex()]}
    if isinstance(v, (list, tuple)):
        return [_encode(x) for x in v]
    return {"d": _digest(v)}                             # float arrays, bytes


def _decode(e):
    if isinstance(e, list):
        return [_decode(x) for x in e]
    if not isinstance(e, dict):
        return e
    if "f" in e:
        return float.fromhex(e["f"])
    if "a" in e:
        return np.array(e["v"], dtype=e["a"])
    if "state" in e:
        return _State(e["state"])
    if "msg" in e:
        chn, ln, err, lvl, txt, crc = e["msg"]
        m = Msg()
        m.chn, m.len, m.err = chn, ln, err
        m.lvl = float(np.uint32(lvl).view(np.float32))
        m.txt[:ln] = bytes.fromhex(txt)
        m.crc[:] = bytes.fromhex(crc)
        return m
    return Digest(e["d"])


class Recorded:
    """A front-end of the unmodified reference (RefLib, RefAirLib, ...) as one test saw it.

    Replaying, it answers every call with what the reference returned when the recording was made, so the test
    compares against the reference on a machine that has no reference sources.  Recording (ACB_RECORD_REFERENCE=1,
    needs oracle/_ref), it forwards to the live library, so the test compares against the reference itself, and
    writes what it saw.  Calls that only feed the reference (INPUTS) return nothing; every call's name and arguments
    go into a running hash that each recorded answer carries, so a replay also checks that the test feeds the
    reference exactly what was recorded.  Numbers, integer tables and messages are stored as they are; float arrays,
    byte strings and channel states as a Digest."""
    INPUTS = {"open_rtl", "open_audio", "open", "block", "run", "audio", "push_block", "feed"}
    ATTRIBUTES = {"fc", "K", "nbch", "which"}

    def __init__(self, path: Path, live=None):
        self._path, self._live, self._h = path, live, hashlib.sha256()
        if live is None:
            if not path.exists():
                raise FileNotFoundError(f"{path.name}: no recording of the reference for this test "
                                        "(ACB_RECORD_REFERENCE=1 with oracle/_ref built writes it)")
            rec = json.loads(gzip.decompress(path.read_bytes()))
            self._calls, self._end = rec["calls"], rec["end"]
        else:
            self._calls, self._end = [], None
        self._next = 0

    def _answer(self, name: str, args, call):
        self._h.update(name.encode() + _canon(list(args)))
        where = self._h.hexdigest()[:8]
        if self._live is not None:
            v = call()
            if name in self.INPUTS:
                assert v is None, name
            else:
                self._calls.append([name, where, _encode(v)])
            return v
        if name in self.INPUTS:
            return None
        assert self._next < len(self._calls), f"{name}: more calls than recorded"
        rname, rwhere, v = self._calls[self._next]
        self._next += 1
        assert (rname, rwhere) == (name, where), f"call {self._next} ({name}) differs from the recording ({rname}) in name or inputs"
        return _decode(v)

    def __getattr__(self, name: str):
        if name.startswith("_"):
            raise AttributeError(name)
        if name in self.ATTRIBUTES:
            return self._answer(name, (), lambda: getattr(self._live, name))
        return lambda *args: self._answer(name, args, lambda: getattr(self._live, name)(*args))

    def finish(self) -> None:
        end = self._h.hexdigest()[:8]
        if self._live is not None:
            self._path.parent.mkdir(parents=True, exist_ok=True)
            data = json.dumps({"calls": self._calls, "end": end}, separators=(",", ":")).encode()
            self._path.write_bytes(gzip.compress(data, 9, mtime=0))
        else:
            assert self._next == len(self._calls) and end == self._end, "the test made fewer calls than recorded, or other inputs"


@contextlib.contextmanager
def recorded(request, open_live, close_live=lambda r: r.close()):
    """Recorded for the running test (tests/golden/reference/<module>.<test>.json.gz); open_live() builds the live
    front-end when recording."""
    name = re.sub(r"[^A-Za-z0-9_.-]+", "_", f"{request.node.module.__name__}.{request.node.name}").strip("_")
    path = RECORDINGS / (name + ".json.gz")
    live = None
    if RECORD:
        ensure_built()
        live = open_live()
    r = Recorded(path, live)
    failed = request.session.testsfailed
    try:
        yield r
        if request.session.testsfailed == failed:       # a failed test neither writes nor checks the rest of the recording
            r.finish()
    finally:
        if live is not None:
            close_live(live)


class Sink:
    """Collects pre-FEC blocks and (optionally) the raw bit stream of orc_demod."""

    def __init__(self, capbits: int = 0):
        self.c = OrcSink()
        self._bits = np.zeros(max(capbits, 1), dtype=np.uint8)
        if capbits:
            self.c.bits = self._bits.ctypes.data_as(C.POINTER(C.c_uint8))
            self.c.capbits = capbits

    def msgs(self):
        out = []
        for i in range(self.c.nmsg):
            m = Msg()
            C.memmove(C.byref(m), C.byref(self.c.msgs[i]), C.sizeof(Msg))
            out.append(m)
        return out

    def bits(self) -> np.ndarray:
        return self._bits[: self.c.nbits].copy()


class OracleStream:
    """Whole path for one stream through the restatement (rtl.c:314-361 order)."""

    def __init__(self, lib: OracleLib, K: int, wf: np.ndarray):
        self.lib, self.K, self.nch = lib, K, wf.shape[0]
        wf = np.ascontiguousarray(wf, dtype=np.float32)
        self.p = lib.lib.orc_stream_new(K, self.nch, wf.ctypes.data)

    def blocks(self, iq: np.ndarray) -> int:
        iq = np.ascontiguousarray(iq, dtype=np.uint8)
        nblk = iq.size // (2048 * self.K)
        return self.lib.lib.orc_stream_blocks(self.p, iq.ctypes.data, nblk)

    def msgs(self):
        out = []
        buf = (Msg * 256)()
        while True:
            n = self.lib.lib.orc_stream_msgs(self.p, buf, 256)
            for i in range(n):
                m = Msg()
                C.memmove(C.byref(m), C.byref(buf[i]), C.sizeof(Msg))
                out.append(m)
            if n < 256:
                return out

    def chan(self, ch: int) -> OrcChan:
        return self.lib.lib.orc_stream_chan(self.p, ch).contents

    def dm(self, ch: int) -> np.ndarray:
        return np.ctypeslib.as_array(self.lib.lib.orc_stream_dm(self.p, ch), shape=(1024,)).copy()

    def close(self):
        if self.p:
            self.lib.lib.orc_stream_free(self.p)
            self.p = None

    def __del__(self):
        self.close()
