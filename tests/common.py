"""Shared helpers for the tests."""
from __future__ import annotations

import json
from pathlib import Path

import numpy as np

GOLDEN = Path(__file__).resolve().parent / "golden"


def load_testwav():
    """(float32 samples [n,4] scaled like sf_read_float, expected dict)"""
    pcm = np.load(GOLDEN / "testwav_pcm16.npz")["pcm"]
    x = pcm.astype(np.float32) / np.float32(32768.0)
    exp = json.load(open(GOLDEN / "testwav_expected.json"))
    return x, exp


def load_synth_k16():
    iq = np.load(GOLDEN / "synth_k16.npz")["iq"]
    exp = json.load(open(GOLDEN / "synth_k16.json"))
    return iq, exp


def msg_tuple_from_json(j):
    return (j["chn"], j["len"], j["err"], bytes.fromhex(j["txt"]), bytes.fromhex(j["crc"]), j["lvl_bits"])


def msg_tuple(m):
    """(chn, len, err, txt, crc, lvl bit pattern) from any of the ctypes Msg flavours."""
    return (m.chn, m.len, m.err, bytes(m.txt[:m.len]), bytes(m.crc), int(np.float32(m.lvl).view(np.uint32)))


def state_tuple_from_json(j):
    return (float.fromhex(j["MskPhi"]), float.fromhex(j["MskDf"]), float.fromhex(j["MskLvlSum"]),
            float.fromhex(j["MskClk"]), j["MskBitCount"], j["MskS"], j["idx"], j["nbits"], j["state"], j["outbits"],
            tuple(float.fromhex(x) for x in j["inb"]))


def emission_model(oracle, dms, cuts, positions: bool = False):
    """The reference's loop as a plain model: walk the emission groups; in each, for each stream and each channel in
    turn, demodMSK on that group's slice of the envelope; then the block FEC.  dms: per stream, a (nch, nout) float32
    envelope; cuts: the first sample of every group (0 is always one).  Returns the surviving messages in emission
    order as (stream, msg_tuple, group start, group end, completion sample) and the final channel states
    [stream][channel].  The completion sample (0-based: the envelope sample whose processing finished the frame) is
    found by feeding shorter prefixes of the slice to copies of the channel state when `positions` is set, else None."""
    import ctypes as C
    import refs

    nout = dms[0].shape[1]
    bounds = sorted({int(c) for c in cuts if 0 <= c < nout} | {0}) + [nout]
    chans = [[oracle.new_chan(c) for c in range(d.shape[0])] for d in dms]

    def copy(ch):
        out = refs.OrcChan()
        C.memmove(C.byref(out), C.byref(ch), C.sizeof(out))
        return out

    def count(before, x):
        sink = refs.Sink()
        oracle.demod(copy(before), x, sink)
        return sink.c.nmsg

    out = []
    for lo, hi in zip(bounds[:-1], bounds[1:]):
        for s, d in enumerate(dms):
            for c in range(d.shape[0]):
                x = np.ascontiguousarray(d[c, lo:hi])
                before = copy(chans[s][c]) if positions else None
                sink = refs.Sink()
                oracle.demod(chans[s][c], x, sink)
                for i, m in enumerate(sink.msgs()):
                    p = None
                    if positions:                        # shortest prefix that yields message i: it completes on its last sample
                        a, b = 1, len(x)
                        while a < b:
                            mid = (a + b) // 2
                            a, b = (mid + 1, b) if count(before, x[:mid]) <= i else (a, mid)
                        p = lo + a - 1
                    f = oracle.fec(m)
                    if f is not None:
                        out.append((s, msg_tuple(f), lo, hi, p))
    return out, chans


def assert_emission_order(got, model):
    """Drained messages (api.Msg, in queue order) against emission_model(): same stream and message at every place,
    its position inside the group the model put it in, and equal to the model's completion sample where known."""
    assert [(m.stream, msg_tuple(m)) for m in got] == [(s, t) for s, t, *_ in model]
    for m, (s, t, lo, hi, p) in zip(got, model):
        assert lo <= m.pos < hi, (s, t[0], m.pos, lo, hi)
        if p is not None:
            assert m.pos == p, (s, t[0], m.pos, p)


def ragged_sizes(K: int, total: int, max_submit: int, seed: int):
    """Submit lengths in samples that cover `total`: below one row, a few rows, one block and 37 rows more (a pipeline
    block and generic tail rows in one submit), an odd count, a couple of rows and one, then random lengths."""
    rng = np.random.default_rng(seed)
    sizes, pos = [], 0
    for n in [K // 3 + 1, 5 * K + 7, 1061 * K + 13, 3, 2 * K + 1]:
        sizes.append(min(n, total - pos, max_submit))
        pos += sizes[-1]
    while pos < total:
        sizes.append(min(int(rng.integers(1, 1500 * K)), total - pos, max_submit))
        pos += sizes[-1]
    return [n for n in sizes if n]


def stream_envelope(ctx, submit, data: np.ndarray, sizes):
    """Feed data (nstreams, nsamples[, 2]) to a streaming context through `submit` in the given lengths and read each
    submit's envelope right after it: (concatenated envelope (nstreams, nout, nch), drained messages)."""
    pieces, msgs, pos = [], [], 0
    for n in sizes:
        m = submit(np.ascontiguousarray(data[:, pos:pos + n]))
        pos += n
        ctx.sync()
        msgs += ctx.drain()
        if m:
            pieces.append(ctx.read_dm(m))
    assert pos == data.shape[1]
    return np.concatenate(pieces, axis=1), msgs


def bits_equal(a: np.ndarray, b: np.ndarray) -> bool:
    from refs import Digest
    if isinstance(b, Digest):
        a, b = b, a
    if isinstance(a, Digest):
        return a == b                                    # a recorded reference array: same shape and float32 bits
    a = np.ascontiguousarray(a, dtype=np.float32)
    b = np.ascontiguousarray(b, dtype=np.float32)
    return a.shape == b.shape and np.array_equal(a.view(np.uint32), b.view(np.uint32))
