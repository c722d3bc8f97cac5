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


def bits_equal(a: np.ndarray, b: np.ndarray) -> bool:
    from refs import Digest
    if isinstance(b, Digest):
        a, b = b, a
    if isinstance(a, Digest):
        return a == b                                    # a recorded reference array: same shape and float32 bits
    a = np.ascontiguousarray(a, dtype=np.float32)
    b = np.ascontiguousarray(b, dtype=np.float32)
    return a.shape == b.shape and np.array_equal(a.view(np.uint32), b.view(np.uint32))
