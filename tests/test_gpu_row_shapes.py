"""The exact channelizers at the row shapes that pick the kernel and cut a row into chunks: K and taps for the
float32 real (air.c) and CS16 (soapy.c / sdrplay.c) streaming front-ends and the u8 path.

k_channelize / k_channelize_real4 walk a row in chunks of 5 sixteen-byte units (20 four-byte taps, 40 u8 taps) with a
shorter last chunk; rows of a K that breaks 16-byte alignment, and the < 1024 rows left over by a streaming submit, go
through k_channelize_generic; taps < K (FIR) pads the table to whole units with zero weights.  Every envelope is held
to two references:
  Bar 1  the oracle's restatement, bit for bit (a zero-padded K-tap table is exactly the taps-tap sum: x*0 = +-0, and
         adding +-0 changes neither D nor |D|);
  Bar 2  a float64 sum of the same products on the same float32 values, within 2*(taps+4)*2^-24 * sum|w||x|, and the
         envelope not identically zero: a mistake shared by the test's table or input and the oracle shows here."""
import json
import os
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

import refs
import row_shapes_worker as rw
from acarsdec_b200 import api, synth
from common import bits_equal, msg_tuple, ragged_sizes, stream_envelope

pytestmark = pytest.mark.gpu
FLAG_REAL, FLAG_CS16 = 2, 4
U8_BIAS = np.float32(127.37)
NROWS = 2 * 1024 + 517                  # rows per stream: two pipeline blocks and a generic tail, cut by ragged submits
FM17 = tuple(130.000 + 0.025 * i for i in range(17))         # three channel groups of 8, the last holding one channel


def assert_bits(got: np.ndarray, want: np.ndarray, what) -> None:
    """got, want: (nout, nch) float32; on a difference, name the first row and channel."""
    assert got.shape == want.shape, (what, got.shape, want.shape)
    got, want = (np.ascontiguousarray(a, dtype=np.float32) for a in (got, want))
    bad = np.argwhere(got.view(np.uint32) != want.view(np.uint32))
    assert len(bad) == 0, f"{what}: {len(bad)} samples differ, first at (row, channel) {tuple(bad[0])}: {got[tuple(bad[0])]!r} vs {want[tuple(bad[0])]!r}"


def bar2(dm: np.ndarray, rows: np.ndarray, wf: np.ndarray, taps: int, what) -> float:
    """dm (nout, nch) envelope; rows (nout, >= taps) float64 or complex128 input values; wf (nch, 2*taps) float32 table.
    Checks |dm - |D64|| against the rounding bound of a taps-term float32 sum and returns the largest ratio
    |dm - |D64|| / sum|w||x| (printed for the record)."""
    w = wf[:, 0::2].astype(np.float64) + 1j * wf[:, 1::2].astype(np.float64)
    x = rows[:, :taps]
    d64 = x @ w.T
    mass = np.abs(x) @ np.abs(w).T
    err = np.abs(dm.astype(np.float64) - np.abs(d64))
    bound = 2 * (taps + 4) * 2.0 ** -24 * mass
    worst = np.unravel_index(np.argmax(err - bound), err.shape)
    assert (err <= bound).all(), f"{what}: |dm - |D64|| = {err[worst]:.3e} > {bound[worst]:.3e} at (row, channel) {worst}"
    assert (dm.max(axis=0) > 0).all(), f"{what}: a channel's envelope is identically zero"
    ratio = float((err / np.where(mass > 0, mass, 1.0)).max())
    print(f"bar2 {what}: max |dm - |D64|| / sum|w||x| = {ratio:.3e}")
    return ratio


def padded(wf: np.ndarray, K: int) -> np.ndarray:
    """a taps-tap table (nch, 2*taps) as a K-tap one with zero weights past `taps`"""
    out = np.zeros((wf.shape[0], 2 * K), dtype=np.float32)
    out[:, :wf.shape[1]] = wf
    return out


def max_blocks_for(nrows: int) -> int:
    return nrows // 1024 + 2


# ------------------------------------------------------------------ float32 real input (air.c)

@pytest.mark.parametrize("K,taps,nch,table", [
    (36, 36, 3, "random"),            # k_channelize_real4: 9 units per row = chunks of 5 + 4
    (204, 204, 17, "air"),            # 51 units = 10 chunks + a 1-unit tail; three channel groups
    (1004, 1004, 17, "air"),          # 251 units = 50 chunks + 1
    (2048, 2048, 17, "air"),          # ACB_MAXK: 512 units = 102 chunks + 2
    (2048, 1021, 9, "random"),        # FIR: taps padded to 1024 = 51 chunks + 1
    (202, 202, 9, "random"),          # K % 4 != 0: k_channelize_generic for every row
    (6, 6, 3, "random"),
    (200, 1, 5, "random"),            # FIR padding: taps_pad 4, 4, 24, 200
    (200, 3, 5, "random"),
    (200, 21, 5, "random"),
    (200, 199, 5, "random"),
])
def test_real_row_shapes(native, oracle, K, taps, nch, table):
    rng = np.random.default_rng([K, taps, nch, 1])
    x = (rng.standard_normal((1, NROWS * K + K // 2 + 1)) * 0.5).astype(np.float32)
    x[0, :K] = 1.0                                                    # a row of one value: every tap weight in the sum
    max_blocks = max_blocks_for(NROWS)
    with api.Context(K, 1, nch, max_blocks, flags=FLAG_REAL, taps=0 if taps == K else taps) as ctx:
        if table == "air":
            rate, fm = K * 12500, FM17[:nch]
            fd, fc, _ = oracle.air_plan(rate, fm)
            wf = oracle.air_wf(rate, fm)
            assert bits_equal(api.build_wf_air(rate, fm), wf)
            assert ctx.set_plan_air(0, fd) == fc
        else:
            wf = (rng.standard_normal((nch, 2 * taps)) / np.sqrt(taps)).astype(np.float32)
            ctx.set_wf(0, wf)
        env, _ = stream_envelope(ctx, ctx.submit_real, x, ragged_sizes(K, x.shape[1], (max_blocks * 1024 - 1) * K, seed=K + taps))
    nout = x.shape[1] // K
    want = oracle.channelize_real(x[0, :nout * K], K, padded(wf, K)).T
    assert_bits(env[0], want, f"real K={K} taps={taps}")
    bar2(env[0], x[0, :nout * K].reshape(nout, K).astype(np.float64), wf, taps, f"real K={K} taps={taps}")


def test_real_two_row_kernel(native, oracle):
    """ACB_REAL_ROWS=2 selects k_channelize<IN_F32REAL> (two rows per thread) in place of k_channelize_real4; it is read
    once per process, so a worker process runs the cases with it.  Its envelopes must be bit-identical to the default
    kernel's in this process and to the oracle, and the profiler must show which kernel ran."""
    env = dict(os.environ, ACB_REAL_ROWS="2")
    r = subprocess.run([sys.executable, str(Path(rw.__file__))], env=env, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-4000:]
    rep = json.loads(r.stdout.strip().splitlines()[-1])
    assert any("k_channelize<1>" in k for k in rep["kernels"]), rep["kernels"]
    assert not any("k_channelize_real4" in k for k in rep["kernels"]), rep["kernels"]
    for name in rw.CASES:
        K, taps, x, wf, _, _ = rw.real_case(name)
        nout = x.shape[1] // K
        want = oracle.channelize_real(x[0, :nout * K], K, padded(wf, K)).T
        got = rw.run_real(name)
        assert_bits(got, want, f"default kernel, {name}")
        assert rep["digests"][name] == rw.digest(want), f"ACB_REAL_ROWS=2 differs from the oracle: {name}"


def test_real_k204_frames(native, oracle):
    """End to end at a non-Airspy K: a synthetic capture at K = 204 (2.55 MS/s) with 17 channels, ragged submits;
    envelope bit for bit, frames and final states against the oracle's demod of the oracle's envelope."""
    K, secs = 204, 0.4
    rate = K * 12500
    fd, fc, _ = oracle.air_plan(rate, FM17)
    plan = synth.StreamPlan(K=K, freqs_hz=tuple(fd), fc_hz=fc, seed=204, noise_sigma=1.0)
    rng = np.random.default_rng(204)
    for ch in range(len(FM17)):
        t = 0.005 + 0.011 * ch
        while True:
            fr = synth.frame_bytes(synth.random_text(rng, int(rng.integers(13, 30))))
            dur = len(fr) * 8 / 2400
            if t + dur + 0.01 > secs:
                break
            plan.bursts.append(synth.Burst(chan=ch, t0=t, frame=fr, amp=float(rng.uniform(10, 25)), phase=float(rng.uniform(0, 6))))
            t += dur + 0.04
    total = int(secs * rate)
    x = synth.render_real(plan, 0, total)[None, :]
    wf = oracle.air_wf(rate, FM17)
    nout = total // K
    max_blocks = max_blocks_for(nout)
    with api.Context(K, 1, len(FM17), max_blocks, flags=FLAG_REAL) as ctx:
        assert ctx.set_plan_air(0, fd) == fc
        env, msgs = stream_envelope(ctx, ctx.submit_real, x, ragged_sizes(K, total, (max_blocks * 1024 - 1) * K, seed=5))
        states = [ctx.get_state(0, c).vec() for c in range(len(FM17))]
    want_dm = oracle.channelize_real(x[0, :nout * K], K, wf)
    assert_bits(env[0], want_dm.T, "real K=204, synthetic capture")
    sink, want = refs.Sink(), []
    for c in range(len(FM17)):
        ch = oracle.new_chan(c)
        oracle.demod(ch, want_dm[c], sink)
        assert states[c] == ch.vec(), c
    for m in sink.msgs():
        f = oracle.fec(m)
        if f is not None:
            want.append(msg_tuple(f))
    frames = [msg_tuple(m) for m in msgs]
    # emission groups are per submit: compare each channel's frames in time order
    for c in range(len(FM17)):
        assert [f for f in frames if f[0] == c] == [f for f in want if f[0] == c], c
    assert sorted(frames) == sorted(want) and len({f[0] for f in want}) >= 12


# ------------------------------------------------------------------ CS16 IQ (soapy.c, sdrplay.c)

def _cs16_submit(ctx, planar):
    if planar:
        return lambda part: ctx.submit_cs16_planar(np.ascontiguousarray(part[..., 0]), np.ascontiguousarray(part[..., 1]))
    return ctx.submit_cs16


def _cs16_rows(iq: np.ndarray, K: int) -> np.ndarray:
    nout = len(iq) // K
    v = iq[:nout * K].astype(np.float64).reshape(nout, K, 2)
    return v[..., 0] + 1j * v[..., 1]


@pytest.mark.parametrize("variant,K,fm,planar", [
    (0, 36, (131.525, 131.550, 131.600), False),          # 9 units per row = chunks of 5 + 4
    (1, 36, (131.525, 131.550, 131.600), True),
    (0, 1004, FM17, False),                               # 251 units = 50 chunks + 1; three channel groups
    (1, 1004, FM17, True),
    (0, 2048, (129.000, 130.500, 131.525, 133.000, 136.900), True),     # ACB_MAXK: 102 chunks + 2
    (1, 2048, (129.000, 130.500, 131.525, 133.000, 136.900), False),
    (0, 162, (131.525, 131.725, 131.825, 131.450, 131.550), False),     # K % 4 != 0: generic kernel for every row
    (1, 162, (131.525, 131.725, 131.825, 131.450, 131.550), True),
])
def test_cs16_row_shapes(native, oracle, variant, K, fm, planar):
    rng = np.random.default_rng([K, variant, 2])
    iq = rng.integers(-32768, 32768, size=(1, NROWS * K + K // 2 + 1, 2), dtype=np.int16)
    iq[0, :K] = 32767                                                  # full-scale rows
    iq[0, K:2 * K] = -32768
    fd, _, fc = oracle.plan(K, fm)
    max_blocks = max_blocks_for(NROWS)
    with api.Context(K, 1, len(fm), max_blocks, flags=FLAG_CS16) as ctx:
        assert ctx.set_plan_cs16(0, fd, variant) == fc
        env, _ = stream_envelope(ctx, _cs16_submit(ctx, planar), iq, ragged_sizes(K, iq.shape[1], (max_blocks * 1024 - 1) * K, seed=K))
    nout = iq.shape[1] // K
    want = oracle.channelize_cs16(variant, iq[0, :nout * K], K, oracle.cs16_osc(variant, K, fd, fc)).T
    assert_bits(env[0], want, f"CS16 variant {variant} K={K}")
    # the folded table (the variant's power-of-two scale inside) gives the envelope directly
    bar2(env[0], _cs16_rows(iq[0], K), api.build_wf_cs16(variant, K, fd, fc), K, f"CS16 variant {variant} K={K}")


@pytest.mark.parametrize("taps,planar", [(5, False), (5, True), (77, False), (77, True)])
def test_cs16_caller_table_fir(native, oracle, taps, planar):
    """taps < K on a CS16 context: the caller's table (acb_set_wf), padded to 8 and 80 taps, nine channels (two groups)."""
    K, nch = 192, 9
    rng = np.random.default_rng([taps, int(planar), 3])
    iq = rng.integers(-32768, 32768, size=(1, NROWS * K + 100, 2), dtype=np.int16)
    wf = (rng.standard_normal((nch, 2 * taps)) / (32768 * np.sqrt(taps))).astype(np.float32)
    max_blocks = max_blocks_for(NROWS)
    with api.Context(K, 1, nch, max_blocks, flags=FLAG_CS16, taps=taps) as ctx:
        ctx.set_wf(0, wf)
        with pytest.raises(api.AcbError):
            ctx.set_plan_cs16(0, [131525000] * nch, 0)                 # the planners only build K-tap tables
        env, _ = stream_envelope(ctx, _cs16_submit(ctx, planar), iq, ragged_sizes(K, iq.shape[1], (max_blocks * 1024 - 1) * K, seed=taps))
    nout = iq.shape[1] // K
    want = oracle.channelize_cs16_table(iq[0, :nout * K], K, taps, wf).T
    assert_bits(env[0], want, f"CS16 K={K} taps={taps}")
    bar2(env[0], _cs16_rows(iq[0], K), wf, taps, f"CS16 K={K} taps={taps}")


# ------------------------------------------------------------------ u8 IQ (rtl.c)

@pytest.mark.parametrize("K,fm,nblk", [
    (24, (131.525, 131.550, 131.600), 3),                 # 3 units per row: one short chunk
    (2048, FM17, 2),                                      # ACB_MAXK: 256 units = 51 chunks + 1
])
def test_u8_row_shapes(native, oracle, K, fm, nblk):
    rng = np.random.default_rng([K, 4])
    iq = rng.integers(0, 256, size=(1, nblk * 2048 * K), dtype=np.uint8)
    iq[0, :2 * K] = 0
    iq[0, 2 * K:4 * K] = 255
    wf = oracle.wf(K, fm)
    fd, _, fc = api.plan(K, fm)
    with api.Context(K, 1, len(fm), nblk) as ctx:
        assert ctx.set_plan(0, fd) == fc
        got = []
        for b0, n in ((0, 1), (1, nblk - 1)):                          # two submits
            ctx.submit_host(np.ascontiguousarray(iq[:, b0 * 2048 * K:(b0 + n) * 2048 * K]), n)
            ctx.sync()
            got.append(ctx.read_dm(n * 1024)[0])
    env = np.concatenate(got)
    assert_bits(env, oracle.channelize(iq[0], K, wf).T, f"u8 K={K}")
    v = (iq[0].astype(np.float32) - U8_BIAS).astype(np.float64).reshape(-1, K, 2)
    bar2(env, v[..., 0] + 1j * v[..., 1], wf, K, f"u8 K={K}")
