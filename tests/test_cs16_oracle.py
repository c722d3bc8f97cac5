"""CS16 front-ends (soapy.c interleaved int16 with /32768.0 in double, sdrplay.c planar int16 with
envelope/4): restatement vs the unmodified references compiled in place, and the product's folded
tables (powers of two moved into the table) vs the literal arithmetic.  CPU only."""
import numpy as np
import pytest

import refs
from acarsdec_b200 import api, synth
from common import bits_equal, msg_tuple

FREQS = (131.525, 131.725, 131.825, 131.450)


@pytest.fixture(params=["soapy", "sdrplay"])
def cs16ref(request):
    with refs.recorded(request, lambda: refs.RefCs16Lib(request.param)) as r:
        yield r


def test_cs16_plan_tables_carry_and_messages(oracle, cs16ref):
    variant = 0 if cs16ref.which == "soapy" else 1
    K = 160
    cs16ref.open(FREQS, K)
    fd, _, fc = oracle.plan(K, FREQS)
    assert cs16ref.fc == fc
    osc = oracle.cs16_osc(variant, K, fd, fc)
    for c in range(len(FREQS)):
        assert bits_equal(osc[c], cs16ref.osc(c)), c
    plan = synth.StreamPlan(K=K, freqs_hz=tuple(fd), fc_hz=fc, seed=12, noise_sigma=1.5)
    rng = np.random.default_rng(12)
    for ch in range(4):
        plan.bursts.append(synth.Burst(chan=ch, t0=0.01 + 0.04 * ch, frame=synth.frame_bytes(synth.random_text(rng, 15 + 8 * ch)),
                                       amp=15.0 + 4 * ch, phase=0.7 * ch))
    nblock = 1024 if variant == 0 else 512                   # demodMSK chunk: soapy.c:246 / sdrplay.c:228
    total = (int(0.5 * plan.rate) // (K * nblock)) * K * nblock + 37 * K + 11      # not a whole number of rows
    iq = synth.render_cs16(plan, 0, total)
    sizes = [4000, 163840, 7, 159, 161, 100000] if variant == 0 else [336, 252, 1000, 7, 159, 161]
    cs16ref.feed(iq, sizes)
    nout = total // K
    dm = oracle.channelize_cs16(variant, iq[: nout * K], K, osc)
    # the reference demodulates in chunks of nblock outputs; what is left sits in dm_buffer / D
    done = (nout // nblock) * nblock
    chans = [oracle.new_chan(c) for c in range(4)]
    sink = refs.Sink()
    got = []
    for b in range(0, done, nblock):
        for c in range(4):
            oracle.demod(chans[c], dm[c, b:b + nblock], sink)
        for m in sink.msgs():
            f = oracle.fec(m)
            if f is not None:
                got.append(msg_tuple(f))
        sink.c.nmsg = 0
    for c in range(4):
        assert cs16ref.counter(c) == nout - done
        assert bits_equal(cs16ref.dm(c, nout - done), dm[c, done:]), c
        assert cs16ref.state(c).vec() == chans[c].vec(), c
    assert [msg_tuple(m) for m in cs16ref.msgs()] == got and len(got) == 4
    # the product's tables fold soapy's /32768.0 and sdrplay's envelope/4 into the oscillator
    wf = api.build_wf_cs16(variant, K, fd, fc)
    scale = np.float32(1 / 32768) if variant == 0 else np.float32(0.25)
    assert bits_equal(wf, osc * scale)


def test_cs16_folded_tables_equal_literal_arithmetic(oracle):
    """fl32(fl64(D + p/32768)) == fl32(D + p') with p' computed from the pre-scaled table, and
    hypot(D)/4 == hypot(D') for the quarter-scaled table: same envelope bits."""
    K = 160
    fd, _, fc = oracle.plan(K, FREQS)
    iq = np.random.default_rng(5).integers(-32768, 32768, size=(64 * K, 2), dtype=np.int16)
    iq[:K] = 32767
    iq[K:2 * K] = -32768
    for variant in (0, 1):
        osc = oracle.cs16_osc(variant, K, fd, fc)
        lit = oracle.channelize_cs16(variant, iq, K, osc)
        scale = np.float32(1 / 32768) if variant == 0 else np.float32(0.25)
        plain = oracle.channelize_cs16(2, iq, K, osc * scale)      # plain D += v*w ; |D|
        assert bits_equal(lit, plain), variant


@pytest.mark.parametrize("K", [160, 36])
def test_cs16_caller_table_restatement(oracle, K):
    """orc_channelize_cs16_table (a CS16 context with acb_set_wf's table) is the literal arithmetic of both front-ends
    when handed their folded planner tables, and at taps < K the same sum over the first `taps` samples: equal to a K-tap
    table zero-padded past `taps` (x*0 = +-0 leaves D and |D| alone) and within rounding of a float64 sum."""
    fm = FREQS if K == 160 else (131.525, 131.550, 131.600)
    fd, _, fc = oracle.plan(K, fm)
    iq = np.random.default_rng(K).integers(-32768, 32768, size=(48 * K, 2), dtype=np.int16)
    iq[:K] = 32767
    iq[K:2 * K] = -32768
    for variant in (0, 1):
        osc = oracle.cs16_osc(variant, K, fd, fc)
        folded = api.build_wf_cs16(variant, K, fd, fc)
        assert bits_equal(oracle.channelize_cs16_table(iq, K, K, folded), oracle.channelize_cs16(variant, iq, K, osc)), variant
    rng = np.random.default_rng(K + 1)
    x = iq.astype(np.float64).reshape(-1, K, 2)
    x = x[..., 0] + 1j * x[..., 1]
    for taps in (1, 5, K - 3):
        wf = (rng.standard_normal((len(fm), 2 * taps)) * 1e-4).astype(np.float32)
        got = oracle.channelize_cs16_table(iq, K, taps, wf)
        padded = np.zeros((len(fm), 2 * K), dtype=np.float32)
        padded[:, :2 * taps] = wf
        assert bits_equal(got, oracle.channelize_cs16(2, iq, K, padded)), taps
        w = wf[:, 0::2].astype(np.float64) + 1j * wf[:, 1::2]
        d64 = x[:, :taps] @ w.T
        mass = np.abs(x[:, :taps]) @ np.abs(w).T
        assert (np.abs(got.T - np.abs(d64)) <= 2 * (taps + 4) * 2.0 ** -24 * mass).all(), taps
        assert got.any()
