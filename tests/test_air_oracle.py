"""The Airspy front-end (air.c: float32 real input at IF = rate/4, partial sums carried across
transfers): restatement vs the unmodified reference compiled in place.  CPU only."""
import numpy as np
import pytest

import refs
from acarsdec_b200 import synth
from common import bits_equal, msg_tuple


@pytest.fixture()
def airref(request):
    with refs.recorded(request, refs.RefAirLib) as r:
        yield r


@pytest.mark.parametrize("rate,freqs", [
    (2500000, (131.525, 131.725, 131.825)),
    (3000000, (131.125, 131.450, 131.475, 131.525, 131.550, 131.725, 131.825, 131.850)),
    (6000000, (129.125, 130.025, 131.550, 131.725)),
    (10000000, (131.525, 136.900)),
])
def test_air_plan_and_table(oracle, airref, rate, freqs):
    airref.open(rate, freqs)
    fd, fc, K = oracle.air_plan(rate, freqs)
    assert (fc, K) == (airref.fc, airref.K)
    wf = oracle.air_wf(rate, freqs)
    for i in range(len(freqs)):
        assert bits_equal(wf[i], airref.wf(i))


def test_air_streaming_carry_and_messages(oracle, airref):
    """Transfers of awkward sizes (the reference carries D and the tap index, air.c:299-338) vs the
    restatement walking the concatenated stream row by row; then frames through demod + FEC."""
    rate, fm = 2500000, (131.525, 131.725, 131.825, 131.450)
    airref.open(rate, fm)
    fd, fc, K = oracle.air_plan(rate, fm)
    wf = oracle.air_wf(rate, fm)
    plan = synth.StreamPlan(K=K, freqs_hz=tuple(fd), fc_hz=fc, seed=9, noise_sigma=1.0)
    rng = np.random.default_rng(4)
    for ch in range(4):
        plan.bursts.append(synth.Burst(chan=ch, t0=0.01 + 0.05 * ch, frame=synth.frame_bytes(synth.random_text(rng, 20 + 10 * ch)),
                                       amp=15.0 + 3 * ch, phase=0.4 * ch))
    total = int(0.62 * rate)
    x = synth.render_real(plan, 0, total)
    chans = [oracle.new_chan(c) for c in range(4)]
    sink = refs.Sink()
    pos, nout_done, got = 0, 0, []
    while pos < total:
        n = min(total - pos, int(rng.integers(K, 60000)))      # >= K so that each transfer emits >= 1 output
        m = airref.transfer(x[pos:pos + n])
        pos += n
        # the restatement on the same prefix of the stream
        want = oracle.channelize_real(x[nout_done * K:(nout_done + m) * K], K, wf)
        for c in range(4):
            assert bits_equal(airref.dm(c, m), want[c]), (pos, c)
            oracle.demod(chans[c], want[c], sink)
            assert airref.state(c).vec() == chans[c].vec(), (pos, c)
        for msg in sink.msgs():
            f = oracle.fec(msg)
            if f is not None:
                got.append(msg_tuple(f))
        sink.c.nmsg = 0
        nout_done += m
    assert [msg_tuple(m) for m in airref.msgs()] == got
    assert len(got) == 4
