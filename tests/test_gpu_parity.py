"""GPU parity tests: the CUDA path, called through the C ABI (ctypes), against the CPU oracle on
identical inputs.  Bar (BASELINE.json north_star): envelope samples and decoded frames bit-exact;
demodulator float state within 1e-5 relative (device sincos is not glibc's — see DESIGN.md) and in
practice bit-exact, which is asserted where the run is short enough for that to be certain."""
import hashlib

import numpy as np
import pytest

import refs
from acarsdec_b200 import api, synth
from common import (bits_equal, load_synth_k16, load_testwav, msg_tuple, msg_tuple_from_json,
                    state_tuple_from_json)

pytestmark = pytest.mark.gpu

REL_TOL = 1e-5      # north_star: "demod float intermediates within 1e-5 rel"


def states_close(a, b, tol=REL_TOL):
    """a, b: vec() tuples.  Integers exact, floats within tol (relative, abs floor 1e-9)."""
    for i, (x, y) in enumerate(zip(a, b)):
        if isinstance(x, tuple):
            if not np.allclose(np.array(x), np.array(y), rtol=tol, atol=1e-7):
                return False
        elif isinstance(x, float) or isinstance(y, float):
            if not np.isclose(x, y, rtol=tol, atol=1e-9):
                return False
        elif x != y:
            return False
    return True


def frames_equal(got, want, lvl_tol=REL_TOL):
    """Decoded frames bit-exact (chn, len, err, txt, crc); lvl within tolerance."""
    if [g[:5] for g in got] != [w[:5] for w in want]:
        return False
    gl = np.array([g[5] for g in got], dtype=np.uint32).view(np.float32)
    wl = np.array([w[5] for w in want], dtype=np.uint32).view(np.float32)
    return np.allclose(gl, wl, rtol=lvl_tol, atol=1e-5)


def oracle_dm(oracle, iq, K, wf):
    """(nsamp, nch) envelope through the restatement."""
    return oracle.channelize(iq, K, wf).T.copy()


# ------------------------------------------------------------------ channelizer (K1)

@pytest.mark.parametrize("K,freqs,nblk", [
    (160, synth.DEFAULT_FREQS_MHZ, 3),                                   # config 2 shape
    (192, (131.525, 131.725, 131.825), 2),                               # nch=3: scalar store path
    (200, (129.125, 130.025, 130.450, 131.125, 131.550), 2),             # odd row units (25)
    (16, (131.525, 131.550, 131.475), 4),                                # tiny K, 2 units per row
    (320, (118.000, 119.500, 121.000, 119.000), 1),                      # RTLMULTMAX
    (160, tuple(130.000 + 0.025 * i for i in range(11)), 2),             # 11 channels: two groups of 8
    (44, (131.525, 131.550), 2),                                         # K % 8 != 0: generic kernel
    (8, (131.525,), 2),
])
def test_channelizer_bit_exact(native, oracle, K, freqs, nblk):
    rng = np.random.default_rng(K * 1000 + len(freqs))
    iq = rng.integers(0, 256, size=(1, nblk * 2048 * K), dtype=np.uint8)
    iq[0, :4096] = 0                 # extremes
    iq[0, 4096:8192] = 255
    wf = oracle.wf(K, freqs)
    assert bits_equal(api.build_wf(K, freqs), wf)
    with api.Context(K, 1, len(freqs), nblk) as ctx:
        fd, _, fc = api.plan(K, freqs)
        assert ctx.set_plan(0, fd) == fc
        ctx.submit_host(iq, nblk)
        ctx.sync()
        got = ctx.read_dm(nblk * 1024)[0]
    want = oracle_dm(oracle, iq, K, wf)
    assert bits_equal(got, want)


def test_channelizer_golden_k16(native, oracle):
    iq, exp = load_synth_k16()
    K, nblk = exp["K"], exp["nblk"]
    with api.Context(K, 1, 3, nblk) as ctx:
        ctx.set_wf(0, oracle.wf(K, exp["freqs_mhz"]))
        ctx.submit_host(iq.reshape(1, -1), nblk)
        ctx.sync()
        dm = ctx.read_dm(nblk * 1024)[0]            # (nsamp, nch)
        sha = hashlib.sha256()
        for b in range(nblk):
            for c in range(3):
                sha.update(np.ascontiguousarray(dm[b * 1024:(b + 1) * 1024, c]).tobytes())
        assert sha.hexdigest() == exp["dm_sha256"]
        got = [msg_tuple(m) for m in ctx.drain()]
        want = [msg_tuple_from_json(j) for j in exp["messages"]]
        assert frames_equal(got, want)
        assert got == want                          # incl. the bit pattern of lvl
        for c in range(3):
            assert states_close(ctx.get_state(0, c).vec(), state_tuple_from_json(exp["final_state"][c]))


def test_channelizer_multistream_distinct_plans(native, oracle):
    K, nblk = 160, 2
    plans = [(131.525, 131.725, 131.825, 131.125), (129.125, 130.025, 130.450, 130.000), (136.900, 136.925, 136.975, 136.750)]
    rng = np.random.default_rng(17)
    iq = rng.integers(0, 256, size=(3, nblk * 2048 * K), dtype=np.uint8)
    with api.Context(K, 3, 4, nblk) as ctx:
        for s, fm in enumerate(plans):
            ctx.set_plan(s, api.plan(K, fm)[0])
        ctx.submit_host(iq, nblk)
        ctx.sync()
        got = ctx.read_dm(nblk * 1024)
    for s, fm in enumerate(plans):
        assert bits_equal(got[s], oracle_dm(oracle, iq[s], K, oracle.wf(K, fm))), s


def test_submit_device_matches_submit_host(native, oracle):
    K, nblk, fm = 160, 2, synth.DEFAULT_FREQS_MHZ
    rng = np.random.default_rng(2)
    iq = rng.integers(0, 256, size=(2, nblk * 2048 * K), dtype=np.uint8)
    with api.Context(K, 2, 8, nblk) as ctx:
        for s in range(2):
            ctx.set_plan(s, api.plan(K, fm)[0])
        ctx.submit_host(iq, nblk)
        ctx.sync()
        a = ctx.read_dm(nblk * 1024)
        sa = [ctx.get_state(s, c).vec() for s in range(2) for c in range(8)]
        ctx.reset()
        d = ctx.device_alloc(iq.nbytes)
        ctx.copy_to_device(d, iq)
        ctx.submit_device(d, nblk, iq.strides[0])
        ctx.sync()
        b = ctx.read_dm(nblk * 1024)
        sb = [ctx.get_state(s, c).vec() for s in range(2) for c in range(8)]
        ctx.device_free(d)
    assert bits_equal(a, b) and sa == sb


# ------------------------------------------------------------------ demod + framing (K2)

def test_testwav_seven_messages(native, oracle):
    """BASELINE config 1: test.wav (4 channels of 12.5 kS/s audio) through the soundfile.c loop."""
    x, exp = load_testwav()
    with api.Context(160, 1, 4, 4, flags=1) as ctx:
        got = []
        for s in range(0, len(x), 4096):
            ctx.submit_dm(x[None, s:s + 4096, :])
            ctx.sync()
            got += [msg_tuple(m) for m in ctx.drain()]
        want = [msg_tuple_from_json(j) for j in exp["messages"]]
        assert len(want) == 7
        assert frames_equal(got, want)
        final = [ctx.get_state(0, c) for c in range(4)]
    for c in range(4):
        assert states_close(final[c].vec(), state_tuple_from_json(exp["final_state"][c])), c
    assert sum(int(f.pos) for f in final) == 4 * len(x)


def test_testwav_bit_exact_state_and_lvl(native, oracle):
    """Stronger than the stated tolerance: on this file the device trajectory is bit-identical to
    the reference's (MskPhi/MskDf/MskClk/MskLvlSum/ring), and so is lvl."""
    x, exp = load_testwav()
    with api.Context(160, 1, 4, 53, flags=1) as ctx:
        ctx.submit_dm(x[None, :, :])
        ctx.sync()
        got = sorted(msg_tuple(m) for m in ctx.drain())
        assert got == sorted(msg_tuple_from_json(j) for j in exp["messages"])
        for c in range(4):
            assert ctx.get_state(0, c).vec() == state_tuple_from_json(exp["final_state"][c]), c


def test_demod_chunking_independence(native):
    """demodMSK's result must not depend on how the stream is cut (state carried in HBM)."""
    x, _ = load_testwav()
    x = x[:24000]
    rng = np.random.default_rng(3)
    with api.Context(160, 1, 4, 24, flags=1) as ctx:
        ctx.submit_dm(x[None])
        ctx.sync()
        ref_msgs = [msg_tuple(m) for m in ctx.drain()]
        ref_state = [ctx.get_state(0, c).vec() for c in range(4)]
        ctx.reset()
        pos, got = 0, []
        while pos < len(x):
            n = int(rng.integers(1, 3000))
            ctx.submit_dm(x[None, pos:pos + n])
            pos += n
            if rng.random() < 0.3:
                ctx.sync()
                got += [msg_tuple(m) for m in ctx.drain()]
        ctx.sync()
        got += [msg_tuple(m) for m in ctx.drain()]
        assert sorted(got) == sorted(ref_msgs)
        assert [ctx.get_state(0, c).vec() for c in range(4)] == ref_state


def test_state_get_set_roundtrip(native):
    x, _ = load_testwav()
    with api.Context(160, 1, 4, 8, flags=1) as ctx:
        ctx.submit_dm(x[None, :5000])
        ctx.sync()
        ctx.drain()
        saved = [ctx.get_state(0, c) for c in range(4)]
        ctx.submit_dm(x[None, 5000:12000])
        ctx.sync()
        a_state = [ctx.get_state(0, c).vec() for c in range(4)]
        a_msgs = [msg_tuple(m) for m in ctx.drain()]
        ctx.reset()
        for c in range(4):
            ctx.set_state(0, c, saved[c])
        ctx.submit_dm(x[None, 5000:12000])
        ctx.sync()
        assert [ctx.get_state(0, c).vec() for c in range(4)] == a_state
        assert [msg_tuple(m) for m in ctx.drain()] == a_msgs and len(a_msgs) >= 1


# ------------------------------------------------------------------ whole path

@pytest.mark.parametrize("K,seed,nstreams", [(160, 3, 1), (192, 4, 1), (160, 10, 5)])
def test_full_path_synthetic_vs_oracle(native, oracle, K, seed, nstreams):
    """Seeded IQ with injected messages: frames, emission order, envelope and states vs the oracle."""
    fm = synth.DEFAULT_FREQS_MHZ
    fd, _, fc = api.plan(K, fm)
    secs = 0.7
    nblk = synth.blocks_for_seconds(K, secs)
    plans = [synth.make_plan(K, fm, fc, seconds=secs, seed=seed + 100 * s) for s in range(nstreams)]
    iq = np.stack([synth.render_blocks(p, 0, nblk).reshape(-1) for p in plans])
    wf = oracle.wf(K, fm)
    with api.Context(K, nstreams, len(fm), nblk) as ctx:
        for s in range(nstreams):
            ctx.set_plan(s, fd)
        half = nblk // 2
        bb = 2048 * K
        ctx.submit_host(np.ascontiguousarray(iq[:, :half * bb]), half)
        ctx.submit_host(np.ascontiguousarray(iq[:, half * bb:]), nblk - half)
        ctx.sync()
        got = ctx.drain()
        dm_tail = ctx.read_dm((nblk - half) * 1024)
        states = [[ctx.get_state(s, c).vec() for c in range(len(fm))] for s in range(nstreams)]
        st = ctx.stats()
    assert st.kernel_launches == 6 and st.chan_launches == 2 and st.demod_launches == 2   # K1+K2+K3 per submit
    total = 0
    for s in range(nstreams):
        o = refs.OracleStream(oracle, K, wf)
        o.blocks(iq[s])
        want = [msg_tuple(m) for m in o.msgs()]
        mine = [msg_tuple(m) for m in got if m.stream == s]
        assert frames_equal(mine, want), s          # same frames in the reference's emission order
        assert mine == want, s
        total += len(want)
        assert bits_equal(dm_tail[s][-1024:], np.stack([o.dm(c) for c in range(len(fm))], axis=1))
        for c in range(len(fm)):
            assert states_close(states[s][c], o.chan(c).vec()), (s, c)
            assert states[s][c] == o.chan(c).vec(), (s, c)
    assert total >= 6 * nstreams
    # global emission order: block-major, then stream, then channel (rtl.c:357-360)
    keys = [(m.block, m.stream, m.chn, m.pos) for m in got]
    assert keys == sorted(keys)


@pytest.mark.parametrize("hook", ["sort", "helpers"])
def test_consumer_thread_paths_agree(native, monkeypatch, hook):
    """The consumer thread orders a submit's frames with a stable bucket pass and, for large submits, fills the records
    on helper threads; the comparison-sort fallback (contexts with an unreasonable bucket table) and the helper path are
    forced here through the library's test hooks and must queue exactly the same records in the same order."""
    K, fm, nstreams = 160, synth.DEFAULT_FREQS_MHZ, 6
    fd, _, fc = api.plan(K, fm)
    secs = 0.5
    nblk = synth.blocks_for_seconds(K, secs)
    iq = np.stack([synth.render_blocks(synth.make_plan(K, fm, fc, seconds=secs, seed=70 + s, msgs_per_chan_per_sec=3.0, text_len=(5, 40)), 0, nblk).reshape(-1)
                   for s in range(nstreams)])

    def run():
        with api.Context(K, nstreams, len(fm), nblk) as ctx:
            for s in range(nstreams):
                ctx.set_plan(s, fd)
            half = nblk // 2
            ctx.submit_host(np.ascontiguousarray(iq[:, :half * 2048 * K]), half)
            ctx.submit_host(np.ascontiguousarray(iq[:, half * 2048 * K:]), nblk - half)
            ctx.sync()
            return ctx.drain_records()

    base = run()
    monkeypatch.setenv("ACB_CONSUMER_SORT" if hook == "sort" else "ACB_CONSUMER_HELPERS_MIN", "1")
    other = run()
    rec = lambda r: [(int(m["stream"]), int(m["chn"]), int(m["len"]), int(m["err"]), float(m["lvl"]), int(m["block"]), int(m["pos"]),
                      int(m["soh_pos"]), bytes(m["txt"][:int(m["len"])]), bytes(m["crc"])) for m in r]
    assert len(base) >= 4 * nstreams and rec(base) == rec(other)
    keys = [(int(m["block"]), int(m["stream"]), int(m["chn"]), int(m["pos"])) for m in base]
    assert keys == sorted(keys)


@pytest.mark.parametrize("lanes", [1, 2, 4, 8, 17, 20, 24, 33, 34, 36, 40, -4, -8])
def test_demod_every_lane_width(native, oracle, lanes, monkeypatch):
    """k_demod2 with 1, 2, 4 and 8 lanes per channel (the context picks by chain count; ACB_DEMOD_LANES forces),
    both bit-clock rounding forms (+16), with and without pinned constants (+32), and the round-1 kernel (negative): same frames, same bit-identical
    state as the oracle; 11 channels so that the last warp carries surplus (shadow) groups at every width."""
    monkeypatch.setenv("ACB_DEMOD_LANES", str(lanes))
    K, fm = 160, tuple(130.000 + 0.025 * i for i in range(11))
    fd, _, fc = api.plan(K, fm)
    secs = 0.5
    nblk = synth.blocks_for_seconds(K, secs)
    plans = [synth.make_plan(K, fm, fc, seconds=secs, seed=40 + s) for s in range(2)]
    iq = np.stack([synth.render_blocks(p, 0, nblk).reshape(-1) for p in plans])
    wf = oracle.wf(K, fm)
    with api.Context(K, 2, len(fm), nblk) as ctx:
        for s in range(2):
            ctx.set_plan(s, fd)
        bb = 2048 * K
        ctx.submit_host(np.ascontiguousarray(iq[:, :2 * bb]), 2)            # launches end mid-bit: general path
        ctx.submit_host(np.ascontiguousarray(iq[:, 2 * bb:]), nblk - 2)
        ctx.sync()
        got = ctx.drain()
        states = [[ctx.get_state(s, c).vec() for c in range(len(fm))] for s in range(2)]
    total = 0
    for s in range(2):
        o = refs.OracleStream(oracle, K, wf)
        o.blocks(iq[s])
        want = [msg_tuple(m) for m in o.msgs()]
        assert [msg_tuple(m) for m in got if m.stream == s] == want, s
        total += len(want)
        for c in range(len(fm)):
            assert states[s][c] == o.chan(c).vec(), (s, c)
    assert total >= 4


def _demod_chunks_vs_oracle(ctx, oracle, dm, chans, chunks):
    """dm: (nstreams, nsamp, nch) fed through submit_dm in `chunks`; after every chunk the device states must be
    bit-identical to the oracle's `chans` [stream][chn] fed the same samples, and the chunk's frames identical, in
    the order (stream, channel, time) one submit queues them.  Returns the number of frames."""
    nst, nsamp, nch = dm.shape
    pos = total = 0
    for n in chunks:
        if pos >= nsamp:
            break
        n = min(n, nsamp - pos)
        ctx.submit_dm(dm[:, pos:pos + n])
        ctx.sync()
        got = [(m.stream, msg_tuple(m)) for m in ctx.drain()]
        want = []
        for s in range(nst):
            for c in range(nch):
                sink = refs.Sink()
                oracle.demod(chans[s][c], dm[s, pos:pos + n, c], sink)
                for m in sink.msgs():
                    f = oracle.fec(m)
                    if f is not None:
                        want.append((s, msg_tuple(f)))
        pos += n
        assert got == want, pos
        for s in range(nst):
            for c in range(nch):
                assert ctx.get_state(s, c).vec() == chans[s][c].vec(), (pos, s, c)
        total += len(want)
    return total


@pytest.mark.parametrize("lanes", [1, 2, 4, 8, 17, 20, 24, 33, 34, 36, 40, -4, -8])
def test_demod_envelope_extremes_every_lane_width(native, oracle, lanes, monkeypatch):
    """tests/test_demod_core.py's zero / huge / tiny envelope on the device, where the lanes of a channel's group split
    the mixer samples: 3000 zeros (lvl = 0: the division guard's slow path), a stretch x1e7, zeros, a stretch x1e-30;
    2 streams x 11 channels, each chain its own slices, odd chunk sizes.  (Denormal envelopes are left out: the reference
    is built -Ofast, which flushes them, the oracle is strict IEEE.)"""
    monkeypatch.setenv("ACB_DEMOD_LANES", str(lanes))
    K, fm = 160, synth.DEFAULT_FREQS_MHZ
    _, _, fc = api.plan(K, fm)
    nblk = synth.blocks_for_seconds(K, 1.0)
    env = oracle.channelize(synth.render_blocks(synth.make_plan(K, fm, fc, seconds=1.0, seed=21), 0, nblk).reshape(-1), K, oracle.wf(K, fm))
    nst, nch = 2, 11
    dm = np.empty((nst, 12000, nch), dtype=np.float32)
    for s in range(nst):
        for c in range(nch):
            a, b, off = env[(s * nch + c) % 8], env[(s * nch + c + 3) % 8], 700 * ((s * nch + c) % 7)
            dm[s, :, c] = np.concatenate([np.zeros(3000, np.float32), a[off:off + 4000] * np.float32(1e7), np.zeros(2000, np.float32),
                                          b[off:off + 3000] * np.float32(1e-30)])
    chans = [[oracle.new_chan(c) for c in range(nch)] for _ in range(nst)]
    with api.Context(K, nst, nch, 2, flags=1) as ctx:
        frames = _demod_chunks_vs_oracle(ctx, oracle, dm, chans, [999, 1023, 777, 1, 1501, 2047, 333] * 4)
    assert frames >= 1


@pytest.mark.parametrize("lanes", [1, 2, 4, 8, 24, 40, -4])
def test_foreign_state_on_the_device(native, oracle, lanes, monkeypatch):
    """tests/test_demod_core.py's foreign states (bit clock far ahead, big MskDf) set with acb_set_state on every chain:
    the device follows the reference from there at every lane width."""
    monkeypatch.setenv("ACB_DEMOD_LANES", str(lanes))
    x, _ = load_testwav()
    foreign = [(4.9, 0.0), (7.5, 0.02), (-3.0, -0.03), (0.1, 0.3)]
    nst, nch = 2, 11
    dm = np.empty((nst, 9000, nch), dtype=np.float32)
    chans = [[None] * nch for _ in range(nst)]
    with api.Context(160, nst, nch, 5, flags=1) as ctx:
        for s in range(nst):
            for c in range(nch):
                i = s * nch + c
                dm[s, :, c] = x[(i % 3) * 1000:(i % 3) * 1000 + 9000, i % 4]
                clk, df = foreign[i % 4]
                st = ctx.get_state(s, c)
                st.MskClk, st.MskDf = clk, df
                ctx.set_state(s, c, st)
                oc = oracle.new_chan(c)
                oc.MskClk, oc.MskDf = clk, df
                chans[s][c] = oc
                assert ctx.get_state(s, c).vec() == oc.vec()
        frames = _demod_chunks_vs_oracle(ctx, oracle, dm, chans, [1001, 37, 2999, 511, 4452])
    assert frames >= 1


def test_corrupted_frames_fec_on_gpu_path(native, oracle):
    K, fm = 160, (131.525, 131.725, 131.825)
    fd, _, fc = api.plan(K, fm)
    plan = synth.make_plan(K, fm, fc, seconds=1.5, seed=21, msgs_per_chan_per_sec=6.0, text_len=(5, 40))
    flips = [[(3, 0x04)], [(5, 0x01), (9, 0x80)], [(7, 0x21)], [(-2, 0x10)], [(2, 1), (4, 2), (6, 4), (8, 8)],
             [(1, 0x40), (-3, 0x02)], [], [(20, 0xFF)], [(0, 0x08), (10, 0x08), (11, 0x08)]]
    for i, b in enumerate(plan.bursts):
        b.frame = synth.corrupt_frame(b.frame, [f for f in flips[i % len(flips)] if f[0] < len(b.frame) - 30])
    nblk = synth.blocks_for_seconds(K, 1.5)
    iq = synth.render_blocks(plan, 0, nblk).reshape(1, -1)
    o = refs.OracleStream(oracle, K, oracle.wf(K, fm))
    o.blocks(iq[0])
    want = [msg_tuple(m) for m in o.msgs()]
    with api.Context(K, 1, 3, nblk) as ctx:
        ctx.set_plan(0, fd)
        ctx.submit_host(iq, nblk)
        ctx.sync()
        got = [msg_tuple(m) for m in ctx.drain()]
        st = ctx.stats()
    assert got == want and any(g[2] > 0 for g in got)
    assert st.fec_dropped > 0 and st.raw_frames == len(got) + st.fec_dropped


def test_argument_errors(native):
    with api.Context(160, 2, 8, 2) as ctx:
        iq = np.zeros((2, 3 * 2048 * 160), dtype=np.uint8)
        with pytest.raises(api.AcbError):
            ctx.submit_host(iq, 3)                       # nblk > max_blocks
        with pytest.raises(api.AcbError):
            ctx.set_plan(0, [118000000, 137000000, 1, 2, 3, 4, 5, 6])     # span too wide
        with pytest.raises(api.AcbError):
            ctx.set_plan(5, api.plan(160, synth.DEFAULT_FREQS_MHZ)[0])     # stream out of range
        assert ctx.sync() == 0 and ctx.drain() == []
    with pytest.raises(api.AcbError):
        api.Context(160, 0, 8, 2)


# ------------------------------------------------------------------ BASELINE-size properties

def test_full_size_replica_property(native, oracle):
    """configs[1] shape at bench scale (many streams x 8 channels x 16 blocks): streams fed the
    same bytes must produce identical envelopes, states and frames (determinism across CTAs/SMs),
    and one of them is checked against the oracle."""
    K, fm, nblk, nstreams = 160, synth.DEFAULT_FREQS_MHZ, 16, 64
    fd, _, fc = api.plan(K, fm)
    base = [synth.render_blocks(synth.make_plan(K, fm, fc, seconds=1.3, seed=40 + i), 0, nblk).reshape(-1) for i in range(2)]
    iq = np.stack([base[s % 2] for s in range(nstreams)])
    with api.Context(K, nstreams, 8, nblk) as ctx:
        for s in range(nstreams):
            ctx.set_plan(s, fd)
        ctx.submit_host(iq, nblk)
        ctx.sync()
        got = ctx.drain()
        dm = ctx.read_dm(nblk * 1024)
        states = [[ctx.get_state(s, c).vec() for c in range(8)] for s in range(nstreams)]
    for s in range(2, nstreams):
        assert bits_equal(dm[s], dm[s % 2])
        assert states[s] == states[s % 2]
    per = {}
    for m in got:
        per.setdefault(m.stream, []).append(msg_tuple(m))
    for s in range(2, nstreams):
        assert per.get(s, []) == per.get(s % 2, [])
    for s in range(2):
        o = refs.OracleStream(oracle, K, oracle.wf(K, fm))
        o.blocks(base[s])
        assert per.get(s, []) == [msg_tuple(m) for m in o.msgs()]
        assert len(per.get(s, [])) > 0


# ------------------------------------------------------------------ other BASELINE configs

def test_config3_64_channels_k192(native, oracle):
    """BASELINE configs[2]: rateMult=192 (2.4 MS/s), 64 channels on a 25 kHz raster across the band,
    one stream: 8 channel groups per tile in K1, 8 warps per stream in K2.  The reference caps at
    16 channels (MAXNBCHANNELS), so the expectation comes from the restatement (pinned <= 16 ch)."""
    K, nblk = 192, 6
    fm = tuple(130.000 + 0.025 * i for i in range(64))
    fd, _, fc = api.plan(K, fm)
    assert fc != 0
    plan = synth.make_plan(K, fm, fc, seconds=nblk * 1024 / 12500, seed=64, msgs_per_chan_per_sec=2.0, text_len=(5, 30), amp=(6.0, 10.0))
    iq = synth.render_blocks(plan, 0, nblk).reshape(1, -1)
    wf = oracle.wf(K, fm)
    o = refs.OracleStream(oracle, K, wf)
    o.blocks(iq[0])
    want = [msg_tuple(m) for m in o.msgs()]
    with api.Context(K, 1, 64, nblk) as ctx:
        ctx.set_plan(0, fd)
        ctx.submit_host(iq, nblk)
        ctx.sync()
        got = [msg_tuple(m) for m in ctx.drain()]
        dm = ctx.read_dm(nblk * 1024)[0]
        for c in (0, 7, 8, 31, 63):
            assert ctx.get_state(0, c).vec() == o.chan(c).vec(), c
    assert bits_equal(dm[-1024:], np.stack([o.dm(c) for c in range(64)], axis=1))
    assert got == want and len(got) >= 20


def test_config4_128_streams(native, oracle):
    """BASELINE configs[3] per-GPU shape (1024 channels = 128 streams x 8): every stream distinct
    (seed = stream index), every stream checked against the oracle."""
    K, fm, nblk, nstreams = 160, synth.DEFAULT_FREQS_MHZ, 4, 128
    fd, _, fc = api.plan(K, fm)
    secs = nblk * 1024 / 12500
    iq = np.stack([synth.render_blocks(synth.make_plan(K, fm, fc, seconds=secs, seed=s, text_len=(5, 25), msgs_per_chan_per_sec=3.0), 0, nblk).reshape(-1)
                   for s in range(nstreams)])
    wf = oracle.wf(K, fm)
    with api.Context(K, nstreams, 8, nblk) as ctx:
        for s in range(nstreams):
            ctx.set_plan(s, fd)
        ctx.submit_host(iq, nblk)
        ctx.sync()
        got = ctx.drain()
    per = {}
    for m in got:
        per.setdefault(m.stream, []).append(msg_tuple(m))
    total = 0
    for s in range(nstreams):
        o = refs.OracleStream(oracle, K, wf)
        o.blocks(iq[s])
        want = [msg_tuple(m) for m in o.msgs()]
        assert per.get(s, []) == want, s
        total += len(want)
    assert total > 300


def test_wide_stream_channel_sharding(native):
    """One stream, channels sharded over the visible GPUs with a single NCCL broadcast of the raw
    block (world size 1 when only one GPU is visible: same code path minus the collective)."""
    import json as _json
    import subprocess
    import sys as _sys
    import torch
    n = min(torch.cuda.device_count(), 2)
    worker = str(__import__("pathlib").Path(__file__).resolve().parent / "wide_stream_worker.py")
    if n >= 2:
        cmd = [_sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={n}",
               "--master-addr", "127.0.0.1", "--master-port", "29533", worker]
    else:
        cmd = [_sys.executable, worker]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-3000:]
    line = [l for l in r.stdout.splitlines() if l.startswith("{")][-1]
    res = _json.loads(line)
    assert res["match"] and res["world"] == max(n, 1) and res["frames"] >= 8


def test_device_block_fec_fuzz_matches_oracle(native, oracle):
    """k_block_fec (one thread per frame) against the restatement's blk_thread on 6000 fuzzed
    frames: clean, 1-3 parity errors, double-bit errors, BCS errors, hopeless ones, short ones."""
    from test_oracle_vs_reference import _fec_cases
    rng = np.random.default_rng(4321)
    raw, want = [], []
    for chn, txt, crc in _fec_cases(rng, 6000):
        a, o = api.Msg(), refs.Msg()
        for m in (a, o):
            m.chn, m.len = chn, len(txt)
            m.txt[:len(txt)] = txt
            m.crc[:] = crc
        raw.append(a)
        want.append(oracle.fec(o))
    with api.Context(160, 1, 1, 1) as ctx:
        got = ctx.block_fec_batch(raw)
    n_out = n_fixed = 0
    for g, w in zip(got, want):
        assert (g is None) == (w is None)
        if g is not None:
            assert (g.len, g.err, bytes(g.txt[:g.len])) == (w.len, w.err, bytes(w.txt[:w.len]))
            n_out += 1
            n_fixed += g.err > 0
    assert n_out > 1000 and n_fixed > 200
