"""The channelizers and the streaming front-ends across several streams with their own plans, several channel groups,
ragged / strided / maximal submits, full-scale input, and the emission order of the streaming front-ends.

The hot paths index by stream (blockIdx.y) and by channel group (blockIdx.z): each stream here has its own channel set,
so its own centre frequency, bins and twiddles, and 17 channels make three groups, the last with a single channel.
Every envelope is held bit for bit to the oracle's operation-for-operation restatement (the literal arithmetic for the
exact kernels, orc_channelize_dft* / orc_channelize_rdft for the fast forms), and the fast forms also to a float64 DFT
computed here.  Frames are compared IN ORDER with a plain model of the reference loop (common.emission_model)."""
import numpy as np
import pytest

import refs
from acarsdec_b200 import api, synth
from common import assert_emission_order, bits_equal, emission_model, msg_tuple

pytestmark = pytest.mark.gpu

FLAG_REAL, FLAG_CS16, FAST = 2, 4, 8
IDEAL_EPS = 1e-6      # |fast - exact DFT bin| <= IDEAL_EPS * the row's total in-band signal (tests/test_fast_oracle.py)
NCH = 17              # three channel groups of 8, the last holding one channel


def _grid_sets(nstreams, base_mhz, seed, span=24):
    """Per stream: NCH channels on the 25 kHz grid above its own base (so its own Fc, and every bin k even, as the u8
    and CS16 fast forms need), in shuffled order so that the residues (k/2) mod 4 appear out of order."""
    rng = np.random.default_rng(seed)
    out = []
    for s in range(nstreams):
        offs = rng.choice(span, size=NCH, replace=False)
        out.append(tuple(round(base_mhz[s] + 0.025 * int(o), 4) for o in offs))
    return out


def _assert_residues(kbin):
    r = [(int(k) // 2) % 4 for k in kbin]
    assert set(r) == {0, 1, 2, 3} and r != sorted(r), r


def _lvl(t):
    return float(np.array([t[5]], dtype=np.uint32).view(np.float32)[0])


# ------------------------------------------------------------------ u8 IQ: fast channelizer, distinct plans per stream

U8_VARIANTS = {                                   # kernel switch -> (environment, the restatement it matches)
    "dft1": ({}, True),                                                   # default: one row per lane, folded
    "rows2": ({"ACB_FAST_ROWS": "2", "ACB_FAST_FOLD8": "0"}, False),     # two rows per lane, 4-way split
    "rows2fold8": ({"ACB_FAST_ROWS": "2", "ACB_FAST_FOLD8": "1"}, True),
    "warps4": ({"ACB_FAST_WARPS": "4"}, True),
}


@pytest.mark.parametrize("variant", list(U8_VARIANTS))
@pytest.mark.parametrize("K", [160, 192])
def test_u8_fast_distinct_plans_three_groups(native, oracle, monkeypatch, K, variant):
    env, fold8 = U8_VARIANTS[variant]
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    nst, secs = 4, 0.5
    sets = _grid_sets(nst, (129.0, 129.7, 130.4, 131.1), seed=K)
    nblk = synth.blocks_for_seconds(K, secs)
    plans, iq, fcs = [], [], set()
    for s, fm in enumerate(sets):
        fd, _, fc = oracle.plan(K, fm)
        fp = oracle.fast_plan(K, fd, fc)
        assert fp is not None, s
        _assert_residues(fp[0])
        plans.append((fd, fc, fp))
        fcs.add(fc)
        p = synth.make_plan(K, fm, fc, seconds=secs, seed=300 + 10 * s + K, msgs_per_chan_per_sec=3.0, text_len=(5, 30), amp=(5.0, 9.0))
        iq.append(synth.render_blocks(p, 0, nblk).reshape(-1))
    assert len(fcs) == nst
    iq = np.stack(iq)
    restated = [oracle.channelize_dft(iq[s], K, kb, tw, fold8) for s, (_, _, (kb, tw)) in enumerate(plans)]
    bb, half = 2048 * K, nblk // 2 + 1
    with api.Context(K, nst, NCH, nblk, flags=FAST) as ctx:
        for s, (fd, fc, _) in enumerate(plans):
            assert ctx.set_plan(s, fd) == fc
        got = []
        for b0, b1 in ((0, half), (half, nblk)):
            ctx.submit_host(np.ascontiguousarray(iq[:, b0 * bb:b1 * bb]), b1 - b0)
            ctx.sync()
            got += ctx.drain()
            dm = ctx.read_dm((b1 - b0) * 1024)
            for s in range(nst):
                assert bits_equal(dm[s], restated[s][:, b0 * 1024:b1 * 1024].T.copy()), (s, b0)
        assert ctx.stats().fast_chan_launches == 2
        states = [[ctx.get_state(s, c).vec() for c in range(NCH)] for s in range(nst)]
    model, chans = emission_model(oracle, restated, range(0, nblk * 1024, 1024))
    assert_emission_order(got, model)
    assert states == [[ch.vec() for ch in row] for row in chans]
    total = 0
    for s in range(nst):                                       # the literal arithmetic decodes the same frames
        o = refs.OracleStream(oracle, K, oracle.wf(K, sets[s]))
        o.blocks(iq[s])
        want = [msg_tuple(m) for m in o.msgs()]
        mine = [msg_tuple(m) for m in got if m.stream == s]
        assert [t[:-1] for t in mine] == [t[:-1] for t in want], s
        for a, b in zip(mine, want):
            assert abs(_lvl(a) - _lvl(b)) <= 1e-3
        total += len(want)
    assert total >= 4 * nst


def test_u8_mixed_raster_takes_the_exact_kernel(native, oracle):
    """One stream with a caller's table: the whole launch takes the exact kernel; planning that stream again brings
    the fast form back."""
    K, nst, nblk = 160, 3, 2
    sets = _grid_sets(nst, (129.2, 130.3, 131.0), seed=5)
    iq = np.random.default_rng(8).integers(0, 256, size=(nst, nblk * 2048 * K), dtype=np.uint8)
    lit = [oracle.channelize(iq[s], K, oracle.wf(K, fm)) for s, fm in enumerate(sets)]
    with api.Context(K, nst, NCH, nblk, flags=FAST) as ctx:
        fds = []
        for s, fm in enumerate(sets):
            fds.append(oracle.plan(K, fm)[0])
            ctx.set_plan(s, fds[-1])
        ctx.set_wf(1, oracle.wf(K, sets[1]))
        ctx.submit_host(iq, nblk)
        ctx.sync()
        dm = ctx.read_dm(nblk * 1024)
        assert ctx.stats().fast_chan_launches == 0
        for s in range(nst):
            assert bits_equal(dm[s], lit[s].T.copy()), s
        ctx.set_plan(1, fds[1])
        ctx.submit_host(iq, nblk)
        ctx.sync()
        dm = ctx.read_dm(nblk * 1024)
        assert ctx.stats().fast_chan_launches == 1
    for s, fm in enumerate(sets):
        fd, _, fc = oracle.plan(K, fm)
        kb, tw = oracle.fast_plan(K, fd, fc)
        assert bits_equal(dm[s], oracle.channelize_dft(iq[s], K, kb, tw, True).T.copy()), s


# ------------------------------------------------------------------ streaming front-ends (CS16, real): helpers

CS16_VARIANTS = (0, 1, 0)          # soapy, sdrplay, soapy: the twiddles carry each variant's scale


def _bursts(plan, nch, seconds, rng, amp):
    for ch in range(nch):
        t = 0.003 + 0.004 * ch
        while True:
            fr = synth.frame_bytes(synth.random_text(rng, int(rng.integers(3, 24))))
            dur = len(fr) * 8 / 2400
            if t + dur + 0.01 > seconds:
                break
            plan.bursts.append(synth.Burst(chan=ch, t0=t, frame=fr, amp=float(rng.uniform(*amp)), phase=float(rng.uniform(0, 6))))
            t += dur + float(rng.uniform(0.01, 0.05))


def _cs16_streams(oracle, K, seconds, seed, nst=3):
    """(iq (nst, n, 2) int16, [(freqs_hz, fc, variant)]) with NCH channels per stream, each stream its own set."""
    sets = _grid_sets(nst, (129.3, 130.1, 131.2), seed=seed)
    n = int(seconds * K * 12500) + 77
    iq, plans = [], []
    for s, fm in enumerate(sets):
        fd, _, fc = oracle.plan(K, fm)
        p = synth.StreamPlan(K=K, freqs_hz=tuple(fd), fc_hz=fc, seed=seed + s, noise_sigma=1.5)
        _bursts(p, NCH, seconds, np.random.default_rng(seed + s), (6.0, 14.0))
        iq.append(synth.render_cs16(p, 0, n))
        plans.append((fd, fc, CS16_VARIANTS[s % len(CS16_VARIANTS)]))
    return np.stack(iq), plans


def _real_streams(oracle, rate, seconds, seed, nst=3):
    """(x (nst, n) float32, [(freqs_hz, fc)], K): NCH channels on the 12.5 kHz raster per stream, each its own set."""
    rng = np.random.default_rng(seed)
    xs, plans = [], []
    n = int(seconds * rate)
    for s in range(nst):
        offs = rng.choice(40, size=NCH, replace=False)
        fm = tuple(round(129.5 + 0.6 * s + 0.0125 * int(o), 4) for o in offs)
        fd, fc, K = oracle.air_plan(rate, fm)
        p = synth.StreamPlan(K=K, freqs_hz=tuple(fd), fc_hz=fc, seed=seed + s, noise_sigma=1.0)
        _bursts(p, NCH, seconds, rng, (8.0, 20.0))
        xs.append(synth.render_real(p, 0, n))
        plans.append((fd, fc, fm))
    return np.stack(xs), plans, K


def _expected_cs16(oracle, iq, K, plans, fast):
    nout = iq.shape[1] // K
    out = []
    for s, (fd, fc, var) in enumerate(plans):
        x = iq[s, :nout * K]
        if fast:
            fp = oracle.fast_plan_cs16(var, K, fd, fc)
            assert fp is not None, s
            _assert_residues(fp[0])
            out.append(oracle.channelize_dft8_cs16(x, K, *fp))
        else:
            out.append(oracle.channelize_cs16(var, x, K, oracle.cs16_osc(var, K, fd, fc)))
    return out


def _expected_real(oracle, x, K, plans, fast):
    nout = x.shape[1] // K
    out = []
    for s, (fd, fc, fm) in enumerate(plans):
        if fast:
            fp = oracle.fast_plan_air(K, fd, fc)
            assert fp is not None, s
            assert len({int(k) % 4 for k in fp[0]}) == 4
            out.append(oracle.channelize_rdft(x[s, :nout * K], K, *fp))
        else:
            out.append(oracle.channelize_real(x[s, :nout * K], K, oracle.air_wf(K * 12500, fm)))
    return out


def _submit(ctx, kind, part, strided):
    """One submit of `part` ((nst, n, 2) int16 or (nst, n) float32), kind 'cs16' | 'planar' | 'real'; `strided` puts
    every stream in a host buffer whose stride is larger than the submit, with the stride passed explicitly."""
    nst, n = part.shape[0], part.shape[1]
    stride = n + 37 if strided else n
    if kind == "real":
        buf = np.zeros((nst, stride), dtype=np.float32)
        buf[:, :n] = part
        return ctx.submit_real(buf[:, :n])
    if kind == "cs16":
        buf = np.zeros((nst, stride, 2), dtype=np.int16)
        buf[:, :n] = part
        return api._check(ctx.lib, ctx.lib.acb_submit_cs16_host(ctx.h, buf.ctypes.data, stride, n))
    xi = np.zeros((nst, stride), dtype=np.int16)
    xq = np.zeros((nst, stride), dtype=np.int16)
    xi[:, :n], xq[:, :n] = part[..., 0], part[..., 1]
    return api._check(ctx.lib, ctx.lib.acb_submit_cs16_planar_host(ctx.h, xi.ctypes.data, xq.ctypes.data, stride, n))


def _ragged_sizes(K, total, seed):
    """Below one row, a few rows, just over 1024 rows, partial blocks whose row count is not a multiple of 32, then random."""
    fixed = [K // 3, 5 * K + 7, 1025 * K + 13, 33 * K + 5, 1, 100 * K + K // 2, 31 * K + 1, 2 * 1024 * K + 999]
    rng = np.random.default_rng(seed)
    out, pos = [], 0
    while pos < total:
        n = fixed[len(out)] if len(out) < len(fixed) else int(rng.integers(1, 1500 * K))
        n = min(n, total - pos)
        out.append(n)
        pos += n
    return out


def _run(ctx, kind, xs, sizes, want, strided_every=2):
    """Feed xs in `sizes` pieces, every `strided_every`-th one from a strided buffer; each submit's envelope checked bit for
    bit against `want` (per stream (nch, nout)).  Returns (frames in queue order, submit boundaries in envelope samples)."""
    pos = done = 0
    frames, cuts = [], []
    for i, n in enumerate(sizes):
        m = _submit(ctx, kind, xs[:, pos:pos + n], strided_every and i % strided_every == 1)
        pos += n
        ctx.sync()
        frames += ctx.drain()
        if m:
            cuts.append(done)
            dm = ctx.read_dm(m)
            for s in range(xs.shape[0]):
                assert bits_equal(dm[s], want[s][:, done:done + m].T.copy()), (i, s, done, m)
            done += m
    assert done == want[0].shape[1]
    return frames, cuts


# ------------------------------------------------------------------ CS16: distinct plans and variants, ragged and strided submits

@pytest.mark.parametrize("planar", [False, True])
@pytest.mark.parametrize("mode", ["exact", "fast2", "fast1"])            # fastW: ACB_FAST_WARPS = W
@pytest.mark.parametrize("K", [160, 192])
def test_cs16_distinct_plans_ragged_strided(native, oracle, monkeypatch, K, mode, planar):
    if mode != "exact":
        monkeypatch.setenv("ACB_FAST_WARPS", mode[-1])
    iq, plans = _cs16_streams(oracle, K, 0.3, seed=K + 3 * planar)
    want = _expected_cs16(oracle, iq, K, plans, mode != "exact")
    nout = want[0].shape[1]
    with api.Context(K, len(plans), NCH, nout // 1024 + 2, flags=FLAG_CS16 | (FAST if mode != "exact" else 0)) as ctx:
        for s, (fd, fc, var) in enumerate(plans):
            assert ctx.set_plan_cs16(s, fd, var) == fc
        got, cuts = _run(ctx, "planar" if planar else "cs16", iq, _ragged_sizes(K, iq.shape[1], K), want)
        st = ctx.stats()
        assert st.fast_chan_launches == (st.chan_launches if mode != "exact" else 0) and st.chan_launches > 0
        states = [[ctx.get_state(s, c).vec() for c in range(NCH)] for s in range(len(plans))]
    model, chans = emission_model(oracle, want, cuts)           # ACB_GROUP_SUBMIT: a group per submit
    assert_emission_order(got, model)
    assert states == [[ch.vec() for ch in row] for row in chans]
    assert len(model) >= 2 * len(plans)


# ------------------------------------------------------------------ real input: distinct plans, K = 200 and 800, exact and fast

@pytest.mark.parametrize("fast", [False, True])
@pytest.mark.parametrize("rate", [2500000, 10000000])
def test_real_distinct_plans_ragged_strided(native, oracle, rate, fast):
    x, plans, K = _real_streams(oracle, rate, 0.3 if rate < 5000000 else 0.25, seed=rate // 100000)
    assert len({fc for _, fc, _ in plans}) == len(plans)
    want = _expected_real(oracle, x, K, plans, fast)
    nout = want[0].shape[1]
    with api.Context(K, len(plans), NCH, nout // 1024 + 2, flags=FLAG_REAL | (FAST if fast else 0)) as ctx:
        for s, (fd, fc, _) in enumerate(plans):
            assert ctx.set_plan_air(s, fd) == fc
        got, cuts = _run(ctx, "real", x, _ragged_sizes(K, x.shape[1], K), want)
        st = ctx.stats()
        assert st.fast_chan_launches == (st.chan_launches if fast else 0) and st.chan_launches > 0
        states = [[ctx.get_state(s, c).vec() for c in range(NCH)] for s in range(len(plans))]
    model, chans = emission_model(oracle, want, cuts)
    assert_emission_order(got, model)
    assert states == [[ch.vec() for ch in row] for row in chans]
    assert len(model) >= len(plans)


# ------------------------------------------------------------------ the largest submit, and one sample more

@pytest.mark.parametrize("kind,fast", [("real", False), ("real", True), ("cs16", True), ("planar", False)])
def test_largest_submit_and_one_more(native, oracle, kind, fast):
    """(max_blocks*1024 + 1)*K - 1 - carry samples: max_blocks*1024 outputs and a carry of K - 1; one sample more is
    ACB_ERR_ARG and changes nothing (carry, buffers): the context goes on with the oracle's envelope, states, frames."""
    mb = 2
    if kind == "real":
        x, plans, K = _real_streams(oracle, 2500000, 0.3, seed=71)
        want = _expected_real(oracle, x, K, plans, fast)
        flags = FLAG_REAL
    else:
        K = 160
        x, plans = _cs16_streams(oracle, K, 0.3, seed=72)
        want = _expected_cs16(oracle, x, K, plans, fast)
        flags = FLAG_CS16
    nst = len(plans)
    with api.Context(K, nst, NCH, mb, flags=flags | (FAST if fast else 0)) as ctx:
        for s, p in enumerate(plans):
            if kind == "real":
                ctx.set_plan_air(s, p[0])
            else:
                ctx.set_plan_cs16(s, p[0], p[2])
        carry0 = 37
        first = 5 * K + carry0
        nmax = (mb * 1024 + 1) * K - 1 - carry0
        assert first + nmax + 1 <= x.shape[1]
        pos, done, frames, cuts = 0, 0, [], []

        def step(n, strided=True):
            nonlocal pos, done
            m = _submit(ctx, kind, x[:, pos:pos + n], strided)
            pos += n
            ctx.sync()
            frames.extend(ctx.drain())
            if m:
                cuts.append(done)
                dm = ctx.read_dm(m)
                for s in range(nst):
                    assert bits_equal(dm[s], want[s][:, done:done + m].T.copy()), (pos, s)
                done += m
            return m

        assert step(first) == 5
        for strided in (False, True):
            with pytest.raises(api.AcbError, match="error -1:"):          # ACB_ERR_ARG
                _submit(ctx, kind, x[:, pos:pos + nmax + 1], strided)
        assert step(nmax) == mb * 1024
        assert step(1) == 1                                        # the carry was K - 1
        for n in _ragged_sizes(K, x.shape[1] - pos, 5)[2:]:
            step(min(n, mb * 1024 * K))
        while pos < x.shape[1]:
            step(min(x.shape[1] - pos, mb * 1024 * K))
        states = [[ctx.get_state(s, c).vec() for c in range(NCH)] for s in range(nst)]
    want = [w[:, :done] for w in want]
    model, chans = emission_model(oracle, want, cuts)
    assert_emission_order(frames, model)
    assert states == [[ch.vec() for ch in row] for row in chans]
    assert len(model) >= nst


# ------------------------------------------------------------------ full-scale input against a float64 DFT

def _full_scale(kind, rng, rows, K):
    """rows x K samples of extremes: constant minimum, constant maximum, alternating, random over the whole range."""
    q = rows // 4
    if kind == "u8":
        x = rng.integers(0, 256, size=(rows, 2 * K), dtype=np.uint8)
        x[:q // 2] = 0
        x[q // 2:q] = 255
        x[q:q + q // 2] = np.tile(np.array([0, 255], np.uint8), K)                 # I = 0, Q = 255
        x[q + q // 2:2 * q] = np.tile(np.array([0, 0, 255, 255], np.uint8), K // 2)  # sample by sample
        x[2 * q:2 * q + q // 2] = np.tile(np.array([255, 0, 0, 255], np.uint8), K // 2)
        return x.reshape(-1)
    if kind == "cs16":
        lo, hi = -32768, 32767
        x = rng.integers(lo, hi + 1, size=(rows, K, 2), dtype=np.int16)
        x[:q // 2] = lo
        x[q // 2:q] = hi
        x[q:q + q // 2, :, 0], x[q:q + q // 2, :, 1] = lo, hi
        x[q + q // 2:2 * q] = np.where((np.arange(K) % 2)[:, None] == 0, lo, hi).astype(np.int16)
        x[2 * q:2 * q + q // 2] = np.where((np.arange(K) % 2)[:, None] == 0, hi, lo).astype(np.int16)
        return x.reshape(-1, 2)
    x = rng.uniform(-1, 1, size=(rows, K))
    x[rows // 2:] *= 1e4
    x[q:q + q // 4] = np.where(np.arange(K) % 2 == 0, 1e4, -1e4)
    return x.astype(np.float32).reshape(-1)


def _ideal(kind, x, K, kbin, scale=1.0):
    """(total in-band signal per row, |exact DFT bin| per channel and row) in float64, as tests/test_fast_oracle.py."""
    if kind == "u8":
        v = x.reshape(-1, K, 2).astype(np.float64)
        xc = v[..., 0] + 1j * v[..., 1]
        total = np.hypot(v[..., 0] - 127.5, v[..., 1] - 127.5).sum(axis=1) / K / 127.5
        norm = K * 127.5
    elif kind == "cs16":
        v = x.reshape(-1, K, 2).astype(np.float64)
        xc = v[..., 0] + 1j * v[..., 1]
        total = np.hypot(v[..., 0], v[..., 1]).sum(axis=1) / K * scale
        norm = K / scale
    else:
        xc = x.reshape(-1, K).astype(np.float64)
        total = np.abs(xc).sum(axis=1) / K
        norm = K
    ideal = np.stack([np.abs(xc @ np.exp(-2j * np.pi * int(k) * np.arange(K) / K)) / norm for k in kbin])
    return total, ideal


@pytest.mark.parametrize("kind", ["u8", "cs16", "real"])
def test_full_scale_input_exact_and_fast(native, oracle, kind):
    """The fast forms' converters are exact over the whole input range (u8: biased sums; CS16: XOR 0x8000 / 0x7fff in the
    mantissa of 2^23): every fast envelope bit-exact against its restatement AND within IDEAL_EPS of the row's total
    in-band signal of the float64 DFT bin; the exact kernels bit-exact against the literal arithmetic."""
    rng = np.random.default_rng({"u8": 1, "cs16": 2, "real": 3}[kind])
    nst = 3
    if kind == "real":
        K = 200
        plans = _real_streams(oracle, K * 12500, 0.001, seed=90)[1]
        rows = 1024 + 333
        flags = FLAG_REAL
    else:
        K = 160
        sets = _grid_sets(nst, (129.3, 130.1, 131.2), seed=91)
        plans = [(*oracle.plan(K, fm)[::2], CS16_VARIANTS[s], fm) for s, fm in enumerate(sets)]
        rows = 2048 if kind == "u8" else 1024 + 333
        flags = FLAG_CS16 if kind == "cs16" else 0
    xs = [_full_scale(kind, rng, rows, K) for _ in range(nst)]
    lit, fast = [], []
    for s in range(nst):
        if kind == "u8":
            fd, fc, _, fm = plans[s]
            fp = oracle.fast_plan(K, fd, fc)
            lit.append(oracle.channelize(xs[s], K, oracle.wf(K, fm)))
            fast.append(oracle.channelize_dft(xs[s], K, *fp, True))
            scale = 1.0
        elif kind == "cs16":
            fd, fc, var, _ = plans[s]
            fp = oracle.fast_plan_cs16(var, K, fd, fc)
            lit.append(oracle.channelize_cs16(var, xs[s], K, oracle.cs16_osc(var, K, fd, fc)))
            fast.append(oracle.channelize_dft8_cs16(xs[s], K, *fp))
            scale = 1.0 / 32768 if var == 0 else 0.25
        else:
            fd, fc, fm = plans[s]
            fp = oracle.fast_plan_air(K, fd, fc)
            lit.append(oracle.channelize_real(xs[s], K, oracle.air_wf(K * 12500, fm)))
            fast.append(oracle.channelize_rdft(xs[s], K, *fp))
            scale = 1.0
        total, ideal = _ideal(kind, xs[s], K, fp[0], scale)
        err = (np.abs(fast[-1].astype(np.float64) - ideal) / total[None, :]).max()
        assert err <= IDEAL_EPS, (s, err)
    for f in (0, FAST):
        want = fast if f else lit
        with api.Context(K, nst, NCH, rows // 1024 + 1, flags=flags | f) as ctx:
            for s in range(nst):
                if kind == "u8":
                    ctx.set_plan(s, plans[s][0])
                elif kind == "cs16":
                    ctx.set_plan_cs16(s, plans[s][0], plans[s][2])
                else:
                    ctx.set_plan_air(s, plans[s][0])
            if kind == "u8":
                ctx.submit_host(np.stack(xs), rows // 1024)
                m = rows
            else:
                m = _submit(ctx, "real" if kind == "real" else "cs16", np.stack(xs), False)
                assert m == rows
            ctx.sync()
            dm = ctx.read_dm(m)
            assert ctx.stats().fast_chan_launches == (1 if f else 0)
        for s in range(nst):
            assert bits_equal(dm[s], want[s].T.copy()), (f, s)


# ------------------------------------------------------------------ emission order of the streaming front-ends

def _group_cuts(unit, period, K, nout):
    if unit == 1:                                       # ACB_GROUP_OUTPUTS
        return list(range(0, nout, period))
    return sorted({0} | {t * period // K for t in range(1, nout * K // period + 2)})   # ACB_GROUP_INPUT: transfer t starts at output floor(tT/K)


@pytest.mark.parametrize("period", [1024, 512, 97])     # soapy.c:247, sdrplay.c:229, and an odd one
def test_cs16_emission_groups_outputs(native, oracle, period):
    K = 160
    iq, plans = _cs16_streams(oracle, K, 0.3, seed=200 + period)
    want = _expected_cs16(oracle, iq, K, plans, True)
    nout = want[0].shape[1]
    with api.Context(K, len(plans), NCH, nout // 1024 + 2, flags=FLAG_CS16 | FAST) as ctx:
        ctx.set_emission_groups(1, period)
        for s, (fd, fc, var) in enumerate(plans):
            ctx.set_plan_cs16(s, fd, var)
        pos, got, i = 0, [], 0
        while pos < nout:                               # whole groups: 1, 3, 2, 5, ... per submit
            rows = min((1, 3, 2, 5, 4)[i % 5] * period, nout - pos)
            assert _submit(ctx, "cs16", iq[:, pos * K:(pos + rows) * K], i % 2 == 1) == rows
            pos += rows
            i += 1
        ctx.sync()
        got = ctx.drain()
    model, _ = emission_model(oracle, want, _group_cuts(1, period, K, nout))
    assert_emission_order(got, model)
    assert len({lo for *_, lo, _, _ in model}) >= 3          # frames in several groups


@pytest.mark.parametrize("T", [65536, 150001])          # air.c's transfer at 2.5 MS/s (327.68 outputs), and one < 1024 K, not a multiple of K
def test_real_emission_groups_input(native, oracle, T):
    x, plans, K = _real_streams(oracle, 2500000, 0.3, seed=T % 1000)
    ntr = x.shape[1] // T
    x = np.ascontiguousarray(x[:, :ntr * T])
    want = _expected_real(oracle, x, K, plans, True)
    nout = want[0].shape[1]
    with api.Context(K, len(plans), NCH, 3 * T // (K * 1024) + 2, flags=FLAG_REAL | FAST) as ctx:
        ctx.set_emission_groups(2, T)
        for s, (fd, fc, _) in enumerate(plans):
            ctx.set_plan_air(s, fd)
        t, i = 0, 0
        while t < ntr:                                   # whole transfers: 1, 3, 2 per submit
            n = min((1, 3, 2)[i % 3], ntr - t)
            _submit(ctx, "real", x[:, t * T:(t + n) * T], i % 2 == 1)
            t += n
            i += 1
        ctx.sync()
        got = ctx.drain()
    model, _ = emission_model(oracle, want, _group_cuts(2, T, K, nout))
    assert_emission_order(got, model)
    assert len(model) >= len(plans)


@pytest.mark.parametrize("case", ["first", "first-sort", "last"])
def test_emission_group_boundary_on_a_completion_sample(native, oracle, monkeypatch, case):
    """Group boundaries put exactly on a frame's completion sample.  'first': a group starts on it, and a frame of a
    higher-numbered channel of the same stream completed earlier, in the preceding group — the frame belongs to its
    group (upper_bound on the group starts; '-sort' takes the consumer's comparison sort instead of the bucket pass).
    'last': a group ends on it, and a frame of a lower-numbered channel completes later, in the following group."""
    if case.endswith("sort"):
        monkeypatch.setenv("ACB_CONSUMER_SORT", "1")
    K = 160
    iq, plans = _cs16_streams(oracle, K, 0.3, seed=404)
    want = _expected_cs16(oracle, iq, K, plans, False)
    nout = want[0].shape[1]
    model, _ = emission_model(oracle, want, [0], positions=True)
    fr = [(s, t[0], p) for s, t, _, _, p in model]
    period = None
    for s, ca, pa in sorted(fr, key=lambda f: f[2]):
        if case == "last":
            if any(sb == s and cb < ca and pa < pb <= 2 * pa + 1 for sb, cb, pb in fr):
                period = pa + 1
        elif pa > 0 and any(sb == s and cb > ca and pb < pa for sb, cb, pb in fr):
            period = pa
        if period:
            break
    assert period and period < nout, fr
    with api.Context(K, len(plans), NCH, nout // 1024 + 1, flags=FLAG_CS16) as ctx:
        ctx.set_emission_groups(1, period)
        for s, (fd, fc, var) in enumerate(plans):
            ctx.set_plan_cs16(s, fd, var)
        assert _submit(ctx, "cs16", iq, False) == nout
        ctx.sync()
        got = ctx.drain()
    model, _ = emission_model(oracle, want, _group_cuts(1, period, K, nout), positions=True)
    assert_emission_order(got, model)


@pytest.mark.parametrize("kind", ["cs16", "real"])
def test_submit_boundary_inside_a_group_cuts_it(native, oracle, kind):
    """A submit that ends inside an emission group splits it: the frames of each submit are queued when it is collected,
    so the order is the model's with every submit boundary as an extra group boundary (include/acars_b200.h)."""
    if kind == "cs16":
        K = 160
        xs, plans = _cs16_streams(oracle, K, 0.3, seed=505)
        want = _expected_cs16(oracle, xs, K, plans, True)
        unit, period = 1, 1024
    else:
        xs, plans, K = _real_streams(oracle, 2500000, 0.3, seed=506)
        want = _expected_real(oracle, xs, K, plans, True)
        unit, period = 2, 65536
    nout = want[0].shape[1]
    with api.Context(K, len(plans), NCH, nout // 1024 + 2, flags=(FLAG_CS16 if kind == "cs16" else FLAG_REAL) | FAST) as ctx:
        ctx.set_emission_groups(unit, period)
        for s, p in enumerate(plans):
            if kind == "cs16":
                ctx.set_plan_cs16(s, p[0], p[2])
            else:
                ctx.set_plan_air(s, p[0])
        got, cuts = _run(ctx, kind, xs, _ragged_sizes(K, xs.shape[1], 17), want)
    groups = _group_cuts(unit, period, K, nout)
    assert set(cuts) - set(groups)                                 # some submit did end inside a group
    model, _ = emission_model(oracle, want, sorted(set(groups) | set(cuts)))
    assert_emission_order(got, model)
