"""The reference-API shim (libacarsdec_compat.so): ABI mirror, symbols, and — on the GPU — the
drop-in behaviour: demodMSK/decodeAcars/initRtl driven by C hosts, including the reference's own
unmodified acarsdec.c linked against the shim (oracle/_ref/acarsdec_b200)."""
import ctypes as C
import os
import re
import subprocess
from pathlib import Path

import numpy as np
import pytest

import refs
from acarsdec_b200 import build, synth
from common import GOLDEN, load_testwav, msg_tuple, msg_tuple_from_json

ROOT = Path(__file__).resolve().parent.parent
PKG = ROOT / "acarsdec_b200"
REFBIN = ROOT / "oracle" / "_ref"


@pytest.fixture()
def refprog(request):
    with refs.recorded(request, refs.RefPrograms) as r:
        yield r


def test_abi_mirror_matches_reference_header(tmp_path, refprog):
    exe = tmp_path / "abi_layout"
    subprocess.run(["gcc", "-DWITH_RTL", '-DHDR="acarsdec_compat.h"', "-I", str(ROOT / "include"), "-o", str(exe),
                    str(ROOT / "oracle" / "abi_layout.c")], check=True)
    mine = subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout
    assert mine == refprog.abi_layout()


def _host(tmp_path) -> Path:
    build.build()
    exe = tmp_path / "wavhost"
    subprocess.run(["gcc", "-O1", "-std=gnu11", "-DWITH_RTL", "-I", str(ROOT / "include"), "-o", str(exe),
                    str(ROOT / "tests" / "host" / "wavhost.c"), "-L", str(PKG), "-lacarsdec_compat", "-lacars_b200",
                    f"-Wl,-rpath,{PKG}", "-lpthread", "-lm"], check=True)
    return exe


def test_compat_library_exports_reference_symbols(tmp_path):
    build.build()
    out = subprocess.run(["nm", "-D", "--defined-only", str(PKG / "libacarsdec_compat.so")], capture_output=True, text=True, check=True).stdout
    defined = set(re.findall(r" T (\w+)", out))
    hdr = (ROOT / "include" / "acarsdec_compat.h").read_text()
    tail = re.sub(r"/\*.*?\*/", "", hdr[hdr.index('extern "C" {'):], flags=re.S)
    declared = set(re.findall(r"^\s*(?:int|void)\s+(\w+)\s*\(", tail, flags=re.M))
    common = {"initMsk", "demodMSK", "initAcars", "decodeAcars", "deinitAcars"}
    rtl = {"initRtl", "runRtlSample", "runRtlCancel", "runRtlClose"}
    air = {"initAirspy", "runAirspySample"}
    soapy = {"initSoapy", "soapySetAntenna", "runSoapySample", "runSoapyClose"}
    sdrplay = {"initSdrplay", "runSdrplaySample"}
    assert declared == common | rtl | air | soapy | sdrplay
    assert common | rtl <= defined
    out = subprocess.run(["nm", "-D", "--defined-only", str(PKG / "libacarsdec_compat_air.so")], capture_output=True, text=True, check=True).stdout
    assert common | air <= set(re.findall(r" T (\w+)", out))
    for lib, want in (("libacarsdec_compat_soapy.so", soapy), ("libacarsdec_compat_sdrplay.so", sdrplay)):
        out = subprocess.run(["nm", "-D", "--defined-only", str(PKG / lib)], capture_output=True, text=True, check=True).stdout
        assert common | want <= set(re.findall(r" T (\w+)", out))
    # and it links into a host that supplies acarsdec.c's globals
    assert _host(tmp_path).exists()


def test_host_decodeAcars_matches_oracle(tmp_path, oracle):
    """decodeAcars() of the shim (host build of frame_sm.h + block FEC) vs the restatement."""
    exe = _host(tmp_path)
    rng = np.random.default_rng(31)
    stream = bytearray()
    for i in range(120):
        fr = bytearray(synth.frame_bytes(synth.random_text(rng, int(rng.integers(0, 200))), prekey=0, etb=bool(i & 1))[2:])
        if i % 4 == 1:
            fr[5 + int(rng.integers(0, 8))] ^= 1 << int(rng.integers(0, 8))       # one parity error: repaired
        if i % 4 == 2 and len(fr) > 30:
            fr[10] ^= 0x03                                                       # double error in one byte
        if i % 7 == 3:
            for _ in range(6):
                fr[int(rng.integers(3, len(fr)))] ^= 1 << int(rng.integers(0, 8))
        stream += fr + bytes(rng.integers(0, 256, size=int(rng.integers(0, 9)), dtype=np.uint8))
    p = tmp_path / "bytes.bin"
    p.write_bytes(bytes(stream))
    out = subprocess.run([str(exe), "bytes", str(p)], capture_output=True, text=True, check=True).stdout.split("\n")
    got = [(int(a), int(b), int(c), bytes.fromhex(t), bytes.fromhex(crc)) for a, b, c, _, crc, t in (l.split() for l in out if l)]
    ch = oracle.new_chan(0)
    sink = refs.Sink()
    ch.MskLvlSum, ch.MskBitCount = 4.0, 1
    want = []
    for byte in stream:
        ch.outbits = byte
        ch.MskLvlSum += 1.0
        ch.MskBitCount += 8
        oracle.lib.orc_decode_byte(C.byref(ch), C.byref(sink.c))
        for m in sink.msgs():
            f = oracle.fec(m)
            if f is not None:
                want.append(f.as_tuple())
        sink.c.nmsg = 0
    assert got == want and len(got) > 60 and any(g[2] > 0 for g in got)


@pytest.mark.gpu
def test_demodMSK_shim_on_testwav(tmp_path):
    """BASELINE config 1 through the reference API: initMsk/initAcars/demodMSK per channel per chunk
    exactly like soundfile.c, state carried in channel_t across calls -> the 7 known messages."""
    exe = _host(tmp_path)
    x, exp = load_testwav()
    p = tmp_path / "testwav.f32"
    x.astype("<f4").tofile(p)
    want = [msg_tuple_from_json(j) for j in exp["messages"]]
    for chunk in (4096, 1000):
        out = subprocess.run([str(exe), "audio", str(p), "4", str(chunk)], capture_output=True, text=True, check=True).stdout
        got = []
        for l in out.strip().split("\n"):
            chn, ln, err, lvl, crc, txt = l.split()
            got.append((int(chn), int(ln), int(err), bytes.fromhex(txt), bytes.fromhex(crc), int(lvl, 16)))
        # emission order depends on the chunking (soundfile.c interleaves channels per chunk)
        assert sorted(got) == sorted(want), chunk
        if chunk == 4096:
            assert got == want


def _strip_time(s: str) -> str:
    s = re.sub(r'"timestamp":[0-9.e+]+', '"timestamp":<time>', s)          # JSON wire format (output.c:244-245)
    return re.sub(r"\d\d/\d\d/\d{4} \d\d:\d\d:\d\d\.\d{3}", "<time>", s)


@pytest.mark.gpu
@pytest.mark.skipif(not (REFBIN / "acarsdec_b200").exists() or not (REFBIN / "acarsdec_ref").exists(),
                    reason="oracle/_ref program builds absent")
@pytest.mark.parametrize("K,outtype", [(160, "2"), (192, "1"), (160, "4")])      # full text, one line, JSON
def test_unmodified_acarsdec_main_links_against_shim(tmp_path, K, outtype):
    """The drop-in claim: the reference's own acarsdec.c/output.c/label.c (unmodified, compiled in
    place) linked against libacarsdec_compat + libacars_b200 prints the same decoded messages as the
    same program linked against its own rtl.c/msk.c/acars.c, on the same IQ capture."""
    orc = refs.OracleLib()
    fm = (131.525, 131.725, 131.825, 131.450, 131.550)
    _, _, fc = orc.plan(K, fm)
    plan = synth.make_plan(K, fm, fc, seconds=1.8, seed=77, text_len=(10, 120), msgs_per_chan_per_sec=3.0)
    nblk = synth.blocks_for_seconds(K, 1.8)
    cap = tmp_path / "cap.iq"
    synth.render_blocks(plan, 0, nblk).tofile(cap)
    args = ["-o", outtype, "-m", str(K), "-r"]
    freqs = [str(f) for f in fm]
    env = dict(os.environ, ACARSDEC_STUB_IQ=str(cap))
    ref = subprocess.run([str(REFBIN / "acarsdec_ref"), *args, "0", *freqs], env=env, capture_output=True, text=True, timeout=120)
    env2 = dict(os.environ, ACARSDEC_B200_BLOCKS="4")
    mine = subprocess.run([str(REFBIN / "acarsdec_b200"), *args, str(cap), *freqs], env=env2, capture_output=True, text=True, timeout=120)
    assert mine.returncode == 0, mine.stderr
    a, b = _strip_time(ref.stdout), _strip_time(mine.stdout)
    assert a.count("<time>") >= 8
    assert a == b


def _run_with_udp_sink(make_cmd, env):
    """Run make_cmd(port) while listening on a free UDP port of 127.0.0.1; returns (returncode, stderr, [datagram, ...])."""
    import socket, threading
    sock = socket.socket(socket.AF_INET, socket.SOCK_DGRAM)
    sock.bind(("127.0.0.1", 0))
    cmd = make_cmd(sock.getsockname()[1])
    sock.settimeout(0.2)
    got, stop = [], threading.Event()

    def rx():
        while True:
            try:
                got.append(sock.recv(65536))
            except socket.timeout:
                if stop.is_set():
                    return

    th = threading.Thread(target=rx)
    th.start()
    try:
        r = subprocess.run(cmd, env=env, capture_output=True, text=True, timeout=120)
    finally:
        stop.set()
        th.join()
        sock.close()
    return r.returncode, r.stderr, got


@pytest.mark.gpu
@pytest.mark.skipif(not (REFBIN / "acarsdec_b200").exists() or not (REFBIN / "acarsdec_ref").exists(),
                    reason="oracle/_ref program builds absent")
@pytest.mark.parametrize("opt", ["-n", "-N", "-j"])          # netout.c: native "sv" datagrams, planeplotter, JSON
def test_unmodified_acarsdec_main_udp_sinks(tmp_path, opt):
    """The UDP wire formats (netout.c:100-153, fed by outputmsg output.c:486-706) of the unmodified program linked against
    the shim: the same datagrams, in the same order, as the program linked against its own DSP."""
    K = 160
    orc = refs.OracleLib()
    fm = (131.525, 131.725, 131.825, 131.450, 131.550)
    _, _, fc = orc.plan(K, fm)
    plan = synth.make_plan(K, fm, fc, seconds=1.2, seed=91, text_len=(10, 120), msgs_per_chan_per_sec=3.0)
    cap = tmp_path / "cap.iq"
    synth.render_blocks(plan, 0, synth.blocks_for_seconds(K, 1.2)).tofile(cap)
    freqs = [str(f) for f in fm]
    args = lambda port: ["-o", "0", opt, f"127.0.0.1:{port}", "-m", str(K), "-r"]
    rc, err, ref = _run_with_udp_sink(lambda port: [str(REFBIN / "acarsdec_ref"), *args(port), "0", *freqs], dict(os.environ, ACARSDEC_STUB_IQ=str(cap)))
    assert rc == 0, err
    rc, err, mine = _run_with_udp_sink(lambda port: [str(REFBIN / "acarsdec_b200"), *args(port), str(cap), *freqs], dict(os.environ, ACARSDEC_B200_BLOCKS="4"))
    assert rc == 0, err
    strip = lambda d: re.sub(r"\d\d/\d\d/\d{4} \d\d:\d\d:\d\d", "<time>", _strip_time(d.decode("latin-1")))
    a, b = [strip(d) for d in ref], [strip(d) for d in mine]
    assert len(a) >= 6 and a == b


@pytest.mark.gpu
def test_rtl_trio_through_test_host(tmp_path, oracle):
    exe = _host(tmp_path)
    K, fm = 160, (131.525, 131.725, 131.825)
    _, _, fc = oracle.plan(K, fm)
    plan = synth.make_plan(K, fm, fc, seconds=1.0, seed=5, text_len=(10, 50))
    iq = synth.render_blocks(plan, 0, 13)
    cap = tmp_path / "cap.iq"
    iq.tofile(cap)
    # a trailing partial block must be dropped with the reference's warning (rtl.c:322-326)
    with open(cap, "ab") as f:
        f.write(bytes(1000))
    out = subprocess.run([str(exe), "rtl", str(K), str(cap), *[str(f) for f in fm]], capture_output=True, text=True, check=True,
                         env=dict(os.environ, ACARSDEC_B200_BLOCKS="5"))
    assert "partial read" in out.stderr
    got = []
    for l in out.stdout.strip().split("\n"):
        chn, ln, err, lvl, crc, txt = l.split()
        got.append((int(chn), int(ln), int(err), bytes.fromhex(txt), bytes.fromhex(crc), int(lvl, 16)))
    o = refs.OracleStream(oracle, K, oracle.wf(K, fm))
    o.blocks(iq)
    assert got == [msg_tuple(m) for m in o.msgs()] and len(got) >= 4


@pytest.mark.gpu
@pytest.mark.skipif(not (REFBIN / "acarsdec_b200_air").exists() or not (REFBIN / "acarsdec_ref_air").exists(),
                    reason="oracle/_ref Airspy program builds absent")
def test_unmodified_acarsdec_main_airspy_front_end(tmp_path):
    """Same drop-in check for the Airspy front-end (-DWITH_AIR hosts): unmodified acarsdec.c + the
    shim's initAirspy/runAirspySample vs unmodified acarsdec.c + air.c, same float32 capture."""
    orc = refs.OracleLib()
    rate, fm = 2500000, (131.525, 131.725, 131.825, 131.450)
    fd, fc, K = orc.air_plan(rate, fm)
    plan = synth.StreamPlan(K=K, freqs_hz=tuple(fd), fc_hz=fc, seed=19, noise_sigma=1.0)
    rng = np.random.default_rng(19)
    for ch in range(4):
        t = 0.01 + 0.04 * ch
        for _ in range(3):
            fr = synth.frame_bytes(synth.random_text(rng, int(rng.integers(10, 60))))
            plan.bursts.append(synth.Burst(chan=ch, t0=t, frame=fr, amp=float(rng.uniform(10, 25)), phase=float(rng.uniform(0, 6))))
            t += len(fr) * 8 / 2400 + 0.05
    cap = tmp_path / "cap.f32"
    synth.render_real(plan, 0, int(1.2 * rate)).tofile(cap)
    freqs = [str(f) for f in fm]
    env = dict(os.environ, ACARSDEC_STUB_AIR=str(cap), ACARSDEC_STUB_AIRRATE=str(rate))
    ref = subprocess.run([str(REFBIN / "acarsdec_ref_air"), "-o", "2", "-s", "0", *freqs], env=env, capture_output=True, text=True, timeout=120)
    env2 = dict(os.environ, ACARSDEC_B200_AIRRATE=str(rate))
    mine = subprocess.run([str(REFBIN / "acarsdec_b200_air"), "-o", "2", "-s", str(cap), *freqs], env=env2, capture_output=True, text=True, timeout=120)
    assert mine.returncode == 0, mine.stderr
    a, b = _strip_time(ref.stdout), _strip_time(mine.stdout)
    assert a.count("<time>") >= 10
    # the shim submits 8 transfers at a time and queues the frames per transfer, channel by channel, like
    # air.c:336 does: byte-identical output, order included
    assert a == b


def _cs16_capture(tmp_path, seed):
    """2 MS/s interleaved CS16 capture with 3 messages on each of 4 channels."""
    orc = refs.OracleLib()
    K, fm = 160, (131.525, 131.725, 131.825, 131.450)
    fd, _, fc = orc.plan(K, fm)
    plan = synth.StreamPlan(K=K, freqs_hz=tuple(fd), fc_hz=fc, seed=seed, noise_sigma=1.0)
    rng = np.random.default_rng(seed)
    for ch in range(4):
        t = 0.01 + 0.04 * ch
        for _ in range(3):
            fr = synth.frame_bytes(synth.random_text(rng, int(rng.integers(10, 60))))
            plan.bursts.append(synth.Burst(chan=ch, t0=t, frame=fr, amp=float(rng.uniform(10, 25)), phase=float(rng.uniform(0, 6))))
            t += len(fr) * 8 / 2400 + 0.05
    cap = tmp_path / "cap.cs16"
    synth.render_cs16(plan, 0, int(1.2 * K * 12500)).tofile(cap)
    return cap, [str(f) for f in fm]


def _same_messages_per_channel(a, b, nch=4):
    def blocks(s):
        return [blk for blk in s.split("\n[#") if blk.strip()]
    assert sorted(blocks(a)) == sorted(blocks(b))
    for ch in "1234"[:nch]:
        assert [x for x in blocks(a) if x.startswith(ch)] == [x for x in blocks(b) if x.startswith(ch)]


@pytest.mark.gpu
@pytest.mark.skipif(not (REFBIN / "acarsdec_b200_soapy").exists() or not (REFBIN / "acarsdec_ref_soapy").exists(),
                    reason="oracle/_ref SoapySDR program builds absent")
def test_unmodified_acarsdec_main_soapy_front_end(tmp_path):
    """-DWITH_SOAPY hosts: unmodified acarsdec.c + the shim's initSoapy/runSoapySample/runSoapyClose vs
    unmodified acarsdec.c + soapy.c over a file-replay SoapySDR stub, same CS16 capture."""
    cap, freqs = _cs16_capture(tmp_path, 23)
    ref = subprocess.run([str(REFBIN / "acarsdec_ref_soapy"), "-o", "2", "-d", str(cap), *freqs], capture_output=True, text=True, timeout=120)
    mine = subprocess.run([str(REFBIN / "acarsdec_b200_soapy"), "-o", "2", "-d", str(cap), *freqs], capture_output=True, text=True, timeout=120)
    assert mine.returncode == 0, mine.stderr
    a, b = _strip_time(ref.stdout), _strip_time(mine.stdout)
    assert a.count("<time>") >= 10
    _same_messages_per_channel(a, b)
    assert a == b            # emission order too: per full dm_buffer, channel by channel (soapy.c:247, sdrplay.c:229)


@pytest.mark.gpu
@pytest.mark.skipif(not (REFBIN / "acarsdec_b200_sdrplay").exists() or not (REFBIN / "acarsdec_ref_sdrplay").exists(),
                    reason="oracle/_ref SDRplay program builds absent")
def test_unmodified_acarsdec_main_sdrplay_front_end(tmp_path):
    """-DWITH_SDRPLAY hosts: the shim's initSdrplay/runSdrplaySample vs sdrplay.c fed planar packets by a
    file-replay mirsdrapi stub, same CS16 capture."""
    cap, freqs = _cs16_capture(tmp_path, 29)
    ref = subprocess.run([str(REFBIN / "acarsdec_ref_sdrplay"), "-o", "2", "-s", *freqs],
                         env=dict(os.environ, ACARSDEC_STUB_SDRPLAY=str(cap)), capture_output=True, text=True, timeout=120)
    mine = subprocess.run([str(REFBIN / "acarsdec_b200_sdrplay"), "-o", "2", "-s", *freqs],
                          env=dict(os.environ, ACARSDEC_B200_CAPTURE=str(cap)), capture_output=True, text=True, timeout=120)
    assert mine.returncode == 0, mine.stderr
    a, b = _strip_time(ref.stdout), _strip_time(mine.stdout)
    assert a.count("<time>") >= 10
    _same_messages_per_channel(a, b)
    assert a == b            # emission order too: per full dm_buffer, channel by channel (soapy.c:247, sdrplay.c:229)
