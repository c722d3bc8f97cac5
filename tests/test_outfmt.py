"""SURVEY §8 f3 — the product's own message formatter (acarsdec_b200/csrc/outfmt.c: outputmsg's field split, label.c's
OOOI rules, the text / one-line / JSON formats and the three UDP payloads) against the reference's output.c / label.c /
netout.c / cJSON.c compiled in place and fed the same blocks (oracle/_ref/ref_outfmt, built by oracle/Makefile from
oracle/ref_output_harness.c).  Byte for byte, over crafted blocks for every label rule and a few thousand random ones."""
import struct
import subprocess

import numpy as np
import pytest

import refs
from acarsdec_b200 import api

NET = {api.FMT_NET_PP: "N", api.FMT_NET_NATIVE: "n", api.FMT_NET_JSON: "j"}


def _block(mode=b"2", addr=b".N123AB", ack=b"\x15", label=b"H1", bid=b"3", text=b"", no=b"M01A", fid=b"XX1234", end=b"\x03", stx=b"\x02"):
    body = (no + fid if bid[:1].isdigit() else b"") + text
    return mode + addr + ack + label + bid + stx + body + end


def _records(blocks):
    """[(chn, freq_hz, txt bytes, lvl, err, sec, usec)] -> the harness's input and the Msg list for the product."""
    raw, msgs = b"", []
    for chn, fr, txt, lvl, err, sec, usec in blocks:
        raw += struct.pack("<iiiif4xqq256s", chn, fr, len(txt), err, lvl, sec, usec, txt.ljust(256, b"\0"))
        m = api.Msg()
        m.chn, m.len, m.err, m.lvl = chn, len(txt), err, lvl
        m.txt[:len(txt)] = txt
        msgs.append(m)
    return raw, msgs


@pytest.fixture()
def ref(request):
    """The reference's programs (refs.RefPrograms) as recorded for this test."""
    with refs.recorded(request, refs.RefPrograms) as r:
        yield r


def _reference(ref, raw, outtype, net, inmode, airflt, emptymsg, labels, station):
    return ref.outfmt(raw, str(outtype), net, str(inmode), str(int(airflt)), str(int(emptymsg)), labels or "-", station or "-")


def _compare(ref, blocks, *, inmode=3, airflt=False, emptymsg=False, labels=None, station="STA1"):
    raw, msgs = _records(blocks)
    n = 0
    for fmt in (api.FMT_FULL, api.FMT_ONELINE, api.FMT_JSON, api.FMT_NET_PP, api.FMT_NET_NATIVE, api.FMT_NET_JSON):
        want = _reference(ref, raw, fmt if fmt in (1, 2, 4) else 0, NET.get(fmt, "-"), inmode, airflt, emptymsg, labels, station)
        assert len(want) == len(msgs)
        for i, (b, m) in enumerate(zip(blocks, msgs)):
            got = api.format_msg(m, fmt, tv_sec=b[5], tv_usec=b[6], freq_hz=b[1], inmode=inmode, airflt=airflt, emptymsg=emptymsg,
                                 labels=labels, station_id=station)
            if fmt == api.FMT_JSON and got is not None:
                got += b"\n"                                           # outputmsg prints the JSON buffer and a newline
            assert got == want[i], (fmt, i, b[2], got, want[i])
            n += got is not None
    return n


T0 = 1700000000

# one text per OOOI rule of label.c that satisfies it, and a near miss that must not
RULE_TEXTS = {
    b"Q1": b"EDDF1234123512361237    KJFKREST", b"Q2": b"EDDF1234", b"QA": b"EDDF1234", b"QB": b"EDDF1234", b"QC": b"EDDF1234",
    b"QD": b"EDDF1234", b"QE": b"EDDF1234KJFK", b"QF": b"EDDF1234KJFK", b"QG": b"EDDF12341235", b"QH": b"EDDF1234",
    b"QK": b"EDDF1234KJFK", b"QL": b"KJFK00001234 EDDFxx", b"QM": b"KJFK0000EDDF", b"QN": b"0000KJFK1234", b"QP": b"EDDFKJFK1234",
    b"QQ": b"EDDFKJFK1234", b"QR": b"EDDFKJFK1234", b"QS": b"EDDFKJFK1234", b"QT": b"EDDFKJFK12341235",
    b"10": b"ARR01ABCDEFGKJFK1234", b"11": b"0123456789ABC/DS KJFK/ETA 1234", b"12": b"EDDF,KJFK", b"15": b"FST01EDDFKJFK",
    b"17": b"ETA 1234,EDDF,KJFK", b"1G": b"EDDF,KJFK", b"20": b"RST0123456789012345678EDDFKJFK", b"21": b"ABCDEF,EDDF,KJFK",
    b"26": b"VER/077\nSCH/AB123/EDDF/KJFK/x\nETA/1234", b"RB": b"VER/077\nSCH/AB123/EDDF/KJFK", b"2N": b"TKO01ABCDEF/01234567EDDFKJFK",
    b"2Z": b"KJFK", b"33": b",0123456789012345678,EDDF,KJFK", b"39": b"GTA010123456789/01234567EDDFKJFK",
    b"44": b"00POS02,N12345W123456,KJFK,1234,5678,9012,3456", b"45": b"AKJFK", b"80": b"012345/DESTxKJFK", b"83": b"EDDF,KJFK",
    b"8D": b"ABCD,012345678901234567890123456789,EDDF,KJFK", b"8E": b"KJFK,1234", b"8S": b"KJFK,1234",
}


def test_every_label_rule_and_its_near_miss(ref):
    blocks = []
    pad = b" " * 24                       # long enough that no rule reads past the text (undefined in the reference)
    for i, (lab, txt) in enumerate(sorted(RULE_TEXTS.items())):
        for bid in (b"5", b"A"):           # downlink (message number + flight id precede the text) and uplink
            blocks.append((i % 8, 131525000 + 25000 * (i % 5), _block(label=lab, bid=bid, text=txt + pad), -18.5 + i, i % 4, T0 + i, 1000 * i))
        miss = bytearray(txt + pad)
        miss[min(4, len(txt) - 1)] ^= 0x01   # disturb a byte most rules guard on or copy
        blocks.append((1, 131725000, _block(label=lab, bid=b"B", text=bytes(miss)), -7.25, 0, T0, 999999))
    assert _compare(ref, blocks) > 500


def test_header_variants_filters_and_escapes(ref):
    b = []
    b.append((0, 131525000, _block(text=b'HELLO "WORLD" \\ back\r\nLINE2\ttab\x01\x1f', end=b"\x17"), -12.34, 1, T0, 123456))   # JSON escapes, ETB
    b.append((3, 131825000, _block(ack=b"A", label=b"_\x7f", bid=b"\0", stx=b"\x03", text=b"", no=b"", fid=b""), -3.0, 0, T0, 0))      # squitter, empty
    b.append((7, 136975000, _block(addr=b"..ABCDE", ack=b"5", label=b"5Z", bid=b"7", text=b"short"), 0.04, 3, T0 + 86400 * 400, 5))
    b.append((2, 131450000, _block(mode=b"X", addr=b".......", label=b"SA", bid=b"9", no=b"S1", fid=b"", text=b""), -99.94, 0, 0, 0))  # tv == 0: no date; short body
    b.append((1, 131550000, _block(bid=b"Z", text=b"x" * 200), 9.96, 0, 1, 1))                                                        # long uplink text
    b.append((4, 131725000, _block(label=b"H1", bid=b"2", text=b"A\nB\rC" + b"y" * 80), -20.05, 2, T0, 500))                          # one-line cut at 59
    for inmode in (0, 2, 3, 5):
        assert _compare(ref, b, inmode=inmode) > 20
    assert _compare(ref, b, airflt=True) > 10                     # -A: uplinks dropped
    assert _compare(ref, b, emptymsg=True) > 10                   # -e: empty messages dropped
    assert _compare(ref, b, labels="H1:5Z") > 5                   # -i H1:5Z
    assert _compare(ref, b, station="") > 20                      # no station id: no "station_id" key


def test_random_blocks(ref):
    rng = np.random.default_rng(12)
    printable = np.frombuffer(bytes(range(32, 127)), dtype=np.uint8)
    free_labels = [b"H1", b"5Z", b"SA", b"_d", b"B9", b"A0", b"C1", b"Q0", b"QX", b"30", b"4T"]        # no OOOI rule: any text length is defined
    blocks = []
    for i in range(1500):
        ln = int(rng.integers(0, 200))
        txt = bytes(rng.choice(printable, ln))
        if rng.random() < 0.1 and ln:
            j = int(rng.integers(0, ln))
            txt = txt[:j] + bytes([int(rng.choice([10, 13, 9, 34, 92, 1, 27]))]) + txt[j + 1:]
        bid = bytes([int(rng.choice(list(b"0123456789ABCXYZ")))])
        blocks.append((int(rng.integers(0, 16)), int(rng.integers(118000, 137000)) * 1000,
                       _block(mode=bytes([int(rng.choice(list(b"2XQ")))]), addr=bytes(rng.choice(list(b".ABC123-"), 7).astype(np.uint8)),
                              ack=bytes([int(rng.choice([0x15, 65, 52]))]), label=free_labels[int(rng.integers(len(free_labels)))], bid=bid,
                              text=txt, no=bytes(rng.choice(printable, 4)), fid=bytes(rng.choice(printable, 6)),
                              end=bytes([int(rng.choice([3, 0x17]))])),
                       float(np.float32(rng.uniform(-45, 5))), int(rng.integers(0, 4)), T0 + int(rng.integers(0, 10**7)), int(rng.integers(0, 10**6))))
    assert _compare(ref, blocks) > 8000


def test_field_split_api():
    m = api.Msg()
    txt = _block(text=b"EDDF1234", label=b"Q2", bid=b"4")
    m.chn, m.len = 2, len(txt)
    m.txt[:len(txt)] = txt
    f = api.msg_fields(m)
    assert (f.mode, f.ack, f.bid, f.label, f.addr, f.no, f.fid) == (b"2", b"!", b"4", b"Q2", b"N123AB", b"M01A", b"XX1234")
    assert f.downlink == 1 and bytes(m.txt[f.txt_off:f.txt_off + f.txt_len]) == b"EDDF1234"
    assert f.has_oooi == 1 and (f.sa, f.eta, f.da) == (b"EDDF", b"1234", b"")
    m.len = 5
    assert api.msg_fields(m) is None
    with pytest.raises(api.AcbError):
        api.format_msg(m, api.FMT_JSON)


@pytest.mark.parametrize("outtype,fmt", [("2", api.FMT_FULL), ("1", api.FMT_ONELINE), ("4", api.FMT_JSON)])
def test_formatter_reproduces_the_reference_programs_stdout(oracle, ref, outtype, fmt):
    """End to end on the CPU: the unmodified reference program (its own DSP and its own output.c) on a synthetic capture,
    against the same capture decoded by the restatement and printed by the product's formatter — same stdout, time stamps
    masked (the program stamps wall-clock time)."""
    from acarsdec_b200 import synth
    K, fm = 160, (131.525, 131.725, 131.825, 131.450, 131.550)
    fd, _, fc = oracle.plan(K, fm)
    plan = synth.make_plan(K, fm, fc, seconds=1.5, seed=123, text_len=(10, 120), msgs_per_chan_per_sec=3.0)
    nblk = synth.blocks_for_seconds(K, 1.5)
    iq = synth.render_blocks(plan, 0, nblk)
    want = ref.acarsdec_rtl(iq, "-o", outtype, "-m", str(K), "-i", "STA1", "-r", "0", *[str(f) for f in fm])
    o = refs.OracleStream(oracle, K, oracle.wf(K, fm))
    o.blocks(iq.reshape(-1))
    mine = b""
    for om in o.msgs():
        m = api.Msg()
        m.chn, m.len, m.err, m.lvl = om.chn, om.len, om.err, om.lvl
        m.txt[:om.len] = om.txt[:om.len]
        # rtl.c:255 keeps the frequency as int <- float <- unsigned: what channel[].Fr holds and the formats print
        s = api.format_msg(m, fmt, tv_sec=T0, tv_usec=123000, freq_hz=api.load().acb_stored_fr(fd[m.chn]), inmode=3, station_id="STA1")
        mine += s + (b"\n" if fmt == api.FMT_JSON else b"")
    assert refs.mask_time(mine).count(b"<time>") >= 8 and want == refs.mask_time(mine)


def _flight_sequence():
    """Downlinks of a handful of aircraft over 25 minutes: route information arriving in pieces, flight ids changing, one
    aircraft falling silent for longer than the table keeps it (600 s) and coming back."""
    rng = np.random.default_rng(5)
    tails = [b".N123AB", b"..G-ABC", b".D-AIXY", b"JA8089.", b".F-GZZZ"]
    fids = [b"XX1234", b"BA0042", b"LH0400", b"JL0005", b"AF0011"]
    texts = [(b"QA", b"EDDF1234"), (b"Q2", b"KJFK0915"), (b"12", b"EDDF,KJFK rest"), (b"H1", b"no route information in here"), (b"2Z", b"RJTT"),
             (b"QE", b"LFPG0830EGLL"), (b"10", b"ARR01ABCDEFGEGLL1015"), (b"5Z", b"")]
    blocks, t = [], T0
    for i in range(90):
        a = int(rng.integers(len(tails))) if i not in range(30, 60) else int(rng.integers(1, len(tails)))      # tail 0 silent for a while
        lab, txt = texts[int(rng.integers(len(texts)))]
        t += int(rng.integers(1, 40)) if i != 45 else 700
        fid = fids[a] if rng.random() < 0.8 else fids[(a + 1) % len(fids)]
        blocks.append((int(rng.integers(0, 8)), 131525000, _block(addr=tails[a], label=lab, bid=bytes([48 + i % 10]), text=txt + b" " * 24, fid=fid,
                                                                   no=b"M%02dA" % (i % 100)), -10.0, 0, t, int(rng.integers(0, 10**6))))
    return blocks


def test_route_json_and_monitor_follow_the_reference_flight_table(ref):
    blocks = _flight_sequence()
    raw, msgs = _records(blocks)
    want = _reference(ref, raw, 5, "-", 3, False, False, None, "STA1")              # -o 5: route JSON
    fl = api.Flights()
    got = [fl.route_json(m, tv_sec=b[5], tv_usec=b[6], station_id="STA1") for b, m in zip(blocks, msgs)]
    got = [g + b"\n" if g else None for g in got]
    assert got == want and sum(g is not None for g in got) >= 4
    # an uplink or a squitter never enters the table (and the reference reads an unset pointer for them in this mode)
    up = api.Msg()
    txt = _block(bid=b"A", label=b"12", text=b"EDDF,KJFK")
    up.len = len(txt)
    up.txt[:len(txt)] = txt
    assert fl.route_json(up, tv_sec=T0) is None
    fl.close()
    mixed = blocks[:40] + [(2, 131525000, _block(bid=b"B", label=b"H1", text=b"uplink text"), -5.0, 0, blocks[39][5] + 5, 0)] + blocks[40:]
    raw, msgs = _records(mixed)
    want = _reference(ref, raw, 3, "-", 3, False, False, None, "STA1")              # -o 3: the monitor screen after every block
    fl = api.Flights()
    got = [fl.monitor(m, 16, tv_sec=b[5], tv_usec=b[6], station_id="STA1") for b, m in zip(mixed, msgs)]
    assert got == want and all(g is not None for g in got)


def test_formatter_fuzz_under_sanitizers(tmp_path):
    """Random and malformed blocks (any bytes, lengths outside 13..248, tiny output buffers, unknown formats) through every
    entry point of outfmt.c, compiled with AddressSanitizer and UBSan."""
    import shutil
    cc = shutil.which("gcc")
    exe = tmp_path / "fuzz_outfmt"
    root = refs.ORACLE_DIR.parent
    r = subprocess.run([cc, "-O1", "-g", "-fsanitize=address,undefined", "-fno-sanitize-recover=undefined", "-I", str(root / "include"), "-o", str(exe),
                        str(root / "tests" / "host" / "fuzz_outfmt.c"), str(root / "acarsdec_b200" / "csrc" / "outfmt.c")], capture_output=True, text=True)
    if r.returncode != 0 and "sanitize" in r.stderr:
        pytest.skip("this gcc has no sanitizer runtime")
    assert r.returncode == 0, r.stderr
    r = subprocess.run([str(exe)], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and r.stdout.startswith("fuzz ok"), r.stderr[-2000:]
