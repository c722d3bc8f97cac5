"""The exact IQ channelizers (k_channelize<IN_U8IQ>, k_channelize<IN_CS16IQ>) reproduce the reference's rounding
only while ptxas keeps every product separately rounded.  cmac2 writes each product as FFMA2(x, w, nz) with nz = -0.0f
passed as a kernel argument: ptxas turns an FFMA2 with a literal -0 addend back into FMUL2 and then contracts
FMUL2 -> FADD2 into FFMA2, even under -fmad=false, which skips a rounding.  The fixtures might not hit an input where
that shows, so these tests read the built library's SASS: every FFMA2 of those kernels must take the kernel argument nz
as its addend, and no FMUL2 may appear.  CPU only (cuobjdump)."""
import re
import shutil
import subprocess
from pathlib import Path

import pytest

KERNELS = {"u8": "_ZN3acb12k_channelizeILi0EEEvPKhmS2_Pfiiiimf", "cs16": "_ZN3acb12k_channelizeILi2EEEvPKhmS2_Pfiiiimf"}


def _cuobjdump() -> str:
    from acarsdec_b200 import build
    cand = Path(build.nvcc()).with_name("cuobjdump")
    if cand.exists():
        return str(cand)
    found = shutil.which("cuobjdump")
    assert found, "cuobjdump not found next to nvcc"
    return found


@pytest.fixture(scope="module")
def dumps(native):
    from acarsdec_b200 import build
    tool = _cuobjdump()
    sass = subprocess.run([tool, "-sass", str(build.LIB)], capture_output=True, text=True, check=True).stdout
    elf = subprocess.run([tool, "-elf", str(build.LIB)], capture_output=True, text=True, check=True).stdout
    return sass, elf


def _function(text: str, header: str, name: str) -> str:
    """The section of a cuobjdump listing that belongs to `name` (`header` introduces each section)."""
    parts = re.split(r"^\s*" + re.escape(header) + r"\s*(\S+)\s*$", text, flags=re.M)
    bodies = [parts[i + 1] for i in range(1, len(parts) - 1, 2) if parts[i] == name]
    assert len(bodies) == 1, f"{name}: {len(bodies)} sections in the listing"
    return bodies[0]


def _nz_offset(elf: str, name: str) -> int:
    """Constant-bank address of the kernel's last parameter, nz (4 bytes): parameter bank base + size - 4."""
    m = re.search(r"^\.nv\.info\." + re.escape(name) + r"\s*$(.*?)(?=^\.\S)", elf, flags=re.M | re.S)
    assert m, f"{name}: no .nv.info section"
    info = m.group(1)
    size = re.search(r"EIATTR_CBANK_PARAM_SIZE\s+Format:\s+EIFMT_HVAL\s+Value:\s+(0x[0-9a-f]+)", info)
    base = re.search(r"EIATTR_PARAM_CBANK\s+Format:\s+EIFMT_SVAL\s+Value:\s+0x[0-9a-f]+\s+(0x[0-9a-f]+)", info)
    assert size and base, f"{name}: parameter bank not described"
    return (int(base.group(1), 16) & 0xFFFF) + int(size.group(1), 16) - 4


def _instructions(body: str):
    """(opcode, operand text) in program order, predicates dropped."""
    out = []
    for m in re.finditer(r"/\*[0-9a-f]{4,}\*/\s+(?:@!?U?P\w+\s+)?([A-Z][A-Z0-9_.]*)\s*([^;]*);", body):
        out.append((m.group(1), m.group(2).strip()))
    return out


@pytest.mark.parametrize("kind", sorted(KERNELS))
def test_exact_channelizer_products_rounded(dumps, kind):
    sass, elf = dumps
    name = KERNELS[kind]
    body = _function(sass, "Function :", name)
    nz = _nz_offset(elf, name)
    ins = _instructions(body)
    ops = [op.split(".")[0] for op, _ in ins]
    assert "FMUL2" not in ops, f"{kind}: FMUL2 in the exact channelizer (products would be contracted)"
    assert ops.count("FFMA2") >= 64, f"{kind}: expected the FFMA2 products of cmac2, found {ops.count('FFMA2')}"
    last_def = {}                      # register -> (opcode, operands) of its latest write in program order
    for op, args in ins:
        base = op.split(".")[0]
        if base == "FFMA2":
            addend = args.split(",")[-1].strip()
            reg = re.match(r"-?\|?(U?R\d+)", addend)
            assert reg and not addend.startswith("-"), f"{kind}: FFMA2 addend {addend!r} is not the run-time -0"
            d = last_def.get(reg.group(1))
            assert d is not None and d[0].startswith("LDC") and f"c[0x0][{nz:#x}]" in d[1], \
                f"{kind}: FFMA2 addend {reg.group(1)} was last written by {d}, not by the load of nz (c[0x0][{nz:#x}])"
        dst = re.match(r"(U?R\d+)\b", args)
        if dst and not base.startswith(("ST", "RED", "ATOM", "BRA", "BSSY", "BSYNC")):
            prefix = "UR" if dst.group(1).startswith("UR") else "R"
            n = int(dst.group(1)[len(prefix):])
            width = 4 if ".128" in op else 2 if (".64" in op or base in ("FFMA2", "FADD2")) else 1
            for k in range(width):
                last_def[prefix + str(n + k)] = (op, args)
