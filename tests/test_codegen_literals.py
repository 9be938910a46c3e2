"""Constants in generated code: every numeric type's edge values, written by the library's own code generator
(tools/aotgen.cc + codegen.cc, built as fuse_query_b200/build.py builds it), must read back with the intended bits
and compile for sm_100a.  Non-finite floats (±inf, NaN with its payload, an f32 literal that overflows to inf) are
the case %a cannot print as CUDA source."""
import os
import re
import struct
import subprocess

import pytest

from fuse_query_b200 import build

# (type, literal text as the s-expression reader takes it, intended value: int, or the float's bit pattern)
CASES = [
    ("i64", "-9223372036854775808", -(1 << 63)),
    ("i64", "9223372036854775807", (1 << 63) - 1),
    ("u64", "18446744073709551615", (1 << 64) - 1),
    ("i8", "-128", -128), ("i8", "127", 127),
    ("i16", "-32768", -32768), ("i16", "32767", 32767),
    ("i32", "-2147483648", -(1 << 31)), ("i32", "2147483647", (1 << 31) - 1),
    ("u8", "255", 255), ("u16", "65535", 65535), ("u32", "4294967295", (1 << 32) - 1),
    ("f32", "3.4028234663852886e38", 0x7F7FFFFF),           # f32 MAX
    ("f32", "1.401298464324817e-45", 0x00000001),           # smallest f32 subnormal
    ("f32", "-0.0", 0x80000000),
    ("f32", "inf", 0x7F800000), ("f32", "-inf", 0xFF800000),
    ("f32", "nan(0x12345)", 0x7FC12345), ("f32", "-nan(0x5)", 0xFFC00005),
    ("f32", "1e39", 0x7F800000), ("f32", "-1e39", 0xFF800000),  # overflow f32: ±inf after the (float) rounding
    ("f64", "1.7976931348623157e308", 0x7FEFFFFFFFFFFFFF),  # f64 MAX
    ("f64", "4.9406564584124654e-324", 0x0000000000000001),  # smallest f64 subnormal
    ("f64", "-0.0", 0x8000000000000000),
    ("f64", "inf", 0x7FF0000000000000), ("f64", "-inf", 0xFFF0000000000000),
    ("f64", "nan(0x12345)", 0x7FF8000000012345), ("f64", "-nan(0x5)", 0xFFF8000000000005),
]

_F32_BITS = lambda x: struct.unpack("<I", struct.pack("<f", x))[0]
_F64_BITS = lambda x: struct.unpack("<Q", struct.pack("<d", x))[0]
_CTYPE = {"i8": "fq_i8", "i16": "fq_i16", "i32": "fq_i32", "i64": "fq_i64", "u8": "fq_u8", "u16": "fq_u16", "u32": "fq_u32",
          "u64": "fq_u64"}


def _constant(ty, text):
    """the value (int) or bit pattern (float) of the one constant of type `ty` in generated `text` (emit and emit_vec
    both hold it)"""
    if ty == "f32":
        m = re.findall(r"\(\(float\)\(([-+0-9a-fx.p]+)\)\)|__int_as_float\(\(int\)0x([0-9a-f]{8})u\)", text)
        assert len(set(m)) == 1, m
        hexf, bits = m[0]
        return int(bits, 16) if bits else _F32_BITS(float.fromhex(hexf))
    if ty == "f64":
        m = re.findall(r"\(\(double\)\(([-+0-9a-fx.p]+)\)\)|__longlong_as_double\(\(long long\)0x([0-9a-f]{16})ull\)", text)
        assert len(set(m)) == 1, m
        hexf, bits = m[0]
        return int(bits, 16) if bits else _F64_BITS(float.fromhex(hexf))
    if ty == "i64" and "((fq_i64)(-9223372036854775807ll - 1))" in text:
        return -(1 << 63)
    m = re.findall(r"\(\(%s\)\((-?[0-9]+)(?:ll|ull|u)?\)\)" % _CTYPE[ty], text)
    assert len(set(m)) == 1, m
    return int(m[0])


@pytest.fixture(scope="module")
def generated(tmp_path_factory):
    tmp = tmp_path_factory.mktemp("literals")
    aotgen = str(tmp / "aotgen")
    subprocess.run(["g++", "-O1", "-std=c++17", "-o", aotgen, os.path.join(build.CSRC, "tools", "aotgen.cc"),
                    os.path.join(build.CSRC, "codegen.cc")], check=True, capture_output=True)
    # One projection per literal, so each generated struct holds exactly one constant.  A literal that prints like an
    # earlier one (-1e39 and -inf) gets another operator, because aotgen emits equal pipes once.  The last line mixes
    # non-finite constants in comparisons, an f32 sum and a predicate.
    seen = []
    lines = []
    for ty, lit, want in CASES:
        lines.append(f"PROJ\tmat\t-\t({'+-*'[seen.count((ty, want))]} (col number) ({ty} {lit}))")
        seen.append((ty, want))
    lines.append("PROJ\tmat\t(> (col number) (f64 nan))\t(< (col number) (f64 inf))\t(+ (col number) (f32 1e39))\t(> (col number) (f64 -inf))")
    pipes, out = tmp / "pipes.txt", tmp / "literals.cu"
    pipes.write_text("\n".join(lines) + "\n")
    subprocess.run([aotgen, str(pipes), str(out)], check=True, capture_output=True)
    blocks = {}
    text = out.read_text()
    for line in lines:
        head = "// " + line + "\n"
        start = text.index(head) + len(head)
        end = text.find("\n// PROJ", start)
        blocks[line] = text[start:end if end >= 0 else len(text)]
    return out, lines, blocks


def test_every_edge_literal_is_emitted_with_its_bits(generated):
    _, lines, blocks = generated
    for (ty, lit, want), line in zip(CASES, lines):
        assert _constant(ty, blocks[line]) == want, (ty, lit, blocks[line])


def test_finite_float_literals_keep_hex_float_text(generated):
    """finite constants stay in %a form (so the generated text of existing pipes does not change)"""
    _, lines, blocks = generated
    assert "((float)(0x1.fffffep+127))" in blocks[lines[12]]
    assert "((double)(-0x0p+0))" in blocks[lines[23]]


def test_generated_constants_compile_for_sm100a(generated):
    out, _, _ = generated
    r = subprocess.run([build.NVCC] + build.ARCH + ["-std=c++17", "--expt-relaxed-constexpr", "-I", os.path.join(build.CSRC, "kernels"),
                        "-c", str(out), "-o", str(out) + ".o"], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
