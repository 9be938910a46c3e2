"""GROUP BY keys of 65..128 bits, without a GPU: the two-word table key's hash (restated in Python, checked against the
kernel's own function compiled for the host), constructed keys that share the low bits of their hash, and the generated
wide pipes compiled for sm_100a — the 128-bit compare-and-swap in shared and global memory, spills no worse than the
64-bit pipe's, and the refusal of a key set over 128 bits."""
import ctypes as C
import functools
import os
import random
import re
import subprocess

import pytest

from fuse_query_b200 import build
from test_collisions_and_scans import CLUSTER_BITS, KERNELS, M64, _cut_function, gb_hash, gb_unhash

NUM = "(col number)"
MOD7 = f"(- {NUM} (* (/ {NUM} (u64 7)) (u64 7)))"
DIV1000 = f"(/ {NUM} (u64 1000))"
LEAVES = "\t".join([f"(sum {NUM})", f"(count {NUM})", f"(min {NUM})", f"(max {NUM})"])


def gb_hash2(lo: int, hi: int, seed: int = 0) -> int:
    """fq_gb_hash2 (kernels/fq_skeleton.cuh): the hash of a two-word key under `seed`"""
    return gb_hash(hi ^ gb_hash(lo ^ seed))


@functools.lru_cache(maxsize=None)
def wide_keys(count: int, low: int = 0x2B2B2B2B2B2):
    """`count` distinct (lo, hi) keys whose unseeded fq_gb_hash2 agree in their low CLUSTER_BITS bits: lo = i, and hi is
    solved for the target hash (fq_gb_hash inverts)"""
    out = []
    for i in range(count):
        target = ((i + 1) << CLUSTER_BITS) | low
        out.append((i, gb_unhash(target) ^ gb_hash(i)))
    return tuple(out)


@pytest.fixture(scope="module")
def kernel_hash2(tmp_path_factory):
    d = tmp_path_factory.mktemp("kernel_hash2")
    src = "\n".join([
        "#include <cstdint>",
        "typedef uint64_t fq_u64;",
        "#define __device__",
        "#define __forceinline__ inline",
        _cut_function(os.path.join(KERNELS, "fq_skeleton.cuh"), "fq_gb_hash"),
        _cut_function(os.path.join(KERNELS, "fq_skeleton.cuh"), "fq_gb_hash2"),
        'extern "C" fq_u64 gb_hash2(fq_u64 lo, fq_u64 hi, fq_u64 seed) { return fq_gb_hash2(lo, hi, seed); }',
    ])
    (d / "h.cc").write_text(src)
    lib_path = str(d / "libh.so")
    subprocess.run(["g++", "-std=c++17", "-O2", "-shared", "-fPIC", "-o", lib_path, str(d / "h.cc")], check=True, capture_output=True)
    lib = C.CDLL(lib_path)
    lib.gb_hash2.restype, lib.gb_hash2.argtypes = C.c_uint64, [C.c_uint64, C.c_uint64, C.c_uint64]
    return lib.gb_hash2


def test_python_wide_hash_equals_the_kernel_source(kernel_hash2):
    rng = random.Random(5)
    edge = [0, 1, M64, M64 - 1, 1 << 63]
    cases = [(a, b, s) for a in edge for b in edge for s in (0, 1, M64)]
    cases += [(rng.getrandbits(64), rng.getrandbits(64), rng.getrandbits(64)) for _ in range(2000)]
    for lo, hi, seed in cases:
        assert kernel_hash2(lo, hi, seed) == gb_hash2(lo, hi, seed), (lo, hi, seed)


@pytest.mark.parametrize("count", [4097, 6000])
def test_constructed_wide_keys_cluster_and_a_new_seed_spreads_them(kernel_hash2, count):
    keys = wide_keys(count)
    assert len(set(keys)) == count
    mask = (1 << CLUSTER_BITS) - 1
    assert len({kernel_hash2(lo, hi, 0) & mask for lo, hi in keys}) == 1
    # under another seed the keys no longer share a home slot of a table of 2^14 slots
    homes = {kernel_hash2(lo, hi, 0x9E3779B97F4A7C15) & ((1 << 14) - 1) for lo, hi in keys}
    assert len(homes) > count // 4


def test_keys_with_one_lo_never_collide():
    """fq_gb_hash is a bijection: with lo fixed, distinct hi give distinct hashes under every seed"""
    rng = random.Random(9)
    for seed in (0, 12345, M64):
        lo = rng.getrandbits(64)
        his = {rng.getrandbits(64) for _ in range(5000)}
        assert len({gb_hash2(lo, hi, seed) for hi in his}) == len(his)


# ---- generated pipes, compiled for sm_100a ----
@pytest.fixture(scope="module")
def aotgen(tmp_path_factory):
    tmp = tmp_path_factory.mktemp("wide_aotgen")
    exe = str(tmp / "aotgen")
    subprocess.run(["g++", "-O1", "-std=c++17", "-o", exe, os.path.join(build.CSRC, "tools", "aotgen.cc"), os.path.join(build.CSRC, "codegen.cc")],
                   check=True, capture_output=True)
    return tmp, exe


def _generate(aotgen, name, keys):
    tmp, exe = aotgen
    pipes, out = tmp / f"{name}.txt", tmp / f"{name}.cu"
    pipes.write_text(f"GRP\tmat\t-\t{' ;; '.join(keys)}\t{LEAVES}\n")
    r = subprocess.run([exe, str(pipes), str(out)], capture_output=True, text=True)
    return r, out


def _kernel_info(ptxas_log, suffix):
    """{kernel suffix: spill bytes (stores + loads)} from `ptxas -v`"""
    m = re.search(r"Function properties for fqk_[0-9a-f]{16}" + suffix + r"\n\s+(\d+) bytes stack frame, (\d+) bytes spill stores, (\d+) bytes spill loads",
                  ptxas_log)
    assert m, ptxas_log
    return int(m.group(2)) + int(m.group(3))


@pytest.fixture(scope="module")
def compiled(aotgen):
    """(ptxas log, SASS) of the 64-bit and the 128-bit pipe"""
    out = {}
    for name, keys in (("narrow", [MOD7]), ("wide", [MOD7, DIV1000])):
        r, cu = _generate(aotgen, name, keys)
        assert r.returncode == 0, r.stderr
        text = cu.read_text()
        assert ("using Key = fq_gb_key2;" in text) == (name == "wide")
        obj = str(cu) + ".o"
        c = subprocess.run([build.NVCC] + build.ARCH + ["-O3", "-std=c++17", "--expt-relaxed-constexpr", "-Xptxas", "-v", "-I", KERNELS,
                            "-c", str(cu), "-o", obj],
                           capture_output=True, text=True)
        assert c.returncode == 0, c.stdout + c.stderr
        sass = subprocess.run([os.path.join(os.path.dirname(build.NVCC), "cuobjdump"), "-sass", obj], capture_output=True, text=True, check=True).stdout
        out[name] = (c.stdout + c.stderr, sass)
    return out


def _function_sass(sass, suffix):
    m = re.search(r"Function : (fqk_[0-9a-f]{16}" + suffix + r")\n(.*?)(?=\n\s+Function : |\Z)", sass, re.S)
    assert m, suffix
    return m.group(2)


def test_wide_groupby_claims_keys_with_128_bit_cas(compiled):
    _, sass = compiled["wide"]
    body = _function_sass(sass, "_groupby")
    assert "ATOMS.CAS.128" in body
    assert "ATOMG.E.CAS.128" in body
    assert "CAS.128" in _function_sass(sass, "_gbmerge")
    _, narrow = compiled["narrow"]
    assert "CAS.128" not in narrow


def test_wide_pipe_spills_no_more_than_the_narrow_one(compiled):
    for suffix in ("_groupby", "_gbmerge"):
        assert _kernel_info(compiled["wide"][0], suffix) <= _kernel_info(compiled["narrow"][0], suffix), suffix


def test_keys_over_128_bits_are_refused(aotgen):
    r, _ = _generate(aotgen, "over", [MOD7, DIV1000, f"(+ {NUM} (u64 1))"])
    assert r.returncode != 0
    assert "GROUP BY keys of 192 bits (values plus one bit per nullable key) do not pack into 64 or 128" in r.stderr
