"""In-tree build of libfuse_gpu.so (CUDA kernels + C ABI) for sm_100a.

    python -m fuse_query_b200.build            # or __graft_entry__.build()

Steps: (1) g++ builds tools/aotgen from the library's own code generator; (2) aotgen writes
generated/aot_kernels.cu for the pipes in aot_pipes.txt; (3) the kernel skeleton is embedded as a
string for NVRTC; (4) nvcc -gencode arch=compute_100a,code=sm_100a builds libfuse_gpu.so.
nvcc cross-compiles without a GPU; the .so is git-ignored but travels to the GPU box.
"""
from __future__ import annotations

import hashlib
import os
import subprocess
import sys

PKG = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(PKG, "csrc")
GEN = os.path.join(CSRC, "generated")
LIB = os.path.join(PKG, "libfuse_gpu.so")
HOST_SRC = ["host/datavalues.cc", "host/functions.cc", "host/planners.cc", "host/pipeline.cc", "bindings/py_host.cc"]
HOST_HDR = ["host/fq_host.h", "host/host_internal.h"]
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]


def _run(cmd, **kw):
    r = subprocess.run(cmd, capture_output=True, text=True, **kw)
    if r.returncode != 0:
        sys.stderr.write(" ".join(cmd) + "\n" + r.stdout + r.stderr)
        raise RuntimeError(f"build step failed: {cmd[0]}")
    return r.stdout + r.stderr


def _sources():
    files = [os.path.join(CSRC, f) for f in ("fuse_gpu.cu", "codegen.cc", "codegen.h", "aot_pipes.txt")]
    files += [os.path.join(CSRC, "kernels", "fq_skeleton.cuh"), os.path.join(CSRC, "kernels", "fq_sort.cuh"), os.path.join(CSRC, "kernels", "fq_utf8.cuh"), os.path.join(CSRC, "tools", "aotgen.cc"),
              os.path.join(os.path.dirname(PKG), "include", "fuse_gpu.h"), os.path.abspath(__file__)]
    files += [os.path.join(CSRC, f) for f in HOST_SRC + HOST_HDR]
    return files


def host_module_path() -> str:
    import sysconfig
    return os.path.join(PKG, "_fuse_host" + sysconfig.get_config_var("EXT_SUFFIX"))


def _digest() -> str:
    h = hashlib.sha256()
    for f in _sources():
        with open(f, "rb") as fh:
            h.update(fh.read())
    return h.hexdigest()


def build(force: bool = False, verbose: bool = False) -> str:
    os.makedirs(GEN, exist_ok=True)
    stamp = os.path.join(GEN, "build.stamp")
    digest = _digest()
    if not force and os.path.exists(LIB) and os.path.exists(host_module_path()) and os.path.exists(stamp) and open(stamp).read() == digest:
        return LIB
    # (1) + (2) precompiled pipes through the library's own code generator
    aotgen = os.path.join(GEN, "aotgen")
    _run(["g++", "-O1", "-std=c++17", "-o", aotgen, os.path.join(CSRC, "tools", "aotgen.cc"), os.path.join(CSRC, "codegen.cc")])
    log = _run([aotgen, os.path.join(CSRC, "aot_pipes.txt"), os.path.join(GEN, "aot_kernels.cu")])
    # (3) skeleton text for NVRTC
    with open(os.path.join(CSRC, "kernels", "fq_skeleton.cuh")) as f:
        skel = f.read().replace("#pragma once\n", "")
    assert ')FQSK"' not in skel
    with open(os.path.join(GEN, "skeleton_embed.h"), "w") as f:
        f.write("// GENERATED from kernels/fq_skeleton.cuh — do not edit.\n")
        # split: a single string literal is limited to 64 KiB by some compilers
        f.write("static const char fq_skeleton_src[] =\n")
        step = 8000
        for i in range(0, len(skel), step):
            f.write('R"FQSK(' + skel[i:i + step] + ')FQSK"\n')
        f.write(";\n")
    # (4) the library
    flags = ["-O3", "-std=c++17", "-lineinfo", "-Xcompiler", "-fPIC,-Wall", "-Xptxas", "-v", "--expt-relaxed-constexpr"]
    objs = []
    for src in (os.path.join(CSRC, "fuse_gpu.cu"), os.path.join(GEN, "aot_kernels.cu")):
        obj = os.path.join(GEN, os.path.basename(src) + ".o")
        out = _run([NVCC] + ARCH + flags + ["-c", src, "-o", obj])
        with open(obj + ".ptxas.log", "w") as f:
            f.write(out)
        objs.append(obj)
    cg = os.path.join(GEN, "codegen.o")
    _run(["g++", "-O2", "-std=c++17", "-fPIC", "-c", os.path.join(CSRC, "codegen.cc"), "-o", cg])
    _run([NVCC] + ARCH + ["-shared", "-o", LIB] + objs + [cg, "-ldl", "-Xlinker", "--no-undefined"])
    # (5) the C++ host mirror of the reference's function / processor / planner surface + its pybind11 view;
    #     it calls nothing but the C ABI of libfuse_gpu.so
    import pybind11
    import sysconfig
    inc = ["-I" + pybind11.get_include(), "-I" + sysconfig.get_paths()["include"]]
    hobjs = []
    procs = []
    for src in HOST_SRC:
        obj = os.path.join(GEN, src.replace("/", "_") + ".o")
        cmd = ["g++", "-O1" if "bindings" in src else "-O2", "-std=c++17", "-fPIC", "-fvisibility=hidden", "-Wall", "-c", os.path.join(CSRC, src), "-o", obj] + inc
        procs.append((cmd, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
        hobjs.append(obj)
    for cmd, pr in procs:
        out, _ = pr.communicate()
        if pr.returncode != 0:
            sys.stderr.write(" ".join(cmd) + "\n" + out)
            raise RuntimeError("build step failed: host mirror")
    _run(["g++", "-shared", "-o", host_module_path()] + hobjs + ["-L" + PKG, "-l:libfuse_gpu.so", "-Wl,-rpath,$ORIGIN"])
    with open(stamp, "w") as f:
        f.write(digest)
    if verbose:
        print(log.strip())
        print("built", LIB)
    return LIB


if __name__ == "__main__":
    build(force="--force" in sys.argv, verbose=True)
