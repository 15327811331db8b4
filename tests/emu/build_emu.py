"""TEST INFRASTRUCTURE ONLY: build `libhqq_b200_emu.so` -- the kernels of hqq_b200/csrc (quantizer, bit-packing, small-M / one-token
forward, tcgen05 GEMM, the decode glue kernels except the cluster argmax) compiled by g++ against tests/emu/include/cuda_runtime.h and
executed on the CPU by cooperative fibers.

The .cu sources are used as they are, except for two textual rewrites CUDA syntax forces on a C++ compiler:
  kernel<<<grid, block, smem, stream>>>(args)   ->  EMU_LAUNCH((kernel), grid, block, smem, stream)(args)
  extern __shared__ ... name[];                 ->  a pointer to the emulator's dynamic shared-memory buffer
Only tests load the result (tests/test_emu_cpu.py, through ctypes, never through hqq_b200._lib)."""
import hashlib
import os
import re
import subprocess

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
CSRC = os.path.join(ROOT, "hqq_b200", "csrc")
OUT = os.path.join(HERE, "_build")
LIB = os.path.join(OUT, "libhqq_b200_emu.so")
SOURCES = ["api.cu", "quantize.cu", "bitpack.cu", "linear_small.cu", "linear_gemm.cu", "linear.cu", "decode_glue.cu"]
CUDA_INC = os.environ.get("CUDA_INCLUDE", "/usr/local/cuda/include")

EXTRA = ''


def rewrite(src: str) -> str:
    out, i = [], 0
    while True:
        j = src.find("<<<", i)
        if j < 0:
            out.append(src[i:])
            break
        k, depth = j, 0
        while k > 0:  # walk back over the kernel expression, template arguments included
            c = src[k - 1]
            if c == ">":
                depth += 1
            elif c == "<":
                depth -= 1
            elif depth == 0 and not (c.isalnum() or c in "_:"):
                break
            k -= 1
        e = src.index(">>>", j)
        out.append(src[i:k])
        out.append(f"EMU_LAUNCH(({src[k:j]}), {src[j + 3:e]})")
        i = e + 3
    s = "".join(out)
    s = re.sub(r"extern\s+__shared__\s+(?:__align__\(\d+\)\s+)?(\w+)\s+(\w+)\[\];",
               r"\1* \2 = reinterpret_cast<\1*>(::emu::dyn_smem);", s)
    return s


def digest() -> str:
    h = hashlib.sha256()
    headers = sorted(f for f in os.listdir(CSRC) if f.endswith(".cuh"))  # every header: a new one must not leave a stale library
    files = [os.path.join(CSRC, f) for f in SOURCES + headers] + [os.path.join(ROOT, "include", "hqq_b200.h"), __file__,
                                                                  os.path.join(HERE, "include", "cuda_runtime.h"),
                                                                  os.path.join(HERE, "emu_runtime.cpp")]
    for f in files:
        with open(f, "rb") as fh:
            h.update(fh.read())
    return h.hexdigest()


def build(force: bool = False) -> str:
    stamp = os.path.join(OUT, "stamp")
    d = digest()
    if not force and os.path.exists(LIB) and os.path.exists(stamp) and open(stamp).read() == d:
        return LIB
    gen = os.path.join(OUT, "gen")
    os.makedirs(gen, exist_ok=True)
    cpps = [os.path.join(HERE, "emu_runtime.cpp")]
    for f in SOURCES:
        p = os.path.join(gen, f[:-3] + ".cpp")
        with open(os.path.join(CSRC, f)) as fh, open(p, "w") as out:
            out.write(f"// generated from hqq_b200/csrc/{f} by tests/emu/build_emu.py -- do not edit\n" + rewrite(fh.read()))
        cpps.append(p)
    extra = os.path.join(gen, "emu_extra.cpp")
    with open(extra, "w") as out:
        out.write(EXTRA)
    cpps.append(extra)
    flags = ["-O1", "-std=c++17", "-fPIC", "-ffp-contract=off", "-w", "-DHQQ_EMU", "-I", os.path.join(HERE, "include"), "-I", CSRC, "-I", CUDA_INC]
    objs = []
    procs = []
    for c in cpps:
        o = os.path.join(OUT, os.path.basename(c)[:-4] + ".o")
        objs.append(o)
        procs.append((c, subprocess.Popen(["g++", *flags, "-c", c, "-o", o], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    for c, p in procs:
        log = p.communicate()[0]
        if p.returncode != 0:
            raise RuntimeError(f"g++ failed on {c}:\n{log[-4000:]}")
    r = subprocess.run(["g++", "-shared", "-Wl,-Bsymbolic", *objs, "-o", LIB], capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("link failed:\n" + r.stderr[-2000:])
    with open(stamp, "w") as fh:
        fh.write(d)
    return LIB


if __name__ == "__main__":
    print(build(force=True))
