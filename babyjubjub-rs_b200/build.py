"""Builds libbjj_cuda.so for sm_100a with nvcc (in-tree, so the .so travels to the GPU box).

One object per translation unit, compiled in parallel (the heavy kernels are minutes of ptxas each),
then linked into babyjubjub-rs_b200/libbjj_cuda.so.  The measurement tools (tools/microbench/*.cu)
are built into babyjubjub-rs_b200/bin/; they are not part of the library.
"""
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OBJ = os.path.join(HERE, "build")
BIN = os.path.join(HERE, "bin")
GEN = os.path.join(CSRC, "generated", "bjj_consts.inc")
LIB = os.path.join(HERE, "libbjj_cuda.so")
LIB_UNITS = ["bjj_cuda.cu", "bjj_multi.cu", "k_verify.cu", "k_verify_base.cu", "k_mulscalar.cu", "k_sign.cu", "k_poseidon.cu", "k_msm.cu"]
MB = os.path.join(HERE, "tools", "microbench")
TOOLS = ["imad_bench.cu", "pipe_probe.cu", "fr_layouts.cu"]
ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]
COMMON = ARCH + ["-O3", "-lineinfo", "-std=c++17", "-diag-suppress", "20091", "-diag-suppress", "177"]


def _stale(target, sources):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(s) > t for s in sources)


def headers():
    out = [os.path.join(CSRC, f) for f in sorted(os.listdir(CSRC)) if f.endswith((".cuh", ".h"))]
    out += [os.path.join(HERE, "..", "include", "bjj_cuda.h"), GEN]
    return out


def generate_constants(force=False):
    gen_py = os.path.join(HERE, "tools", "gen_constants.py")
    if force or _stale(GEN, [gen_py]):
        subprocess.check_call([sys.executable, gen_py, GEN])
    return GEN


def _run(cmd, log):
    p = subprocess.run(cmd, cwd=CSRC, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if log is not None:
        log.append(p.stdout)
    if p.returncode != 0:
        raise RuntimeError("command failed: %s\n%s" % (" ".join(cmd), p.stdout))


def build(force=False, verbose=False, tools=True):
    generate_constants()
    os.makedirs(OBJ, exist_ok=True)
    os.makedirs(BIN, exist_ok=True)
    nvcc = os.environ.get("NVCC", "nvcc")
    hdrs = headers()
    logs = []
    jobs = []
    objs = []
    for unit in LIB_UNITS:
        src = os.path.join(CSRC, unit)
        obj = os.path.join(OBJ, unit[:-3] + ".o")
        objs.append(obj)
        if force or _stale(obj, [src] + hdrs):
            cmd = [nvcc] + COMMON + ["-Xcompiler", "-fPIC"] + (["-Xptxas", "-v"] if verbose else []) + ["-c", src, "-o", obj]
            jobs.append(cmd)
    if tools:
        for unit in TOOLS:
            src = os.path.join(MB, unit)
            exe = os.path.join(BIN, unit[:-3])
            mb_hdrs = [os.path.join(MB, f) for f in os.listdir(MB) if f.endswith(".cuh")]
            if force or _stale(exe, [src] + hdrs + mb_hdrs):
                jobs.append([nvcc] + COMMON + ["-I", CSRC, "-o", exe, src])
    if jobs:
        with ThreadPoolExecutor(max_workers=min(len(jobs), os.cpu_count() or 1)) as ex:
            list(ex.map(lambda c: _run(c, logs), jobs))
    if force or _stale(LIB, objs):
        _run([nvcc] + ARCH + ["-shared", "-o", LIB + ".tmp"] + objs, logs)
        os.replace(LIB + ".tmp", LIB)
    if verbose:
        print("\n".join(logs))
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
