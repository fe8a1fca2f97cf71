"""Builds libarroyo_b200.so in-tree with nvcc for sm_100a (no JIT cache: the .so travels with the
repo snapshot to the GPU box)."""
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libarroyo_b200.so")
SOURCES = ["abi.cu", "window_agg.cu", "shuffle.cu", "join.cu", "session.cu", "updating_agg.cu", "ttl_join.cu"]
HEADERS = ["common.cuh", "dict.cuh", "bdict.cuh", "ingest_two_pass.cuh", "scan.cuh", "planner.h", "arrow_io.h", "op.h", os.path.join("..", "..", "include", "arroyo_b200.h")]


def nvcc_path() -> str:
    p = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(p):
        raise RuntimeError("nvcc not found")
    return p


def is_stale() -> bool:
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    for f in SOURCES + HEADERS:
        if os.path.getmtime(os.path.join(CSRC, f)) > t:
            return True
    return os.path.getmtime(os.path.abspath(__file__)) > t


def build(force: bool = False, verbose: bool = False) -> str:
    if not force and not is_stale():
        return LIB
    objs = []
    flags = [
        "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-lineinfo",
        "-Xcompiler", "-fPIC,-Wall,-Wno-unused-function", "--expt-relaxed-constexpr",
    ]
    if verbose:
        flags += ["-Xptxas", "-v"]
    for knob in ("AB_INGEST_MIN_BLOCKS", "AB_INGEST_PREFETCH", "AB_P1_THREADS", "AB_P1_RPT"):  # tuning knobs for experiments
        if os.environ.get(knob):
            flags += [f"-D{knob}=" + os.environ[knob]]
    build_dir = os.path.join(HERE, "build")
    os.makedirs(build_dir, exist_ok=True)
    procs = []
    for s in SOURCES:
        o = os.path.join(build_dir, s.replace(".cu", ".o"))
        objs.append(o)
        cmd = [nvcc_path(), *flags, "-c", os.path.join(CSRC, s), "-o", o]
        procs.append((s, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    failed = False
    for s, p in procs:
        out, _ = p.communicate()
        if p.returncode != 0:
            failed = True
            sys.stderr.write(f"--- nvcc {s} failed ---\n{out}\n")
        elif verbose or out.strip():
            sys.stderr.write(f"--- nvcc {s} ---\n{out}\n")
    if failed:
        raise RuntimeError("nvcc compilation failed")
    tmp = LIB + ".tmp"  # link beside the target, then rename: a reader never sees a half-written library
    cmd = [nvcc_path(), "-gencode", "arch=compute_100a,code=sm_100a", "-shared", "-o", tmp, *objs, "-lcudart"]
    subprocess.check_call(cmd)
    os.replace(tmp, LIB)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
