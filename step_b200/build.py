"""Build libstep_b200.so (hand-written sm_100a kernels + C ABI) in-tree with nvcc.

`python -m step_b200.build` or `__graft_entry__.build()`.  nvcc cross-compiles without a GPU.
"""
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libstep_b200.so")
SOURCES = ["ts_encoder.cu", "ts_train.cu", "tc_encoder.cu", "tc_attn_train.cu", "graph_learn.cu", "trunk.cu", "trunk_fc.cu", "tc_gemm.cu", "gw_glue.cu", "optim.cu", "gwnet.cu"]
ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]


def nvcc_path() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found: libstep_b200.so cannot be built")


def needs_rebuild() -> bool:
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [os.path.join(HERE, "..", "include", "step_b200.h")]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False) -> str:
    if not force and not needs_rebuild():
        return LIB
    nvcc = nvcc_path()
    objs = []
    procs = []
    os.makedirs(os.path.join(HERE, "build"), exist_ok=True)
    for src in SOURCES:
        obj = os.path.join(HERE, "build", src.replace(".cu", ".o"))
        objs.append(obj)
        cmd = [nvcc, *ARCH, "-O3", "-lineinfo", "-std=c++17", "-Xcompiler", "-fPIC", *os.environ.get("STEP_B200_NVCC_FLAGS", "").split(),
               "-c", os.path.join(CSRC, src), "-o", obj]
        if verbose:
            cmd.insert(1, "-Xptxas=-v")
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    for src, p in procs:
        out, _ = p.communicate()
        if verbose or p.returncode:
            sys.stderr.write(out)
        if p.returncode:
            raise RuntimeError(f"nvcc failed on {src}")
    cmd = [nvcc, *ARCH, "-shared", "-o", LIB, *objs]
    subprocess.run(cmd, check=True)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
