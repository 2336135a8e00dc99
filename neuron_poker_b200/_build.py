"""Build neuron_poker_b200/libnpk.so (CUDA kernels + C ABI) in-tree with nvcc for sm_100a.

nvcc cross-compiles without a GPU; the built library travels to the GPU box with the repository snapshot.
"""
import os
import shutil
import subprocess

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libnpk.so")
SOURCES = ["npk_capi.cu", "npk_kernels.cu", "npk_mixed.cu", "npk_ranges.cu", "npk_holdem.cu", "npk_showdown_equity.cu",
           "npk_exact_equity.cu", "npk_tables.cpp"]
HEADERS = ["npk_kernels.h", "npk_device.cuh", "npk_mc.cuh", "npk_enum_plan.cuh", "npk_tables.h", "npk_holdem_launch.h",
           os.path.join("..", "..", "include", "npk.h"), os.path.join("..", "..", "include", "npk_holdem.h")]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-Xcompiler", "-fPIC", "-Xcompiler", "-Wall", "--threads", "4"]


def _nvcc():
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found: libnpk.so cannot be built (set NVCC=/path/to/nvcc)")


def stale():
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, f) for f in SOURCES + HEADERS]
    return any(os.path.exists(d) and os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False, defines=(), out=None):
    """Compile libnpk.so if missing or older than its sources.  Returns the library path.
    `defines` / `out` build an experimental variant next to it (tools/: kernel experiments select it with NPK_LIBRARY)."""
    if not force and not stale() and out is None:
        return LIB
    objs = []
    procs = []
    tag = "" if out is None else "_" + os.path.splitext(os.path.basename(out))[0]
    os.makedirs(os.path.join(HERE, "build"), exist_ok=True)
    for src in SOURCES:
        obj = os.path.join(HERE, "build", os.path.splitext(src)[0] + tag + ".o")
        cmd = [_nvcc()] + NVCC_FLAGS + ["-D" + d for d in defines] + (["-Xptxas", "-v"] if verbose else []) + \
              ["-c", os.path.join(CSRC, src), "-o", obj]
        procs.append((cmd, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
        objs.append(obj)
    for cmd, pr in procs:
        log, _ = pr.communicate()
        if verbose and log:
            print(log)
        if pr.returncode:
            raise RuntimeError("nvcc failed: %s\n%s" % (" ".join(cmd), log))
    target = LIB if out is None else out
    link = [_nvcc(), "-shared", "-o", target] + objs + ["-gencode", "arch=compute_100a,code=sm_100a"]
    subprocess.check_call(link)
    return target


FAST = os.path.join(HERE, "_npkfast.so")
FAST_SRC = os.path.join(CSRC, "npk_pyfast.c")


def build_fast(force=False):
    """Compile the CPython binding of npk_equity_one (csrc/npk_pyfast.c) in-tree with gcc.  Returns its path."""
    import sysconfig
    if not force and os.path.exists(FAST) and os.path.getmtime(FAST) >= os.path.getmtime(FAST_SRC):
        return FAST
    cc = os.environ.get("CC") or shutil.which("gcc") or shutil.which("cc")
    if not cc:
        raise RuntimeError("no C compiler for neuron_poker_b200/_npkfast.so")
    subprocess.check_call([cc, "-O2", "-Wall", "-shared", "-fPIC", "-I" + sysconfig.get_paths()["include"],
                           "-I" + os.path.join(HERE, "..", "include"), FAST_SRC, "-o", FAST])
    return FAST


if __name__ == "__main__":
    import sys
    defs = [a[2:] for a in sys.argv[1:] if a.startswith("-D")]
    outs = [a[2:] for a in sys.argv[1:] if a.startswith("-o")]
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv, defines=defs, out=outs[0] if outs else None))
    if not outs:
        print(build_fast(force="--force" in sys.argv))
