"""In-tree build of libmdir_b200.so (sm_100a only; nvcc cross-compiles without a GPU).

    python -m mdir_b200.build [--force] [--selftest]

The shared library lands next to this file (mdir_b200/libmdir_b200.so: git-ignored,
but it travels to the GPU box with the gpurun snapshot)."""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libmdir_b200.so")
SOURCES = ["api.cu", "pool_head.cu", "clahe.cu", "topk.cu", "ranks.cu", "sim_scan.cu", "evaluate.cu", "colorspace.cu", "mining.cu", "gemm_f64.cu", "shard_merge.cu", "composite.cu", "compact.cu", "diffusion.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
              "-Xcompiler", "-fPIC", "--expt-relaxed-constexpr"]


def _nvcc():
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if cand and (os.path.isabs(cand) and os.path.exists(cand) or not os.path.isabs(cand)):
            return cand
    raise RuntimeError("nvcc not found")


def _stale(target, deps):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False):
    """Compile every .cu under csrc/ and link libmdir_b200.so.  Returns the library path."""
    hdrs = [os.path.join(CSRC, "common.cuh"), os.path.join(os.path.dirname(HERE), "include", "mdir_b200.h"),
            os.path.abspath(__file__)]
    objdir = os.path.join(HERE, "build")
    os.makedirs(objdir, exist_ok=True)
    nvcc = _nvcc()
    objs = []
    procs = []
    for src in SOURCES:
        s = os.path.join(CSRC, src)
        o = os.path.join(objdir, src.replace(".cu", ".o"))
        objs.append(o)
        if force or _stale(o, [s] + hdrs):
            cmd = [nvcc] + NVCC_FLAGS + ["-c", s, "-o", o]
            if verbose:
                print(" ".join(cmd))
            procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT)))
    for src, pr in procs:
        out, _ = pr.communicate()
        if pr.returncode != 0:
            raise RuntimeError("nvcc failed on %s:\n%s" % (src, out.decode()))
    if force or procs or _stale(LIB, objs):
        cmd = [nvcc, "-shared", "-o", LIB] + objs + ["-gencode", "arch=compute_100a,code=sm_100a", "-cudart", "static"]
        r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT)
        if r.returncode != 0:
            raise RuntimeError("link failed:\n%s" % r.stdout.decode())
    return LIB


def build_selftest(force=False):
    """tools/selftest.cu: a torch-free GPU self-test binary (used under gpurun for quick kernel bring-up)."""
    root = os.path.dirname(HERE)
    src = os.path.join(root, "tools", "selftest.cu")
    out = os.path.join(root, "tools", "selftest")
    if not os.path.exists(src):
        return None
    build(force=force)
    if force or _stale(out, [src, LIB]):
        cmd = [_nvcc(), "-gencode", "arch=compute_100a,code=sm_100a", "-O2", "-std=c++17", src, "-o", out,
               "-L" + HERE, "-lmdir_b200", "-Xlinker", "-rpath", "-Xlinker", "$ORIGIN/../mdir_b200"]
        r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT)
        if r.returncode != 0:
            raise RuntimeError("selftest build failed:\n%s" % r.stdout.decode())
    return out


if __name__ == "__main__":
    lib = build(force="--force" in sys.argv, verbose=True)
    print("built", lib)
    if "--selftest" in sys.argv:
        print("built", build_selftest(force="--force" in sys.argv))
