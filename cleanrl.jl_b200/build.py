"""Build libcleanrl_cuda.so in-tree with nvcc for sm_100a (no CPU fallback, no other arch)."""
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OUT = os.path.join(HERE, "libcleanrl_cuda.so")
SOURCES = ["gae.cu", "rollout.cu", "update.cu", "update_tc.cu", "dqn.cu", "ddpg.cu", "tblog.cu", "api.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-Xcompiler", "-fPIC", "-Xcompiler", "-fvisibility=hidden"] + os.environ.get("CRL_NVCC_EXTRA", "").split()


def _nvcc():
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found")


def needs_build():
    if not os.path.exists(OUT):
        return True
    t = os.path.getmtime(OUT)
    headers = ("cleanrl_cuda.h", "cleanrl_ddpg.h", "cleanrl_td3.h", "cleanrl_sac.h", "cleanrl_c51.h")
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [os.path.join(HERE, "..", "include", h) for h in headers]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False):
    if not force and not needs_build():
        return OUT
    nvcc = _nvcc()
    objdir = os.path.join(HERE, "build")
    os.makedirs(objdir, exist_ok=True)
    procs = []
    for src in SOURCES:
        obj = os.path.join(objdir, src.replace(".cu", ".o"))
        cmd = [nvcc] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-c", os.path.join(CSRC, src), "-o", obj]
        procs.append((src, obj, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    objs = []
    for src, obj, p in procs:
        out, _ = p.communicate()
        if verbose or p.returncode != 0:
            sys.stderr.write(out)
        if p.returncode != 0:
            raise RuntimeError("nvcc failed on %s" % src)
        objs.append(obj)
    # api.cu exports the extern "C" ABI with default visibility via the header attributes below
    cmd = [nvcc, "-shared", "-o", OUT] + objs + ["-gencode", "arch=compute_100a,code=sm_100a", "-ldl", "-lpthread"]
    subprocess.check_call(cmd)
    return OUT


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
