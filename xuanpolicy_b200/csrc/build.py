"""Builds libxb200.so (hand-written sm_100a kernels + C ABI) in-tree with nvcc.

    python -m xuanpolicy_b200.csrc.build [--force]

nvcc cross-compiles without a GPU.  The environment TU is built with -fmad=false so that no fp64 multiply-add
is contracted (bit-exact physics); every TU gets -lineinfo so ncu's source page maps to these files.
"""
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.dirname(HERE)
OUT = os.path.join(PKG, "libxb200.so")
OBJ = os.path.join(HERE, "_obj")
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]
COMMON = ["-O3", "-std=c++17", "-lineinfo", "-Xcompiler", "-fPIC", "-Xptxas", "-v"] + os.environ.get("XB_NVCC_EXTRA", "").split()
SOURCES = {
    "api.cu": [],
    "env_classic.cu": ["-fmad=false"],
    "buffer.cu": [],
    "gae.cu": [],
    "ppo_loss.cu": [],
    "dist_loss.cu": [],
    "ppokl_loss.cu": [],
    "sample.cu": [],
    "optim.cu": [],
    "peer_comm.cu": [],
    "host_utils.cu": [],
    "mlp_epilogue.cu": [],
    "normalize.cu": [],
    "dense_tc.cu": [],
    "mlp_trunk.cu": [],
}
# every header in this directory (a forgotten one leaves stale objects behind: normalize.cuh once was)
HEADERS = sorted(f for f in os.listdir(HERE) if f.endswith((".cuh", ".inc"))) + [os.path.join("..", "..", "include", "xb200.h")]


def _stale(target, deps):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def _compile(src, extra, force, log, obj_dir=None):
    obj = os.path.join(obj_dir or OBJ, src.replace(".cu", ".o"))
    deps = [os.path.join(HERE, src)] + [os.path.join(HERE, h) for h in HEADERS]
    if force or _stale(obj, deps):
        cmd = [NVCC] + ARCH + COMMON + extra + ["-c", os.path.join(HERE, src), "-o", obj]
        r = subprocess.run(cmd, capture_output=True, text=True)
        log.append("$ " + " ".join(cmd) + "\n" + r.stdout + r.stderr)
        if r.returncode != 0:
            raise RuntimeError("nvcc failed for %s:\n%s%s" % (src, r.stdout, r.stderr))
    return obj


def build(force=False, verbose=False, out=None, obj_dir=None, extra=()):
    """`out` / `obj_dir` / `extra`: a second, differently flagged build next to the product library (e.g. the
    -DXB_DENSE_TS timeline build of tools/profile/dense_timeline.py); the defaults build xuanpolicy_b200/libxb200.so."""
    out, obj_dir = out or OUT, obj_dir or OBJ
    os.makedirs(obj_dir, exist_ok=True)
    log = []
    with ThreadPoolExecutor(max_workers=min(8, len(SOURCES))) as ex:
        objs = list(ex.map(lambda kv: _compile(kv[0], kv[1] + list(extra), force, log, obj_dir), SOURCES.items()))
    if force or _stale(out, objs):
        cmd = [NVCC] + ARCH + ["-shared", "-o", out] + objs + ["-cudart", "static"]
        r = subprocess.run(cmd, capture_output=True, text=True)
        log.append("$ " + " ".join(cmd) + "\n" + r.stdout + r.stderr)
        if r.returncode != 0:
            raise RuntimeError("link failed:\n%s%s" % (r.stdout, r.stderr))
    with open(os.path.join(obj_dir, "build.log"), "a") as f:
        f.write("\n".join(log))
    if verbose:
        print("\n".join(log))
    return out


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose=True))
