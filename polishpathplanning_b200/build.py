"""Builds libppp_gpu.so IN-TREE with nvcc for sm_100a (cross-compiles without a GPU).

    python -m polishpathplanning_b200.build [--force]

The .so lands next to this file (git-ignored, but it travels to the GPU box with the snapshot).
"""
import concurrent.futures
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OUT = os.path.join(HERE, "libppp_gpu.so")
OUT_CHECK = os.path.join(HERE, "libppp_gpu_check.so")   # -DPPP_CHECK_BOUNDS: device-side index assertions (tests/test_gpu_bounds.py)
OBJ_DIR = os.path.join(HERE, "csrc", "_obj")
OBJ_DIR_CHECK = os.path.join(HERE, "csrc", "_obj", "check")
SOURCES = ["api.cu", "scan.cu", "grid.cu", "knn.cu", "slices.cu", "exchange.cu", "mls.cu", "voxel.cu"]
HEADERS = ["ppp_internal.cuh", "ppp_device.cuh", "sortnet.cuh", os.path.join("..", "..", "include", "ppp_gpu.h")]

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-lineinfo", "-O3", "-std=c++17",
    "--fmad=false",            # parity: no FMA contraction anywhere (SURVEY.md §7.3)
    "-Xcompiler", "-fPIC,-O2,-ffp-contract=off",
    "--expt-extended-lambda", "--expt-relaxed-constexpr",
    "-Xptxas", "-v",
]


def nvcc():
    p = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(p):
        raise RuntimeError("nvcc not found: libppp_gpu.so cannot be built (there is no CPU fallback)")
    return p


def _stale(target, deps):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps if os.path.exists(d))


def _compile(src, force, check=False):
    obj = os.path.join(OBJ_DIR_CHECK if check else OBJ_DIR, src.replace(".cu", ".o"))
    deps = [os.path.join(CSRC, src)] + [os.path.join(CSRC, h) for h in HEADERS]
    if force or _stale(obj, deps):
        cmd = [nvcc()] + NVCC_FLAGS + (["-DPPP_CHECK_BOUNDS"] if check else []) + ["-c", os.path.join(CSRC, src), "-o", obj]
        r = subprocess.run(cmd, capture_output=True, text=True)
        log = r.stdout + r.stderr
        with open(obj + ".log", "w") as f:
            f.write(" ".join(cmd) + "\n" + log)
        if r.returncode != 0:
            raise RuntimeError("nvcc failed for %s:\n%s" % (src, log))
        return obj, True
    return obj, False


def build(force=False, verbose=False, check=False):
    """check=True builds libppp_gpu_check.so (device-side bounds assertions) instead of the product library."""
    out = OUT_CHECK if check else OUT
    os.makedirs(OBJ_DIR_CHECK if check else OBJ_DIR, exist_ok=True)
    with concurrent.futures.ThreadPoolExecutor(max_workers=len(SOURCES)) as ex:
        res = list(ex.map(lambda s: _compile(s, force, check), SOURCES))
    objs = [o for o, _ in res]
    if force or any(c for _, c in res) or _stale(out, objs):
        cmd = [nvcc(), "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", out] + objs
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError("link failed:\n" + r.stdout + r.stderr)
    if verbose:
        for o in objs:
            with open(o + ".log") as f:
                sys.stdout.write(f.read())
    return out


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv, check="--check" in sys.argv))
