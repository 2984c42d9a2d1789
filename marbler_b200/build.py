"""Build marbler_b200/libmarbler_b200.so in-tree with nvcc for sm_100a (no JIT cache, no torch extension)."""
import os
import shutil
import subprocess

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB_PATH = os.path.join(HERE, "libmarbler_b200.so")
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
              "-shared", "-Xcompiler", "-fPIC"]


def sources():
    out = []
    for root in (CSRC, os.path.join(os.path.dirname(HERE), "include")):
        for f in sorted(os.listdir(root)):
            out.append(os.path.join(root, f))
    return out


def is_stale():
    if not os.path.exists(LIB_PATH):
        return True
    t = os.path.getmtime(LIB_PATH)
    return any(os.path.getmtime(s) > t for s in sources())


def build(force=False, verbose=False):
    """Compile the CUDA library if it is missing or older than its sources (one nvcc per translation
    unit, in parallel, then one link).  Returns the .so path."""
    if not force and not is_stale():
        return LIB_PATH
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        raise RuntimeError("marbler_b200: nvcc not found and %s is missing/stale" % LIB_PATH)
    from concurrent.futures import ThreadPoolExecutor
    objdir = os.path.join(HERE, "build")
    os.makedirs(objdir, exist_ok=True)
    units = sorted(f for f in os.listdir(CSRC) if f.endswith(".cu"))
    compile_flags = [f for f in NVCC_FLAGS if f != "-shared"]

    def compile_one(u):
        obj = os.path.join(objdir, u[:-3] + ".o")
        cmd = [nvcc] + compile_flags + (["-Xptxas", "-v"] if verbose else []) + ["-c", "-o", obj, os.path.join(CSRC, u)]
        res = subprocess.run(cmd, capture_output=True, text=True)
        if res.returncode != 0:
            raise RuntimeError("marbler_b200: nvcc failed on %s\n%s%s" % (u, res.stdout, res.stderr))
        return obj, res.stderr

    with ThreadPoolExecutor(max(1, min(len(units), os.cpu_count() or 1))) as ex:
        results = list(ex.map(compile_one, units))
    if verbose:
        for _, log in results:
            print(log)
    # --no-undefined: a launcher that launchers.h declares and no unit instantiates fails the link instead of leaving an
    # undefined symbol in the library
    res = subprocess.run([nvcc, "-shared", "-Xlinker", "--no-undefined", "-o", LIB_PATH] + [o for o, _ in results],
                         capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("marbler_b200: link failed\n" + res.stdout + res.stderr)
    return LIB_PATH


if __name__ == "__main__":
    print(build(force=True, verbose=True))
