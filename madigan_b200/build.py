"""Build ``madigan_b200/libmadigan_b200.so`` in-tree with nvcc for sm_100a.

``python -m madigan_b200.build`` (or ``__graft_entry__.build()``).  nvcc
cross-compiles without a GPU; the two translation units compile in parallel.

Flags that matter for parity: ``-fmad=false`` (no FMA contraction: the ledger's
risk gates, and therefore the bit-exact positions, depend on every rounding).
"""
import hashlib
import os
import shutil
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
# MDG_LIB_VARIANT=<name> (profiling only): build/load libmadigan_b200.<name>.so next to the product library, so
# that one GPU session can time several MDG_EXTRA_NVCC_FLAGS variants of a kernel side by side
_VARIANT = os.environ.get("MDG_LIB_VARIANT", "")
OBJ = os.path.join(HERE, "csrc", "_obj", _VARIANT) if _VARIANT else os.path.join(HERE, "csrc", "_obj")
LIB = os.path.join(HERE, f"libmadigan_b200.{_VARIANT}.so" if _VARIANT else "libmadigan_b200.so")

NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-fmad=false", "-Xcompiler", "-fPIC", "-Xcompiler", "-O2"]


def _nvcc():
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found: the CUDA library cannot be built")


def _extra_flags():
    """MDG_EXTRA_NVCC_FLAGS lets a profiling run try a variant (e.g. -DMDG_MINB16=2) without editing sources."""
    return os.environ.get("MDG_EXTRA_NVCC_FLAGS", "").split()


def _deps_hash(src="", defs=()):
    """Hash of everything one object depends on: its source, every header, and the flags."""
    h = hashlib.sha256()
    files = [f for f in sorted(os.listdir(CSRC)) if f.endswith((".cuh", ".h")) or f == src]
    files.append(os.path.join("..", "..", "include", "madigan_b200.h"))
    for f in files:
        p = os.path.join(CSRC, f)
        if os.path.isfile(p):
            h.update(f.encode())
            h.update(open(p, "rb").read())
    h.update(" ".join(NVCC_FLAGS + list(defs) + _extra_flags()).encode())
    return h.hexdigest()


def _units():
    return [("mdg_api.o", "mdg_api.cu", []), ("mdg_aux.o", "mdg_aux.cu", []), ("mdg_replay.o", "mdg_replay.cu", []),
            ("mdg_per.o", "mdg_per.cu", []), ("mdg_rewardnorm.o", "mdg_rewardnorm.cu", []), ("mdg_tearsheet.o", "mdg_tearsheet.cu", [])]


def build(force=False, verbose=False, ptxas_info=False):
    """Compile if sources changed since the last build; returns the path of the .so."""
    os.makedirs(OBJ, exist_ok=True)
    flags = list(NVCC_FLAGS) + _extra_flags() + (["-Xptxas", "-v"] if ptxas_info else [])

    def stale(u):
        obj, src, defs = u
        st = os.path.join(OBJ, obj + ".hash")
        return (force or ptxas_info or not os.path.exists(os.path.join(OBJ, obj)) or not os.path.exists(st)
                or open(st).read().strip() != _deps_hash(src, defs))

    todo = [u for u in _units() if stale(u)]
    if not todo and os.path.exists(LIB):
        return LIB
    nvcc = _nvcc()

    def compile_one(u):
        obj, src, defs = u
        cmd = [nvcc] + flags + defs + ["-c", os.path.join(CSRC, src), "-o", os.path.join(OBJ, obj)]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode == 0:
            with open(os.path.join(OBJ, obj + ".hash"), "w") as f:
                f.write(_deps_hash(src, defs))
        return u, r

    # biggest unit first so the pool's critical path is the cap-16 kernel
    units = todo
    with ThreadPoolExecutor(max_workers=min(8, os.cpu_count() or 2)) as ex:
        results = list(ex.map(compile_one, units))
    log = []
    for (obj, src, defs), r in results:
        if verbose or ptxas_info:
            log.append(f"== {obj}\n{r.stderr}")
        if r.returncode != 0:
            raise RuntimeError(f"nvcc failed for {src} {defs}:\n{r.stdout}\n{r.stderr}")
    objs = [os.path.join(OBJ, u[0]) for u in _units()]
    cmd = [nvcc, "-shared", "-o", LIB] + objs + ["-gencode", "arch=compute_100a,code=sm_100a", "-lcudart"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"link failed:\n{r.stdout}\n{r.stderr}")
    if log:
        print("\n".join(log))
    return LIB


if __name__ == "__main__":
    path = build(force="--force" in sys.argv, verbose="-v" in sys.argv, ptxas_info="--ptxas" in sys.argv)
    print(path)
