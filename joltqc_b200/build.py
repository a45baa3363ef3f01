"""In-tree build of the CUDA library (libjoltqc_b200.so) for sm_100a.

nvcc is driven directly (no cmake): one object per bra class from csrc/jk_inst.cu (J/K) and from
csrc/jk_grad_inst.cu (J/K energy gradient) plus the engine, linked into joltqc_b200/libjoltqc_b200.so.
Objects are cached under joltqc_b200/_build/ and rebuilt when any csrc file is newer.
"""
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OBJ = os.path.join(HERE, "_build")
LIB = os.path.join(HERE, "libjoltqc_b200.so")
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-lineinfo",
         "-Xcompiler", "-fPIC", "-ccbin", "/usr/bin/g++", "-I", CSRC]
BRA = [(i, j) for i in range(5) for j in range(i + 1)]


def _newest_src():
    return max(os.path.getmtime(os.path.join(CSRC, f)) for f in os.listdir(CSRC))


def _run(cmd):
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("nvcc failed: %s\n%s\n%s" % (" ".join(cmd), r.stdout, r.stderr))
    return r.stderr


def build(force=False, verbose=False, jobs=None, extra_flags=None, out=None, objdir=None):
    """extra_flags: e.g. ["-DJQC_WARP_FORCE_ACC=40", "-DJQC_WARP_FORCE_REGS=168"] for a tuning build
    (forces a full rebuild; see tools/tune_warp.py)."""
    global FLAGS, OBJ, LIB
    if extra_flags:
        FLAGS = FLAGS + list(extra_flags)
        force = True
    if out:       # variant build: own output file and object directory
        LIB = os.path.abspath(out)
        OBJ = objdir or (OBJ + "_" + os.path.splitext(os.path.basename(out))[0])
    os.makedirs(OBJ, exist_ok=True)
    stamp = _newest_src()
    todo = []
    objs = []
    for unit in ("jk_inst", "jk_grad_inst"):
        for i, j in BRA:
            o = os.path.join(OBJ, f"{unit}_{i}{j}.o")
            objs.append(o)
            if force or not os.path.exists(o) or os.path.getmtime(o) < stamp:
                todo.append([NVCC] + FLAGS + [f"-DJQC_LI={i}", f"-DJQC_LJ={j}", "-c", os.path.join(CSRC, unit + ".cu"), "-o", o])
    o = os.path.join(OBJ, "engine.o")
    objs.append(o)
    if force or not os.path.exists(o) or os.path.getmtime(o) < stamp:
        todo.append([NVCC] + FLAGS + ["-c", os.path.join(CSRC, "engine.cu"), "-o", o])
    if todo:
        # heaviest first
        todo.sort(key=lambda c: -sum(int(x[-1]) for x in c if x.startswith("-DJQC_L")))
        with ThreadPoolExecutor(jobs or os.cpu_count()) as ex:
            for cmd, err in zip(todo, ex.map(_run, todo)):
                if verbose and err.strip():
                    print(err, file=sys.stderr)
    if todo or not os.path.exists(LIB):
        _run([NVCC, "-shared", "-o", LIB] + objs + ["-lcudart"])
    return LIB


if __name__ == "__main__":
    outs = [a[6:] for a in sys.argv[1:] if a.startswith("--out=")]
    print(build(force="--force" in sys.argv, verbose=True, extra_flags=[a for a in sys.argv[1:] if a.startswith("-D")],
                out=outs[0] if outs else None))
