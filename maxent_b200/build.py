"""Build libmaxent_b200.so in-tree with nvcc for sm_100a (no JIT cache: the .so travels to the GPU box).

    python -m maxent_b200.build            # incremental
    python -m maxent_b200.build --force
"""
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
CSRC = os.path.join(HERE, "csrc")
OBJ = os.path.join(HERE, "build")
LIB = os.path.join(HERE, "libmaxent_b200.so")
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
         "-Xcompiler", "-fPIC", "-I" + os.path.join(ROOT, "include"), "-I" + CSRC]
SWEEP2_NT = (4, 5, 6, 7, 8, 9, 10, 12, 16, 20, 24, 28, 32)    # spectrum-per-CTA engine (csrc/mx_sweep2.cuh); > 10: wide


def _units():
    units = [("mx_api.o", "mx_api.cu", []), ("mx_svd.o", "mx_svd.cu", []), ("mx_dispatch.o", "mx_dispatch.cu", []),
             ("mx_hilbert.o", "mx_hilbert.cu", []), ("mx_resolvent.o", "mx_resolvent.cu", [])]
    for nt in SWEEP2_NT:
        units.append(("mx_sweep2_nt%d.o" % nt, "mx_sweep2_inst.cu", ["-DMX_NT=%d" % nt]))
    return units


def _newest_source():
    t = 0.0
    for d in (CSRC, os.path.join(ROOT, "include")):
        for f in os.listdir(d):
            t = max(t, os.path.getmtime(os.path.join(d, f)))
    return t


def build(force=False, verbose=False):
    os.makedirs(OBJ, exist_ok=True)
    src_t = _newest_source()
    if not force and os.path.exists(LIB) and os.path.getmtime(LIB) >= src_t:
        return LIB

    def compile_one(u):
        obj, src, extra = u
        out = os.path.join(OBJ, obj)
        if not force and os.path.exists(out) and os.path.getmtime(out) >= src_t:
            return out
        cmd = [NVCC] + FLAGS + extra + ["-c", os.path.join(CSRC, src), "-o", out]
        if verbose:
            cmd.insert(1, "-Xptxas=-v")
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError("nvcc failed for %s:\n%s" % (src, r.stderr))
        if verbose:
            sys.stderr.write(r.stderr)
        return out

    with ThreadPoolExecutor(max_workers=min(8, os.cpu_count() or 1)) as ex:
        objs = list(ex.map(compile_one, _units()))
    r = subprocess.run([NVCC, "-shared", "-o", LIB] + objs + ["-lcudart"], capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("link failed:\n" + r.stderr)
    return LIB


def build_variant(tag, defines, nts=(7,), verbose=False):
    """A/B builds of the sweep kernel: recompile the listed tile-count instantiations with extra -D flags into
    build/<tag>/ and link them with the other objects of the default build -> libmaxent_b200_<tag>.so
    (selected at run time with MAXENT_B200_LIB, see tools/ab_bench.py)."""
    build()
    odir = os.path.join(OBJ, tag)
    os.makedirs(odir, exist_ok=True)
    objs = []
    for obj, src, extra in _units():
        m = [nt for nt in nts if obj == "mx_sweep2_nt%d.o" % nt]
        if not m:
            objs.append(os.path.join(OBJ, obj))
            continue
        out = os.path.join(odir, obj)
        cmd = [NVCC] + FLAGS + extra + ["-D" + d for d in defines] + ["-c", os.path.join(CSRC, src), "-o", out]
        if verbose:
            cmd.insert(1, "-Xptxas=-v")
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError("nvcc failed for %s [%s]:\n%s" % (src, tag, r.stderr))
        if verbose:
            sys.stderr.write(r.stderr)
        objs.append(out)
    lib = os.path.join(HERE, "libmaxent_b200_%s.so" % tag)
    r = subprocess.run([NVCC, "-shared", "-o", lib] + objs + ["-lcudart"], capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("link failed:\n" + r.stderr)
    return lib


if __name__ == "__main__":
    if "--variant" in sys.argv:          # python -m maxent_b200.build --variant <tag> [-DNAME[=V] ...]
        tag = sys.argv[sys.argv.index("--variant") + 1]
        print(build_variant(tag, [a[2:] for a in sys.argv if a.startswith("-D")], verbose="-v" in sys.argv))
    else:
        print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
