"""Build libtik.so in-tree with nvcc for sm_100a (no torch / pybind dependency: plain C ABI).

    python -m temporal_inverse_kinematics_b200.build [--force] [-v]
"""
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libtik.so")
SOURCES = ["geometry.cu", "fk.cu", "stem.cu", "stem_block.cu", "stgcn_simt.cu", "rowgemm_tf32.cu", "stgcn_umma.cu", "gcn_fused.cu", "tcn_halo.cu", "plan.cu", "latency.cu", "pack.cu", "lbs.cu", "keypoints.cu", "fit.cu", "fit_shape.cu"]
HEADERS = ["tik_common.cuh", "fk_device.cuh", "fit_device.cuh", "umma_prepared.h", "umma_ptx.cuh", os.path.join("..", "..", "include", "tik.h")]


def _nvcc():
    for c in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if c and os.path.exists(c):
            return c
    raise RuntimeError("nvcc not found")


def _stale():
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, s) for s in SOURCES + HEADERS] + [os.path.abspath(__file__)]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False):
    """Compiles every CUDA source for sm_100a into temporal_inverse_kinematics_b200/libtik.so."""
    if not force and not os.environ.get("TIK_BUILD_VARIANT") and not _stale():
        return LIB
    objs = []
    flags = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17", "-Xcompiler", "-fPIC",
             "--expt-relaxed-constexpr"]
    if verbose:
        flags += ["-Xptxas", "-v"]
    variant = os.environ.get("TIK_BUILD_VARIANT")   # A/B library next to the product one: build/libtik_<name>.so with -D<NAME>
    obj_dir = os.path.join(HERE, "build", variant) if variant else os.path.join(HERE, "build")
    if variant:
        flags += ["-D" + variant.upper()]
    procs = []
    os.makedirs(obj_dir, exist_ok=True)
    for s in SOURCES:
        o = os.path.join(obj_dir, s.replace(".cu", ".o"))
        objs.append(o)
        procs.append((s, subprocess.Popen([_nvcc(), *flags, "-c", os.path.join(CSRC, s), "-o", o],
                                          stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    failed = False
    for s, p in procs:
        out, _ = p.communicate()
        if verbose or p.returncode != 0:
            sys.stderr.write(out)
        failed |= p.returncode != 0
    if failed:
        raise RuntimeError("nvcc failed")
    out = os.path.join(HERE, "build", f"libtik_{variant}.so") if variant else LIB
    subprocess.check_call([_nvcc(), "-shared", "-Wno-deprecated-gpu-targets", "-o", out, *objs, "-cudart", "static"])
    return out


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
