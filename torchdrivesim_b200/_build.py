"""Builds libtds_b200.so (hand-written sm_100a CUDA + the C ABI of include/tds_b200.h) with nvcc.

The library is built IN-TREE (torchdrivesim_b200/_build/libtds_b200.so) so that it travels with the
repository snapshot to the GPU box; nvcc cross-compiles sm_100a without a GPU.
"""
import os
import shutil
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(_HERE, "csrc")
OUT_DIR = os.path.join(_HERE, "_build")
LIB_PATH = os.path.join(OUT_DIR, "libtds_b200.so")
SOURCES = ["common.cu", "kinematic.cu", "collision.cu", "map.cu", "map_segments.cu", "offroad.cu", "range_scan.cu", "raster.cu", "raster_g32.cu", "raster_g128.cu", "raster_g256.cu", "rollout.cu", "time_to_collision.cu"]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
    # every fp32 mul/add separately rounded, as the reference's eager CPU ops (see csrc/tds_common.cuh)
    "-fmad=false",
    "-Xcompiler", "-fPIC",
]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found: cannot build libtds_b200.so")


def _stale() -> bool:
    if not os.path.exists(LIB_PATH):
        return True
    t = os.path.getmtime(LIB_PATH)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [os.path.join(_HERE, "..", "include", "tds_b200.h")]
    return any(os.path.getmtime(d) > t for d in deps)


def build_library(force: bool = False, verbose: bool = False, extra_flags=(), out_path: str = None) -> str:
    """extra_flags / out_path build an experimental variant next to the default library (profiling aid)."""
    lib_path = out_path or LIB_PATH
    if not force and out_path is None and not _stale():
        return LIB_PATH
    os.makedirs(OUT_DIR, exist_ok=True)
    nvcc = _nvcc()
    objs = []
    procs = []
    tag = "" if out_path is None else "." + os.path.basename(out_path)
    for src in SOURCES:
        obj = os.path.join(OUT_DIR, src.replace(".cu", tag + ".o"))
        cmd = [nvcc] + NVCC_FLAGS + list(extra_flags) + (["-Xptxas", "-v"] if verbose else []) + \
            ["-c", os.path.join(CSRC, src), "-o", obj]
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
        objs.append(obj)
    for src, p in procs:
        out, _ = p.communicate()
        if verbose or p.returncode != 0:
            print(out)
        if p.returncode != 0:
            raise RuntimeError(f"nvcc failed on {src}")
    subprocess.check_call([nvcc, "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", lib_path] + objs + ["-lcudart"])
    return lib_path


if __name__ == "__main__":
    import sys
    print(build_library(force=True, verbose="-v" in sys.argv))
