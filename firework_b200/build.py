"""Builds libfirework_b200.so (and the static archive libfirework_b200.a) in-tree with nvcc for sm_100a.

No torch involved; plain C ABI.  Every translation unit is compiled on its own (in parallel) into build/*.o, then
linked into the shared library the Python host loads and archived into the static library a Rust `build.rs` would link
(INTEGRATION.md; BASELINE.json north_star: "a CUDA static library built by build.rs").
"""
from __future__ import annotations

import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OBJ_DIR = os.path.join(HERE, "build")
LIB = os.path.join(HERE, "libfirework_b200.so")
STATIC_LIB = os.path.join(HERE, "libfirework_b200.a")
CLI = os.path.join(HERE, "bin", "firework")          # native driver (csrc/cli_main.cpp), links the static archive
LINK_LIBS = ["-lcudart_static", "-lz", "-ldl", "-lpthread", "-lrt"]   # zlib: PNG inflate / deflate (images.cpp), .yml.gz (cli)
SOURCES = ["api.cu", "multi_gpu.cu", "kernels_extend.cu", "kernels_walk.cu", "kernels_shade.cu", "kernels_probe.cu",
           "kernels_adaptive.cu", "kernels_denoise.cu", "scene_host.cpp", "yaml_lite.cpp", "formats.cpp", "images.cpp"]
HEADERS = ["fw_types.h", "scene_host.h", "yaml_lite.h", "device_math.cuh", "intersect.cuh", "shade.cuh", "wavefront.cuh",
           "wavefront_types.h", "launch.h", "api_internal.h", "walk.cuh", os.path.join("..", "..", "include", "firework_b200.h")]

NVCC_FLAGS = [
    "-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo",
    # Rust never contracts a*b+c; first-hit ids / t must match the reference's arithmetic (DESIGN.md).
    "--fmad=false",
    "-Xcompiler", "-fPIC", "-ccbin", "/usr/bin/g++",
]


def _sources():
    return [s for s in SOURCES if os.path.exists(os.path.join(CSRC, s))]


def _deps():
    return [os.path.join(CSRC, s) for s in _sources() + HEADERS + ["cli_main.cpp"] if os.path.exists(os.path.join(CSRC, s))] + [os.path.abspath(__file__)]


def needs_build(target: str = LIB) -> bool:
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in _deps())


def _obj_stale(src: str, obj: str) -> bool:
    """An object is rebuilt when its source, any header or this script changed (headers are shared by most units)."""
    if not os.path.exists(obj):
        return True
    t = os.path.getmtime(obj)
    hdrs = [os.path.join(CSRC, h) for h in HEADERS if os.path.exists(os.path.join(CSRC, h))]
    return any(os.path.getmtime(d) > t for d in [src, os.path.abspath(__file__)] + hdrs)


def build(force: bool = False, verbose: bool = False) -> str:
    out = os.environ.get("FW_LIB_OUT", LIB)
    extra = os.environ.get("FW_NVCC_EXTRA", "").split()
    variant = bool(extra) or out != LIB          # experiment builds get their own object directory
    obj_dir = OBJ_DIR + ("_" + os.path.splitext(os.path.basename(out))[0] if variant else "")
    if not force and not variant and not needs_build(LIB) and not needs_build(STATIC_LIB) and not needs_build(CLI):
        return LIB
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    os.makedirs(obj_dir, exist_ok=True)
    logs = []

    def compile_one(src_name: str):
        src = os.path.join(CSRC, src_name)
        obj = os.path.join(obj_dir, os.path.splitext(src_name)[0] + ".o")
        if not force and not _obj_stale(src, obj):
            return obj
        cmd = [nvcc] + NVCC_FLAGS + extra + (["-Xptxas", "-v"] if verbose else []) + ["-c", "-o", obj, src]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            sys.stderr.write(r.stdout + r.stderr)
            raise RuntimeError(f"nvcc failed compiling {src_name}")
        if verbose:
            logs.append(r.stderr)
        return obj

    with ThreadPoolExecutor(max_workers=min(8, os.cpu_count() or 1)) as ex:
        objs = list(ex.map(compile_one, _sources()))
    # -ldl: NCCL is bound at run time (multi_gpu.cu dlopens libnccl.so.2 when fw_render_multi is first called)
    # (linked with g++ directly: `nvcc -shared` would add a device-link stub compiled for its default sm_52)
    cuda_lib = os.path.join(os.path.dirname(os.path.dirname(nvcc)), "lib64")
    r = subprocess.run(["/usr/bin/g++", "-shared", "-o", out] + objs + ["-L" + cuda_lib] + LINK_LIBS,
                       capture_output=True, text=True)
    if r.returncode != 0:
        sys.stderr.write(r.stdout + r.stderr)
        raise RuntimeError("linking libfirework_b200.so failed")
    if not variant:
        if os.path.exists(STATIC_LIB):
            os.remove(STATIC_LIB)
        r = subprocess.run(["ar", "rcs", STATIC_LIB] + objs, capture_output=True, text=True)
        if r.returncode != 0:
            sys.stderr.write(r.stdout + r.stderr)
            raise RuntimeError("archiving libfirework_b200.a failed")
        # the native command-line driver: plain g++ against the static archive, exactly what a build.rs / Makefile would do
        os.makedirs(os.path.dirname(CLI), exist_ok=True)
        r = subprocess.run(["/usr/bin/g++", "-O2", "-std=c++17", "-o", CLI, os.path.join(CSRC, "cli_main.cpp"), STATIC_LIB, "-L" + cuda_lib] + LINK_LIBS,
                           capture_output=True, text=True)
        if r.returncode != 0:
            sys.stderr.write(r.stdout + r.stderr)
            raise RuntimeError("building the firework command-line driver failed")
    if verbose:
        print("\n".join(logs))
    return out


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
