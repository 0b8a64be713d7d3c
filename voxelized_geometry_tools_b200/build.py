"""In-tree nvcc build of libvgt_b200.so (the C-ABI shared library, sm_100a only).

    python -m voxelized_geometry_tools_b200.build [--force] [--verbose]

The library lands next to this file so it travels with the repo snapshot to the GPU box.
nvcc cross-compiles without a GPU, so this also runs in the CPU-only dev container.
"""
from __future__ import annotations

import hashlib
import os
import shutil
import subprocess
import sys
from pathlib import Path

PACKAGE_DIR = Path(__file__).resolve().parent
CSRC = PACKAGE_DIR / "csrc"
INCLUDE = PACKAGE_DIR.parent / "include"
LIBRARY = PACKAGE_DIR / "libvgt_b200.so"
_OBJ_DIR = PACKAGE_DIR / "_obj"
_STAMP = _OBJ_DIR / "sources.sha1"

ARCH_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a"]
COMMON_FLAGS = ["-std=c++17", "-O3", "-lineinfo", "-Xcompiler", "-fPIC,-fvisibility=hidden",
                "-I", str(INCLUDE)]

# (source, extra flags). The voxelizer must not contract a*b+c into FMA: its DDA reproduces the
# double-precision CPU path bit for bit (see csrc/voxelizer_kernels.cu).
TRANSLATION_UNITS = [
    ("capi_common.cu", []),
    ("edt_kernels.cu", []),
    ("voxelizer_kernels.cu", ["-fmad=false"]),
    # the SDF queries evaluate the reference's double expressions as written
    ("sdf_queries.cu", ["-fmad=false"]),
    # the mesh rasterizer's "cell touched" test is a double comparison mirrored as written
    ("mesh_rasterizer.cu", ["-fmad=false"]),
    # the reference's file formats (host code; zlib for the compressed forms)
    ("grid_files.cu", []),
    # connected components of the component maps (union-find labelling)
    ("connected_components.cu", []),
]


def _nvcc() -> str:
    for candidate in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", shutil.which("nvcc")):
        if candidate and Path(candidate).exists():
            return candidate
    raise RuntimeError("nvcc not found; cannot build libvgt_b200.so")


def _host_compiler_flags() -> list[str]:
    # The image exports CXX=/opt/gcc/bin/g++ (a wrapper); nvcc wants the system g++.
    if Path("/usr/bin/g++").exists():
        return ["-ccbin", "/usr/bin/g++"]
    return []


def _sources_signature() -> str:
    digest = hashlib.sha1()
    for path in sorted(list(CSRC.glob("*.cu")) + list(CSRC.glob("*.cuh")) + list(INCLUDE.glob("*.h"))
                       + [Path(__file__)]):
        digest.update(path.name.encode())
        digest.update(path.read_bytes())
    return digest.hexdigest()


def build(force: bool = False, verbose: bool = False) -> Path:
    signature = _sources_signature()
    if (not force and LIBRARY.exists() and _STAMP.exists()
            and _STAMP.read_text().strip() == signature):
        return LIBRARY
    nvcc = _nvcc()
    _OBJ_DIR.mkdir(exist_ok=True)
    objects = []
    for source, extra in TRANSLATION_UNITS:
        obj = _OBJ_DIR / (Path(source).stem + ".o")
        command = ([nvcc] + _host_compiler_flags() + ARCH_FLAGS + COMMON_FLAGS + extra
                   + (["-Xptxas", "-v"] if verbose else [])
                   + ["-c", str(CSRC / source), "-o", str(obj)])
        result = subprocess.run(command, capture_output=True, text=True)
        if verbose or result.returncode != 0:
            sys.stderr.write(" ".join(command) + "\n" + result.stdout + result.stderr)
        if result.returncode != 0:
            raise RuntimeError(f"nvcc failed on {source}")
        objects.append(str(obj))
    link = ([nvcc] + _host_compiler_flags() + ARCH_FLAGS + ["-shared", "-o", str(LIBRARY)]
            + objects + ["-lz"])
    result = subprocess.run(link, capture_output=True, text=True)
    if result.returncode != 0:
        sys.stderr.write(" ".join(link) + "\n" + result.stdout + result.stderr)
        raise RuntimeError("nvcc link failed")
    _STAMP.write_text(signature)
    return LIBRARY


if __name__ == "__main__":
    path = build(force="--force" in sys.argv, verbose="--verbose" in sys.argv)
    print(path)
