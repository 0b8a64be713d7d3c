"""ctypes front-end for the connected-components oracle (TEST INFRASTRUCTURE ONLY).

Only ``tests/`` may import this module; the product package never does
(tests/test_no_oracle_in_product.py enforces it). It compiles ``components_oracle.cpp``
(the reference's ComputeConnectedComponents, topology_computation.hpp:138-196, restated) into
``oracle/_build/libvgt_components_oracle.so`` when that is missing or older than the source.
"""
from __future__ import annotations

import ctypes
import hashlib
import os
import shutil
import subprocess
from pathlib import Path

import numpy as np

_HERE = Path(__file__).resolve().parent
_SOURCE = _HERE / "components_oracle.cpp"
_LIB_PATH = _HERE / "_build" / "libvgt_components_oracle.so"
_STAMP_PATH = _HERE / "_build" / "libvgt_components_oracle.stamp"


def _compiler() -> str:
    # (the system compiler, as oracle/Makefile picks it)
    return "/usr/bin/g++" if os.access("/usr/bin/g++", os.X_OK) else (shutil.which("g++") or "g++")


def build(force: bool = False) -> Path:
    """Compiles the oracle if needed; returns the .so path."""
    stamp = hashlib.sha1(_SOURCE.read_bytes()).hexdigest()
    if (not force and _LIB_PATH.exists() and _STAMP_PATH.exists()
            and _STAMP_PATH.read_text().strip() == stamp):
        return _LIB_PATH
    _LIB_PATH.parent.mkdir(exist_ok=True)
    partial = _LIB_PATH.with_name(f"{_LIB_PATH.name}.{os.getpid()}")
    subprocess.run([_compiler(), "-std=c++17", "-O2", "-fPIC", "-Wall", "-Wextra", "-shared",
                    "-o", str(partial), str(_SOURCE)], check=True, capture_output=True)
    os.replace(partial, _LIB_PATH)
    _STAMP_PATH.write_text(stamp)
    return _LIB_PATH


_lib = None


def lib() -> ctypes.CDLL:
    global _lib
    if _lib is None:
        handle = ctypes.CDLL(str(build()))
        handle.vgt_oracle_connected_components.argtypes = [
            ctypes.c_void_p, ctypes.c_int, ctypes.c_int64, ctypes.c_int64, ctypes.c_int64,
            ctypes.POINTER(ctypes.c_uint32)]
        handle.vgt_oracle_connected_components.restype = ctypes.c_int
        _lib = handle
    return _lib


def connected_components(cells):
    """ComputeConnectedComponents (topology_computation.hpp:138-196) as the component maps call
    it, by the reference's serial scan and breadth-first fill, on a COPY of `cells` (a structured
    [nx, ny, nz] array of 8-byte {occupancy, component} or 16-byte {occupancy, object_id,
    component, spatial_segment} cells). Returns (the labelled copy, the number of components)."""
    labelled = np.array(cells, copy=True, order="C")
    if labelled.ndim != 3 or labelled.dtype.itemsize not in (8, 16):
        raise ValueError("cells must be an [nx, ny, nz] array of 8- or 16-byte cells")
    count = ctypes.c_uint32()
    code = lib().vgt_oracle_connected_components(
        labelled.ctypes.data, labelled.dtype.itemsize, *labelled.shape, ctypes.byref(count))
    if code != 0:
        raise RuntimeError(f"oracle connected components failed with code {code}")
    return labelled, int(count.value)
