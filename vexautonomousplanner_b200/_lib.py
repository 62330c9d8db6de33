"""Loader for libvap.so (the sm_100a CUDA engine behind include/vap.h).

There is no CPU fallback: if the shared library is missing or cannot be loaded the product raises.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
SO_PATH = os.environ.get("VAP_LIB_PATH") or os.path.join(_HERE, "libvap.so")   # VAP_LIB_PATH: A/B builds of the engine
SRC_DIR = os.path.join(_HERE, "csrc")
SOURCES = ["vap_kernels.cu"]
HEADER = os.path.join(os.path.dirname(_HERE), "include", "vap.h")

NVCC_FLAGS = os.environ.get("VAP_NVCC_EXTRA", "").split() + ["-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo",
              "-fmad=false",            # load-bearing: the reference never fuses multiply-add
              "-Xcompiler", "-fPIC", "-shared"]

# every symbol include/vap.h declares (tests check the list against the header and the .so)
SYMBOLS = [
    "vap_version", "vap_last_error", "vap_build_path", "vap_fit_splines", "vap_eval", "vap_build_lut",
    "vap_lut_index_row_ints", "vap_build_lut_index", "vap_build_props", "vap_query_tables", "vap_build_dgrid", "vap_dist_sample", "vap_fwd_bwd", "vap_resample",
    "vap_gl", "vap_turn_profile", "vap_lerp", "vap_wheel_trajectory",
    "vap_event_scratch_ints", "vap_pass_row_slots", "vap_velocity_profile", "vap_time_profile", "vap_workspace_bytes", "vap_profile_batch", "vap_summary", "vap_pack_rows", "vap_export_rows", "vap_format_doubles", "vap_row_text_stride",
    "vap_format_rows", "vap_compact_rows", "vap_splice_plan", "vap_splice_actions", "vap_row_kinds",
    "vap_parse_doubles", "vap_line_starts", "vap_line_offsets", "vap_line_kinds", "vap_parse_rows", "vap_compare_bodies",
    "vap_footprint_check", "vap_pose_planes", "vap_pair_check",
"vap_bench_dfma", "vap_test_div_const", "vap_test_div_recip", "vap_build_lerp_recip", "vap_diag_read",
]

_lib = None


class VapError(RuntimeError):
    pass


def build(force: bool = False, verbose: bool = False) -> str:
    """Compile the CUDA engine in-tree for sm_100a (nvcc cross-compiles without a GPU)."""
    srcs = [os.path.join(SRC_DIR, s) for s in SOURCES]
    deps = srcs + [os.path.join(SRC_DIR, f) for f in os.listdir(SRC_DIR) if f.endswith(".cuh")] + [HEADER]
    if not force and os.path.exists(SO_PATH) and all(os.path.getmtime(SO_PATH) >= os.path.getmtime(d) for d in deps):
        return SO_PATH
    nvcc = os.environ.get("NVCC", "nvcc")
    cmd = [nvcc] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-o", SO_PATH] + srcs
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise VapError("nvcc failed:\n" + r.stdout + r.stderr)
    if verbose:
        print(r.stderr)
    return SO_PATH


def lib():
    """ctypes handle of libvap.so; raises VapError when the extension has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(SO_PATH):
            raise VapError(f"{SO_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                           "(there is no CPU fallback)")
        L = C.CDLL(SO_PATH)
        L.vap_version.restype = C.c_int
        L.vap_last_error.restype = C.c_char_p
        for name in SYMBOLS[2:]:
            getattr(L, name).restype = C.c_int
        L.vap_event_scratch_ints.restype = C.c_int64
        L.vap_pass_row_slots.restype = C.c_int64
        L.vap_lut_index_row_ints.restype = C.c_int64
        L.vap_workspace_bytes.restype = C.c_int64
        _lib = L
    return _lib


def check(rc: int, what: str = "") -> None:
    if rc != 0:
        raise VapError(f"{what}: {lib().vap_last_error().decode()} (rc={rc})")
