"""ctypes binding of libcemk.so (include/cemk.h).  No CPU fallback: a missing library is an error."""
from __future__ import annotations

import ctypes as C
import os
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
# CEMK_LIB_PATH: A/B tools point this at a prebuilt variant under build_variants/ (never set by the product path)
LIB_PATH = os.environ.get("CEMK_LIB_PATH") or os.path.join(_HERE, "libcemk.so")
SRC = [os.path.join(_HERE, "csrc", n) for n in ("cemk.cu", "rollout_core.h", "warp_dsl.h", "kmodel.h")]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17", "-DCEMK_STEP_SYNC", "-DCEMK_PHASE_SYNC=18",
              "-use_fast_math", "-shared", "-Xcompiler", "-fPIC"]


def build_library(force=False, verbose=False):
    """nvcc cross-compile of csrc/cemk.cu for sm_100a into the package directory (in-tree)."""
    hdr = os.path.join(_HERE, "..", "include", "cemk.h")
    deps = SRC + [hdr]
    fresh = os.path.exists(LIB_PATH) and all(os.path.getmtime(LIB_PATH) >= os.path.getmtime(p) for p in deps)
    if fresh and not force:
        return LIB_PATH
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    cmd = [nvcc] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-o", LIB_PATH, SRC[0]]
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("nvcc failed:\n" + res.stdout + res.stderr)
    if verbose:
        print(res.stderr)
    return LIB_PATH


_lib = None

_vp, _i, _f = C.c_void_p, C.c_int, C.c_float
_SIGS = {
    "cemk_version": ([], _i),
    "cemk_last_error": ([], C.c_char_p),
    "cemk_sizeof_kmodel": ([], _i),
    "cemk_create": ([_vp, _i, _i, C.POINTER(_vp)], _i),
    "cemk_destroy": ([_vp], _i),
    "cemk_set_model": ([_vp, _vp, _i], _i),
    "cemk_set_dof": ([_vp, _i], _i),
    "cemk_set_order": ([_vp, _i], _i),
    "cemk_set_horizon": ([_vp, _i, _vp, _vp, _vp, _vp], _i),
    "cemk_sample": ([_vp, _i, _vp, _vp, _vp, _vp, _vp, _vp], _i),
    "cemk_jax_normal": ([_vp, C.c_uint, C.c_uint, _i, C.c_uint, C.c_uint, C.c_uint, _vp, _vp], _i),
    "cemk_project": ([_vp, _i, _i, _vp, _vp, _vp, _vp, _vp], _i),
    "cemk_rollout_cost": ([_vp, _i, _i, _vp, _vp, _vp, _vp, _vp, _f, _f, _f, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp], _i),
    "cemk_step_states": ([_vp, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp], _i),
    "cemk_cost_batch": ([_vp, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _f, _f, _f, _vp, _vp], _i),
    "cemk_argsort_topk": ([_vp, _i, _vp, _i, _i, _vp, _vp, _i, _vp, _vp, _vp, _vp], _i),
    "cemk_topk_pack": ([_vp, _i, _vp, _i, _i, _vp, _i, _vp, _vp, _vp], _i),
    "cemk_merge_sorted_lists": ([_vp, _i, _i, _vp, _i, _vp, _vp, _vp, _vp], _i),
    "cemk_mean_cov": ([_vp, _i, _vp, _vp, _vp, _vp, _f, _f, _f, _vp, _vp, _vp], _i),
    "cemk_set_option": ([_vp, C.c_char_p, _i], _i),
    "cemk_fp32_fma_peak": ([_vp, C.POINTER(C.c_double)], _i),
    "cemk_tick_record": ([_vp, _i, _i, _i, _i, _i, _vp, _vp, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp], _i),
    "cemk_launch_count": ([_vp], C.c_longlong),
}
EXPORTS = tuple(_SIGS)


def load():
    """Load libcemk.so and declare every prototype of include/cemk.h.  Raises if it is missing."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(nvcc, sm_100a).  There is no CPU fallback for the planner.")
    lib = C.CDLL(LIB_PATH)
    for name, (args, ret) in _SIGS.items():
        fn = getattr(lib, name)
        fn.argtypes, fn.restype = args, ret
    _lib = lib
    return lib


def check(status, lib=None):
    if status != 0:
        lib = lib or load()
        raise RuntimeError(f"libcemk error {status}: {lib.cemk_last_error().decode()}")
