"""Builds (nvcc, sm_100a) and loads the C-ABI shared library ``lib/libyinyang_b200.so``.

The library is the product; this module only binds it with ctypes (signatures mirror
``include/yinyang_b200.h``).  There is no CPU fallback: if the library cannot be built or loaded,
or no CUDA device is present, compute calls raise.
"""
from __future__ import annotations

import ctypes
import os
import subprocess
from concurrent.futures import ThreadPoolExecutor

_HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(_HERE, "csrc")
LIB_DIR = os.path.join(_HERE, "lib")
LIB_PATH = os.path.join(LIB_DIR, "libyinyang_b200.so")
HEADER = os.path.join(os.path.dirname(_HERE), "include", "yinyang_b200.h")
SOURCES = ["yy_rules_kernels.cu", "yy_tree.cu", "yy_probe.cu", "yy_nn.cu", "yy_fused.cu", "yy_dataset.cu", "yy_learn.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17", "-fmad=false",
              "-Xcompiler", "-fPIC", "-diag-suppress", "177"]


def _stale() -> bool:
    if not os.path.exists(LIB_PATH):
        return True
    t = os.path.getmtime(LIB_PATH)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [HEADER]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False) -> str:
    """Compile every .cu for sm_100a and link the shared library in-tree (cross-compiles without a GPU)."""
    if not force and not _stale():
        return LIB_PATH
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    os.makedirs(LIB_DIR, exist_ok=True)
    # One builder at a time (torchrun starts every rank at once on a fresh checkout): the others wait on the lock and then
    # find the library up to date.  Objects and the library are written under temporary names and renamed into place, so
    # nobody ever dlopens a half-written file.
    import fcntl
    with open(os.path.join(LIB_DIR, ".build.lock"), "w") as lock:
        fcntl.flock(lock, fcntl.LOCK_EX)
        try:
            if not force and not _stale():
                return LIB_PATH
            return _build_locked(nvcc, verbose)
        finally:
            fcntl.flock(lock, fcntl.LOCK_UN)


def _build_locked(nvcc, verbose):
    objdir = os.path.join(LIB_DIR, "obj")
    os.makedirs(objdir, exist_ok=True)

    def one(src):
        obj = os.path.join(objdir, src.replace(".cu", ".o"))
        tmp = obj + f".tmp{os.getpid()}"
        cmd = [nvcc, *NVCC_FLAGS, "-c", os.path.join(CSRC, src), "-o", tmp]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"nvcc failed for {src}:\n{r.stdout}\n{r.stderr}")
        if verbose and r.stderr:
            print(r.stderr)
        os.replace(tmp, obj)
        return obj

    with ThreadPoolExecutor(max_workers=len(SOURCES)) as ex:
        objs = list(ex.map(one, SOURCES))
    tmp = LIB_PATH + f".tmp{os.getpid()}"
    r = subprocess.run([nvcc, "-shared", "-o", tmp, *objs], capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"link failed:\n{r.stdout}\n{r.stderr}")
    os.replace(tmp, LIB_PATH)
    return LIB_PATH


class EngineConfig(ctypes.Structure):
    """yy_engine_config (include/yinyang_b200.h)."""
    _fields_ = [
        ("rows", ctypes.c_int32), ("cols", ctypes.c_int32), ("n_games", ctypes.c_int32), ("n_sims", ctypes.c_int32),
        ("rule_flags", ctypes.c_uint32), ("mode_flags", ctypes.c_uint32), ("evaluator", ctypes.c_int32),
        ("edges_per_game", ctypes.c_int32), ("temperature_threshold", ctypes.c_int32),
        ("replay_capacity", ctypes.c_int32), ("nn_channels", ctypes.c_int32), ("nn_blocks", ctypes.c_int32),
        ("device", ctypes.c_int32), ("leaves_per_step", ctypes.c_int32), ("cpuct", ctypes.c_float), ("descents_per_step", ctypes.c_int32),
        ("dirichlet_alpha", ctypes.c_double),
        ("dirichlet_epsilon", ctypes.c_double), ("seed", ctypes.c_uint64),
    ]


class SelfPlayStats(ctypes.Structure):
    _fields_ = [("moves", ctypes.c_int64), ("evals", ctypes.c_int64), ("games_finished", ctypes.c_int64),
                ("examples", ctypes.c_int64), ("sims", ctypes.c_int64), ("overflow", ctypes.c_int32),
                ("max_depth", ctypes.c_int32), ("tower_evals", ctypes.c_int64)]


class GemmStats(ctypes.Structure):
    """yy_gemm_stats (include/yinyang_b200.h)."""
    _fields_ = [("sums", ctypes.c_void_p), ("out", ctypes.c_void_p), ("ldo", ctypes.c_int32), ("y", ctypes.c_void_p),
                ("ldy", ctypes.c_int32), ("mean_invstd", ctypes.c_void_p)]


class ConvGeom(ctypes.Structure):
    """yy_conv_geom (include/yinyang_b200.h)."""
    _fields_ = [("rows", ctypes.c_int32), ("cols", ctypes.c_int32), ("cin", ctypes.c_int32), ("flip", ctypes.c_int32)]


class TreeView(ctypes.Structure):
    """yy_tree_view (include/yinyang_b200.h)."""
    _fields_ = [("max_nodes", ctypes.c_int32), ("edges_cap", ctypes.c_int32), ("W", ctypes.c_int32),
                ("n_nodes", ctypes.c_void_p), ("n_edges_used", ctypes.c_void_p), ("node_black", ctypes.c_void_p),
                ("node_white", ctypes.c_void_p), ("node_edge_base", ctypes.c_void_p), ("node_n_edges", ctypes.c_void_p),
                ("node_player", ctypes.c_void_p), ("node_flags", ctypes.c_void_p), ("node_value", ctypes.c_void_p),
                ("edge_N", ctypes.c_void_p), ("edge_W", ctypes.c_void_p), ("edge_P", ctypes.c_void_p),
                ("edge_child_meta", ctypes.c_void_p), ("edge_action", ctypes.c_void_p)]


class ReplayView(ctypes.Structure):
    _fields_ = [("black", ctypes.c_void_p), ("white", ctypes.c_void_p), ("counts", ctypes.c_void_p),
                ("game_serial", ctypes.c_void_p), ("ply", ctypes.c_void_p), ("player", ctypes.c_void_p),
                ("results", ctypes.c_void_p), ("results_capacity", ctypes.c_int32)]


_P = ctypes.c_void_p
_I = ctypes.c_int
_I64 = ctypes.c_int64
_U32 = ctypes.c_uint32
_F = ctypes.c_float

# name -> (restype, argtypes); every symbol include/yinyang_b200.h declares
SIGNATURES = {
    "yy_abi_version": (_I, []),
    "yy_last_error": (ctypes.c_char_p, []),
    "yy_device_count": (_I, []),
    "yy_launch_count": (_I64, []),
    "yy_legal_mask": (_I, [_I, _I, _U32, _P, _P, _P, _P, _I64, _P]),
    "yy_step": (_I, [_I, _I, _U32, _P, _P, _P, _P, _I64, _P]),
    "yy_ended": (_I, [_I, _I, _U32, _P, _P, _P, _P, _I64, _P]),
    "yy_env_step": (_I, [_I, _I, _U32, _P, _P, _P, _P, _P, _P, _I64, _P]),
    "yy_pack_boards": (_I, [_I, _I, _P, _P, _P, _I64, _P]),
    "yy_unpack_boards": (_I, [_I, _I, _P, _P, _P, _P, _P, _I64, _P]),
    "yy_random_playout": (_I, [_I, _I, _U32, ctypes.c_uint64, _P, _P, _P, _P, _I64, _P]),
    "yy_engine_workspace_bytes": (_I64, [ctypes.POINTER(EngineConfig)]),
    "yy_engine_create": (_P, [ctypes.POINTER(EngineConfig), _P, _I64]),
    "yy_engine_destroy": (None, [_P]),
    "yy_nn_weight_bytes": (_I64, [_I, _I, _I, _I]),
    "yy_nn_weight_layout": (_I, [_I, _I, _I, _I, ctypes.POINTER(_I64)]),
    "yy_engine_load_weights": (_I, [_P, _P, _I64]),
    "yy_search": (_I, [_P, _P, _P, _P, _P, _P, _P, _P]),
    "yy_search_begin": (_I, [_P, _P, _P, _P, _P, _P, _P]),
    "yy_search_advance": (_I, [_P, _P, _P, ctypes.POINTER(ctypes.c_int32), _P]),
    "yy_search_counts": (_I, [_P, _P, _P, _P]),
    "yy_engine_tree_view": (_I, [_P, ctypes.POINTER(TreeView)]),
    "yy_engine_leaf_black": (_P, [_P]),
    "yy_engine_leaf_white": (_P, [_P]),
    "yy_engine_leaf_active": (_P, [_P]),
    "yy_evaluate": (_I, [_P, _P, _P, _I64, _P, _P, _P, _P]),
    "yy_evaluate_form": (_I, [_P, _P, _P, _I64, ctypes.c_int32, _P, _P, _P, _P]),
    "yy_engine_set_profiling": (_I, [_P, _I]),
    "yy_engine_get_profile": (_I, [_P, ctypes.POINTER(_I64), ctypes.POINTER(ctypes.c_double), ctypes.POINTER(_I64)]),
    "yy_engine_set_debug_stamps": (_I, [_P, _P]),
    "yy_engine_set_debug_flags": (_I, [_P, _I]),
    "yy_selfplay_reset": (_I, [_P, _P]),
    "yy_selfplay_run": (_I, [_P, ctypes.c_int32, _P]),
    "yy_selfplay_advance": (_I, [_P, _I64, _P]),
    "yy_selfplay_set_quota": (_I, [_P, _I64]),
    "yy_selfplay_set_random_stream": (_I, [_P, _P, _P, ctypes.c_int32, ctypes.c_int32]),
    "yy_selfplay_set_playout_cap": (_I, [_P, ctypes.c_double, ctypes.c_int32]),
    "yy_arena_run": (_I, [_P, _P, _I64, _P, _P, _P, _P, ctypes.c_int32, _P, _P, _P]),
    "yy_selfplay_get_stats": (_I, [_P, ctypes.POINTER(SelfPlayStats), _P]),
    "yy_selfplay_replay": (_I, [_P, ctypes.POINTER(ReplayView)]),
    "yy_selfplay_stats_dev": (_P, [_P]),
    "yy_engine_game_black": (_P, [_P]),
    "yy_engine_game_white": (_P, [_P]),
    "yy_engine_game_player": (_P, [_P]),
    "yy_augment_samples": (_I, [_I, _I, _P, _P, _P, _P, _P, _I64, _P, _P, _P, _P]),
    "yy_dataset_samples": (_I, [_I, _I, _P, _P, _P, _P, _P, _I64, _P, _P, _P, _P]),
    "yy_lrn_gemm": (_I, [_P, _I, _I, _P, _I, _I, _P, _I, _I, _I, _I, _P, _I, _I, _I, _I, _P, _I64, _I, _P, _P, _P, _P]),
    "yy_lrn_pack_b": (_I, [_P, _P, _I64, _I, _I, _I, _P, _P]),
    "yy_lrn_pack_b_bytes": (_I64, [_I, _I]),
    "yy_lrn_gemm_debug_stamps": (_I, [_P]),
    "yy_lrn_transpose": (_I, [_P, _I, _P, _I, _I, _I, _I, _I64, _I64, _P]),
    "yy_lrn_im2col_t": (_I, [_P, _I, _P, _I, _I64, _I, _I, _I, _P]),
    "yy_lrn_conv_weight_t": (_I, [_P, _P, _I, _P, _I, _I, _P]),
    "yy_lrn_planes_nhwc": (_I, [_P, _P, _I64, _I, _P]),
    "yy_lrn_colsum": (_I, [_P, _I, _I, _I, _P, _P]),
    "yy_lrn_bn_forward": (_I, [_P, _I, _I, _I, _P, _P, _P, _I, _P, _I, _I, _F, _F, _P, _I, _P, _P, _P, _P]),
    "yy_lrn_bn_backward": (_I, [_P, _I, _P, _I, _P, _I, _I, _I, _P, _P, _P, _P, _I, _P, _I, _P, _P, _P, _P, _I, _I, _P]),
    "yy_lrn_heads_loss": (_I, [_P, _I, _P, _I, _P, _I, _I, _P, _P, _P, _I, _P, _I, _P, _I, _P, _P, _P, _P, _P, _P]),
    "yy_lrn_adam": (_I, [_P, _P, _P, _P, _I64, _F, _F, _F, _F, _F, _P, _P]),
    "yy_probe_tf32_mn": (_I, [_P, _P, _P, _I, _I, _I, _P]),
    "yy_probe_umma": (_I, [_P, _P, _P, _I, _I, _I, _I, _I, _P]),
}

_lib = None


def lib() -> ctypes.CDLL:
    """Load (building first if stale) the shared library and attach signatures."""
    global _lib
    if _lib is None:
        path = build()
        L = ctypes.CDLL(path)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(L, name)
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib


class YinYangError(RuntimeError):
    pass


def check(rc: int) -> None:
    if rc != 0:
        msg = lib().yy_last_error()
        raise YinYangError(f"yinyang_b200 error {rc}: {msg.decode() if msg else ''}")
