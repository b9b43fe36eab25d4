"""ctypes binding of the C ABI in include/az_engine.h (libaz_engine.so, built in-tree by nvcc).

There is no fallback: if the library is missing or fails to load, `load()` raises.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

PKG_DIR = os.path.dirname(os.path.abspath(__file__))
REPO_ROOT = os.path.dirname(PKG_DIR)
CSRC = os.path.join(PKG_DIR, "csrc")
LIB_PATH = os.environ.get("AZ_ENGINE_LIB") or os.path.join(PKG_DIR, "libaz_engine.so")  # override: A/B builds of the library
SOURCES = ["az_engine.cu", "az_mlp.cu", "az_conv.cu", "az_resnet_pipe.cu", "az_resnet_wide.cu", "az_cnn.cu"]
HEADERS = ["az_eval.cuh", "c4_bitboard.cuh", "tcgen05.cuh", os.path.join("..", "..", "include", "az_engine.h")]

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
    "-fmad=false",  # fp64 PUCT must round every operation separately, like CPython
    "-shared", "-Xcompiler", "-fPIC",
]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if cand and (os.path.isabs(cand) and os.path.exists(cand) or not os.path.isabs(cand)):
            return cand
    return "nvcc"


def _stale() -> bool:
    if not os.path.exists(LIB_PATH):
        return True
    t = os.path.getmtime(LIB_PATH)
    deps = [os.path.join(CSRC, s) for s in SOURCES] + [os.path.normpath(os.path.join(CSRC, h)) for h in HEADERS]
    return any(os.path.exists(d) and os.path.getmtime(d) > t for d in deps)


def build_library(force: bool = False, verbose: bool = False) -> str:
    """nvcc -gencode arch=compute_100a,code=sm_100a ... -> alphazero-implementation_b200/libaz_engine.so"""
    if not force and not _stale():
        return LIB_PATH
    # one nvcc -c per source, in parallel (each takes 10-30 s), then one link
    objdir = os.path.join(PKG_DIR, "build")
    os.makedirs(objdir, exist_ok=True)
    compile_flags = [f for f in NVCC_FLAGS if f != "-shared"]
    jobs = []
    for src in SOURCES:
        obj = os.path.join(objdir, src.replace(".cu", ".o"))
        cmd = [_nvcc(), *compile_flags, "-c", "-o", obj, os.path.join(CSRC, src)]
        if verbose:
            cmd.insert(1, "-Xptxas=-v")
        jobs.append((cmd, obj, subprocess.Popen(cmd, cwd=CSRC, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True)))
    objs = []
    for cmd, obj, proc in jobs:
        out, err = proc.communicate()
        if proc.returncode != 0:
            raise RuntimeError(f"nvcc failed ({' '.join(cmd)}):\n{out}\n{err}")
        if verbose:
            print(err)
        objs.append(obj)
    link = [_nvcc(), "-gencode", "arch=compute_100a,code=sm_100a", "-shared", "-Xcompiler", "-fPIC", "-o", LIB_PATH, *objs]
    proc = subprocess.run(link, cwd=CSRC, capture_output=True, text=True)
    if proc.returncode != 0:
        raise RuntimeError(f"link failed ({' '.join(link)}):\n{proc.stdout}\n{proc.stderr}")
    return LIB_PATH


def library_available() -> bool:
    return os.path.exists(LIB_PATH)


class AzConfig(C.Structure):
    _fields_ = [
        ("height", C.c_int32), ("width", C.c_int32), ("count", C.c_int32), ("num_games", C.c_int32),
        ("num_simulations", C.c_int32), ("device", C.c_int32), ("lanes_per_tree", C.c_int32), ("hot_nodes_plus1", C.c_int32),
        ("c_puct", C.c_double),
    ]


class AzStats(C.Structure):
    _fields_ = [(n, C.c_uint64) for n in ("simulations", "evaluations", "levels", "children_created", "backup_nodes",
                                           "moves", "episodes", "children_scanned")]


class AzEvalCacheStats(C.Structure):
    _fields_ = [(n, C.c_uint64) for n in ("rows", "hits", "followers", "failed_claims", "evictions")]


class AzRootNoise(C.Structure):
    _fields_ = [("alpha", C.c_double), ("fraction", C.c_float), ("seed", C.c_uint64), ("slot_offset", C.c_int64)]


class AzReuseStats(C.Structure):
    _fields_ = [(n, C.c_uint64) for n in ("retained", "fresh", "dropped", "nodes", "visits")]


class AzPlayoutCap(C.Structure):
    _fields_ = [("fast_sims", C.c_int32), ("p_full", C.c_float), ("seed", C.c_uint64), ("slot_offset", C.c_int64),
                ("visit_budget", C.c_int32)]


class AzCapStats(C.Structure):
    _fields_ = [(n, C.c_uint64) for n in ("full_searches", "fast_searches", "samples_recorded", "samples_dropped", "simulations")]


class AzResnetDesc(C.Structure):
    _fields_ = [
        ("num_blocks", C.c_int32), ("num_channels", C.c_int32), ("operand_format", C.c_int32), ("variant", C.c_int32),
        ("trunk_w", C.c_void_p), ("trunk_b", C.c_void_p), ("head_conv_w", C.c_void_p), ("head_conv_b", C.c_void_p),
        ("fc_policy_w", C.c_void_p), ("fc_policy_b", C.c_void_p), ("fc_value_w", C.c_void_p), ("fc_value_b", C.c_void_p),
    ]


class AzCnnDesc(C.Structure):
    _fields_ = [
        ("operand_format", C.c_int32), ("reserved", C.c_int32), ("conv_w", C.c_void_p), ("conv_b", C.c_void_p), ("fc_w", C.c_void_p),
        ("fc_b", C.c_void_p), ("head_w", C.c_void_p), ("head_b", C.c_void_p), ("workspace", C.c_void_p), ("workspace_bytes", C.c_int64),
    ]


FMT_BF16, FMT_F16 = 0, 1

P = C.c_void_p  # device pointers and streams cross the boundary as plain addresses
I32, I64 = C.c_int32, C.c_int64

# name -> (restype, argtypes); the single source of truth for tests/test_abi.py as well
SIGNATURES = {
    "az_abi_version": (I32, []),
    "az_last_error": (C.c_char_p, [P]),
    "az_create": (I32, [C.POINTER(AzConfig), C.POINTER(P)]),
    "az_destroy": (I32, [P]),
    "az_device_bytes": (I64, [P]),
    "az_device": (I32, [P]),
    "az_env_step": (I32, [P, P, P, P, P, I64, P, P, P, P, P, P, P, P]),
    "az_state_info": (I32, [P, P, P, P, I64, P, P, P, P]),
    "az_masked_softmax": (I32, [P, P, P, I64, P, P]),
    "az_encode_states": (I32, [P, P, P, P, I64, P, I32, P]),
    "az_reset_games": (I32, [P, C.c_uint64, C.c_uint64, I32, P]),
    "az_set_roots": (I32, [P, P, P, P, I32, P]),
    "az_run_simulations": (I32, [P, I32, I32, P]),
    "az_run_move_step": (I32, [P, I32, I32, P, P, P]),
    "az_select_leaves": (I32, [P, P]),
    "az_gather_leaves": (I32, [P, P, I32, P]),
    "az_expand_backup": (I32, [P, P, P, I32, P]),
    "az_expand_backup_select": (I32, [P, P, P, I32, P]),
    "az_leaf_info": (I32, [P, P, P, P, P, P, P]),
    "az_root_stats": (I32, [P, P, P, P, P, P, P, P, P]),
    "az_tree_capacity": (I32, [P]),
    "az_export_tree": (I32, [P, I32, P, P, P, P, C.POINTER(I32)]),
    "az_sample_moves": (I32, [P, P, P, P]),
    "az_episode_counts": (I32, [P, C.POINTER(I64), C.POINTER(I64), P]),
    "az_drain_episodes": (I32, [P, I64, I64, P, P, P, P, P, P, P, P, P, C.POINTER(I64), C.POINTER(I64), P]),
    "az_swap_episode_ring": (I32, [P, C.POINTER(I32), P]),
    "az_ring_counts": (I32, [P, I32, C.POINTER(I64), C.POINTER(I64), P]),
    "az_read_episode_ring": (I32, [P, I32, I64, I64, P, P, P, P, P, P, P, P, P, P]),
    "az_get_stats": (I32, [P, C.POINTER(AzStats), P]),
    "az_reset_stats": (I32, [P, P]),
    "az_selftest_division": (I32, [P, I64, C.c_uint64, C.POINTER(I64)]),
    "az_launch_count": (I64, [P]),
    "az_mlp_create": (I32, [I32, C.POINTER(P)]),
    "az_mlp_destroy": (I32, [P]),
    "az_mlp_last_error": (C.c_char_p, [P]),
    "az_mlp_set_operand_format": (I32, [P, I32]),
    "az_mlp_set_weights": (I32, [P, P, P, P, P, P, P, P, P, P]),
    "az_mlp_forward": (I32, [P, P, I64, P, P, P]),
    "az_mlp_forward_leaves": (I32, [P, P, P, P, P]),
    "az_mlp_launch_count": (I64, [P]),
    "az_leaf_players": (I32, [P, C.POINTER(P)]),
    "az_leaf_compact": (I32, [P, C.POINTER(P), C.POINTER(P)]),
    "az_set_leaf_compaction": (I32, [P, I32]),
    "az_set_eval_cache": (I32, [P, I32]),
    "az_bump_eval_epoch": (I32, [P, P]),
    "az_get_eval_cache_stats": (I32, [P, C.POINTER(AzEvalCacheStats), P]),
    "az_set_root_noise": (I32, [P, C.POINTER(AzRootNoise)]),
    "az_apply_root_noise": (I32, [P, P]),
    "az_root_noise_values": (I32, [P, P, P]),
    "az_set_greedy_from": (I32, [P, I32]),
    "az_set_symmetric_eval": (I32, [P, I32]),
    "az_set_subtree_reuse": (I32, [P, I32]),
    "az_advance_roots": (I32, [P, P, P, P]),
    "az_get_reuse_stats": (I32, [P, C.POINTER(AzReuseStats), P]),
    "az_set_playout_cap": (I32, [P, C.POINTER(AzPlayoutCap)]),
    "az_search_budgets": (I32, [P, P, P, P]),
    "az_get_cap_stats": (I32, [P, C.POINTER(AzCapStats), P]),
    "az_leaf_mirror": (I32, [P, C.POINTER(P)]),
    "az_mirror_states": (I32, [P, P, P, P, I64, P, P, P]),
    "az_trunk_weight_bytes": (I64, [I32]),
    "az_resnet_pipe_weight_bytes": (I64, [I32, I32]),
    "az_trunk_forward_leaves": (I32, [P, P, P, I32, P, P]),
    "az_resnet_forward_leaves": (I32, [P, P, P, I32, P, P, P, P, P, P, P, P, P]),
    "az_resnet_forward_leaves_v2": (I32, [P, C.POINTER(AzResnetDesc), P, P, P]),
    "az_trunk_set_cta_pair": (I32, [I32]),
    "az_resnet_wide_set_timing": (I32, [P, I32]),
    "az_cnn_conv_weight_bytes": (I64, []),
    "az_cnn_fc_weight_bytes": (I64, []),
    "az_cnn_workspace_bytes": (I64, [I64]),
    "az_cnn_forward_leaves": (I32, [P, C.POINTER(AzCnnDesc), P, P, P]),
    "az_leaf_arrays": (I32, [P, C.POINTER(P), C.POINTER(P), C.POINTER(P), C.POINTER(I32)]),
}

_lib = None


def load() -> C.CDLL:
    """Load libaz_engine.so.  Raises if it has not been built: there is no CPU path."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(nvcc, sm_100a).  This package has no CPU or PyTorch fallback."
        )
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the symbol is missing
        fn.restype = res
        fn.argtypes = args
    if lib.az_abi_version() != 1:
        raise RuntimeError(f"libaz_engine.so ABI version {lib.az_abi_version()} != 1; rebuild")
    _lib = lib
    return lib
