"""TEST INFRASTRUCTURE — ctypes wrapper of tests/native/c4_openings_oracle.c: the forced-playouts oracle (which includes the cap,
reuse and noise oracles and oracle/c4_oracle.c; all unchanged) plus the library's opt-in opening positions, and a plain-Python
restatement of the opening rule.  Built on first use with gcc into a temporary directory (keyed by the sources' contents), so the
tests never write into the tree."""
from __future__ import annotations

import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

from cap_oracle import STATS, _philox4x32_10
from forced_oracle import FORCED_STATS
from oracle.c4oracle import SelfPlayResult, _Cfg, _p, _wrap_cb

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NATIVE = os.path.join(ROOT, "tests", "native")
SRC = os.path.join(NATIVE, "c4_openings_oracle.c")
DEPS = (SRC, os.path.join(NATIVE, "c4_forced_oracle.c"), os.path.join(NATIVE, "c4_cap_oracle.c"), os.path.join(NATIVE, "c4_reuse_oracle.c"),
        os.path.join(NATIVE, "c4_noise_oracle.c"), os.path.join(ROOT, "oracle", "c4_oracle.c"))
OPEN_TAG = 0xA0000000

_lib = None


def lib() -> C.CDLL:
    """gcc -O2 -ffp-contract=off (every fp32 / fp64 operation rounds on its own, as in the oracle and the kernels)."""
    global _lib
    if _lib is None:
        h = hashlib.sha256(b"".join(open(p, "rb").read() for p in DEPS)).hexdigest()[:16]
        path = os.path.join(tempfile.gettempdir(), f"c4_openings_oracle_{os.getuid()}_{h}.so")
        if not os.path.exists(path):
            tmp = f"{path}.{os.getpid()}.tmp"
            subprocess.run(["gcc", "-O2", "-ffp-contract=off", "-fopenmp", "-shared", "-fPIC", "-std=gnu11", "-o", tmp, SRC, "-lm"],
                           check=True)
            os.replace(tmp, path)
        _lib = C.CDLL(path)
    return _lib


class _OpenCfg(C.Structure):
    _fields_ = [("bb0", C.c_void_p), ("bb1", C.c_void_p), ("player", C.c_void_p), ("n_positions", C.c_int32), ("min_plies", C.c_int32),
                ("max_plies", C.c_int32), ("seed", C.c_uint64), ("slot_offset", C.c_int64)]


def _cfg(positions, min_plies, max_plies, seed, slot_offset):
    """-> (struct, the arrays it points into)"""
    if positions is None:
        keep = ()
        return _OpenCfg(None, None, None, 0, min_plies, max_plies, int(seed) & (2**64 - 1), slot_offset), keep
    keep = (np.ascontiguousarray(positions[0], np.uint64), np.ascontiguousarray(positions[1], np.uint64),
            np.ascontiguousarray(positions[2], np.uint8))
    return _OpenCfg(*(k.ctypes.data for k in keep), len(keep[0]), min_plies, max_plies, int(seed) & (2**64 - 1), slot_offset), keep


def openings_c(first_slot, n, step, positions=None, min_plies=0, max_plies=0, seed=0, init=(0, 0, 0)):
    """c4o_openings: the openings of global slots first_slot .. first_slot + n - 1 at move step `step` -> (bb0, bb1, player)"""
    cfg, keep = _cfg(positions, min_plies, max_plies, seed, 0)
    o0, o1, pl = np.zeros(n, np.uint64), np.zeros(n, np.uint64), np.zeros(n, np.uint8)
    lib().c4o_openings(C.byref(cfg), C.c_int64(first_slot), C.c_int(n), C.c_uint32(step), C.c_uint64(init[0]), C.c_uint64(init[1]),
                       C.c_int(init[2]), _p(o0, C.c_uint64), _p(o1, C.c_uint64), _p(pl, C.c_uint8))
    return o0, o1, pl


# ---- plain-Python restatement (integers and a cell grid; no bitboard tricks) ----------------------------------------------------
def _cells(b0, b1):
    return [[0 if b0 >> (7 * c + r) & 1 else 1 if b1 >> (7 * c + r) & 1 else -1 for c in range(7)] for r in range(6)]


def _four(g, who):
    for r in range(6):
        for c in range(7):
            for dr, dc in ((0, 1), (1, 0), (1, 1), (1, -1)):
                if all(0 <= r + i * dr < 6 and 0 <= c + i * dc < 7 and g[r + i * dr][c + i * dc] == who for i in range(4)):
                    return True
    return False


def drop(b0, b1, pl, col):
    """-> the position after `pl` drops in `col` (None if the column is full)"""
    h = sum(((b0 | b1) >> (7 * col + r)) & 1 for r in range(6))
    if h == 6:
        return None
    bit = 1 << (7 * col + h)
    return (b0 | bit, b1, 1) if pl == 0 else (b0, b1 | bit, 0)


def ended(b0, b1):
    g = _cells(b0, b1)
    return _four(g, 0) or _four(g, 1) or all(g[5][c] >= 0 for c in range(7))


def _x(seed, g, s, j):
    x = _philox4x32_10([g & 0xFFFFFFFF], [g >> 32], [s], [OPEN_TAG | j], seed & 0xFFFFFFFF, (seed >> 32) & 0xFFFFFFFF)
    return [int(v[0]) for v in x]


def opening_py(g, s, positions=None, min_plies=0, max_plies=0, seed=0, init=(0, 0, 0)):
    """The rule of include/az_engine.h for one game -> ((bb0, bb1, player), the columns played)"""
    x0 = _x(seed, g, s, 0)
    if positions is None:
        b0, b1, pl = init
    else:
        i = (x0[0] * len(positions[0])) >> 32
        b0, b1, pl = int(positions[0][i]), int(positions[1][i]), int(positions[2][i])
    r = min_plies + ((x0[1] * (max_plies - min_plies + 1)) >> 32)
    cols = []
    if ended(b0, b1):
        return (b0, b1, pl), cols
    for j in range(1, r + 1):
        cand = [c for c in range(7) if drop(b0, b1, pl, c) is not None and not ended(*drop(b0, b1, pl, c)[:2])]
        if not cand:
            break
        c = cand[(_x(seed, g, s, j)[0] * len(cand)) >> 32]
        b0, b1, pl = drop(b0, b1, pl, c)
        cols.append(c)
    return (b0, b1, pl), cols


def selfplay_openings(E, S, uniforms, positions=None, min_plies=0, max_plies=0, seed=0, slot_offset=0, off=False, k=0.0, full=None,
                      fast_sims=None, V=0, visit_budget=False, eps=0.0, eta=None, greedy_from=-1, quota=None, c_puct=1.0, eval_kind=1,
                      init=(0, 0, 0), py_eval=None) -> tuple[SelfPlayResult, dict]:
    """Self-play whose games start from their openings (`off` = the mode off), with the other arguments and outputs of
    `forced_oracle.selfplay_forced` (k = 0: no forcing)."""
    quota = E if quota is None else quota
    uniforms = np.ascontiguousarray(uniforms, np.float64).reshape(-1, E)
    max_steps = uniforms.shape[0]
    full = np.ones((max_steps, E), np.uint8) if full is None else np.ascontiguousarray(full, np.uint8).reshape(max_steps, E)
    fast_sims = S if fast_sims is None else fast_sims
    eta = None if eta is None else np.ascontiguousarray(eta, np.float32).reshape(max_steps, E, 7)
    n_ep_cap = int(min(quota, E * max_steps + E))  # an opening may leave a game a single ply
    max_samples = E * max_steps  # one sample per searched ply at most
    quota = int(min(quota, 2**31 - 1))
    ep_slot = np.zeros(n_ep_cap, np.int32); ep_len = np.zeros(n_ep_cap, np.int32); ep_step = np.zeros(n_ep_cap, np.int32)
    ep_out = np.zeros((n_ep_cap, 2), np.int8)
    cfg = _Cfg(E, S, eval_kind, init[2], quota, max_steps, c_puct, init[0], init[1])
    ocfg, keep_o = _cfg(positions, min_plies, max_plies, seed, slot_offset)
    s0 = np.zeros(max_samples, np.uint64); s1 = np.zeros(max_samples, np.uint64); sp = np.zeros(max_samples, np.uint8)
    sc = np.zeros((max_samples, 7), np.int32)
    st = np.zeros(len(STATS), np.int64)
    fst = np.zeros(len(FORCED_STATS), np.int64)
    last = np.zeros((E, 7), np.int32)
    ne, ns, nst, nu, nsim, nev, ndrop = (C.c_int64(0) for _ in range(7))
    cb, keep = _wrap_cb(py_eval)
    err = lib().c4o_selfplay_openings(C.byref(cfg), None if off else C.byref(ocfg), C.c_double(k), C.c_int(V), C.c_int(fast_sims),
                                      C.c_int(1 if visit_budget else 0), _p(full, C.c_uint8), _p(uniforms, C.c_double), cb, None,
                                      C.c_float(eps), None if eta is None else _p(eta, C.c_float), C.c_int(int(greedy_from)),
                                      _p(ep_slot, C.c_int32), _p(ep_len, C.c_int32), _p(ep_step, C.c_int32), _p(ep_out, C.c_int8),
                                      _p(s0, C.c_uint64), _p(s1, C.c_uint64), _p(sp, C.c_uint8), _p(sc, C.c_int32), C.c_int64(max_samples),
                                      C.byref(ne), C.byref(ns), C.byref(nst), C.byref(nu), C.byref(nsim), C.byref(nev), C.byref(ndrop),
                                      _p(st, C.c_int64), _p(fst, C.c_int64), _p(last, C.c_int32))
    if err:
        raise RuntimeError(f"c4o_selfplay_openings error {err}")
    n_ep, n_s = ne.value, ns.value
    extra = {k_: int(v) for k_, v in zip(STATS, st)}
    extra.update({k_: int(v) for k_, v in zip(FORCED_STATS, fst)})
    extra["samples_dropped"] = ndrop.value
    extra["last_counts"] = last
    return (SelfPlayResult(ep_slot[:n_ep], ep_len[:n_ep], ep_step[:n_ep], ep_out[:n_ep], s0[:n_s], s1[:n_s], sp[:n_s], sc[:n_s],
                           nst.value, nu.value, nsim.value, nev.value), extra)
