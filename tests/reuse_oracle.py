"""TEST INFRASTRUCTURE — ctypes wrapper of tests/native/c4_reuse_oracle.c: the noise oracle (tests/native/c4_noise_oracle.c, which
includes oracle/c4_oracle.c; both unchanged) plus the library's opt-in subtree reuse.  Built on first use with gcc into a temporary
directory (keyed by the sources' contents), so the tests never write into the tree."""
from __future__ import annotations

import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

from oracle.c4oracle import SelfPlayResult, _Cfg, _p, _wrap_cb

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SRC = os.path.join(ROOT, "tests", "native", "c4_reuse_oracle.c")
DEPS = (SRC, os.path.join(ROOT, "tests", "native", "c4_noise_oracle.c"), os.path.join(ROOT, "oracle", "c4_oracle.c"))
STATS = ("retained", "fresh", "dropped", "nodes", "visits", "max_used")

_lib = None


def lib() -> C.CDLL:
    """gcc -O2 -ffp-contract=off (every fp32 / fp64 operation rounds on its own, as in the oracle and the kernels)."""
    global _lib
    if _lib is None:
        h = hashlib.sha256(b"".join(open(p, "rb").read() for p in DEPS)).hexdigest()[:16]
        path = os.path.join(tempfile.gettempdir(), f"c4_reuse_oracle_{os.getuid()}_{h}.so")
        if not os.path.exists(path):
            tmp = f"{path}.{os.getpid()}.tmp"
            subprocess.run(["gcc", "-O2", "-ffp-contract=off", "-fopenmp", "-shared", "-fPIC", "-std=gnu11", "-o", tmp, SRC, "-lm"],
                           check=True)
            os.replace(tmp, path)
        _lib = C.CDLL(path)
    return _lib


def _stats(st) -> dict:
    return {k: int(v) for k, v in zip(STATS, st)}


def advance_reuse(bb0, bb1, player, S1, cols, S, V, S2=0, export_slots=None, c_puct=1.0, eval_kind=1, py_eval=None):
    """S1 simulations on every root, the move `cols[i]` on every root under the retention rule (S new simulations per search,
    max_root_visits V), S2 more simulations; -> status [E] (1 = illegal column), the trees of `export_slots` (default: all) in the
    engine's export format (W, N, P, first_child as [n, cap] arrays with cap = roundup8(1 + 7 V), used [n]) and the reuse stats."""
    E = len(bb0)
    bb0 = np.ascontiguousarray(bb0, np.uint64); bb1 = np.ascontiguousarray(bb1, np.uint64)
    player = np.ascontiguousarray(player, np.uint8); cols = np.ascontiguousarray(cols, np.uint8)
    slots = np.arange(E, dtype=np.int32) if export_slots is None else np.ascontiguousarray(export_slots, np.int32)
    n, cap = len(slots), (1 + 7 * V + 7) & ~7
    W = np.zeros((n, cap), np.float64); N = np.zeros((n, cap), np.uint32); P = np.zeros((n, cap), np.float32)
    CB = np.zeros((n, cap), np.uint32); used = np.zeros(n, np.int32)
    status = np.zeros(E, np.uint8); st = np.zeros(len(STATS), np.int64)
    cb, keep = _wrap_cb(py_eval)
    err = lib().c4o_advance_reuse(C.c_int(E), _p(bb0, C.c_uint64), _p(bb1, C.c_uint64), _p(player, C.c_uint8), C.c_int(S1), C.c_int(S2),
                                  C.c_int(S), C.c_int(V), C.c_double(c_puct), C.c_int(eval_kind), cb, None, _p(cols, C.c_uint8),
                                  _p(status, C.c_uint8), C.c_int(n), _p(slots, C.c_int32), C.c_int(cap), _p(W, C.c_double),
                                  _p(N, C.c_uint32), _p(P, C.c_float), _p(CB, C.c_uint32), _p(used, C.c_int32), _p(st, C.c_int64))
    if err:
        raise RuntimeError(f"c4o_advance_reuse error {err}")
    return dict(status=status, W=W, N=N, P=P, first_child=CB, used=used, stats=_stats(st))


def selfplay_reuse(E, S, V, uniforms, eps=0.0, eta=None, greedy_from=-1, quota=None, c_puct=1.0, eval_kind=1, init=(0, 0, 0),
                   py_eval=None) -> tuple[SelfPlayResult, dict]:
    """`noise_oracle.selfplay_noise` with subtree reuse under max_root_visits V (>= S); -> (result, reuse stats).  `eta` None =
    no noise."""
    quota = E if quota is None else quota
    uniforms = np.ascontiguousarray(uniforms, np.float64).reshape(-1, E)
    max_steps = uniforms.shape[0]
    eta = None if eta is None else np.ascontiguousarray(eta, np.float32).reshape(max_steps, E, 7)
    n_ep_cap = int(min(quota, E * max_steps // 7 + E))  # a game lasts at least 7 plies
    max_samples = n_ep_cap * 42
    quota = int(min(quota, 2**31 - 1))
    ep_slot = np.zeros(n_ep_cap, np.int32); ep_len = np.zeros(n_ep_cap, np.int32); ep_step = np.zeros(n_ep_cap, np.int32)
    ep_out = np.zeros((n_ep_cap, 2), np.int8)
    cfg = _Cfg(E, S, eval_kind, init[2], quota, max_steps, c_puct, init[0], init[1])
    s0 = np.zeros(max_samples, np.uint64); s1 = np.zeros(max_samples, np.uint64); sp = np.zeros(max_samples, np.uint8)
    sc = np.zeros((max_samples, 7), np.int32)
    st = np.zeros(len(STATS), np.int64)
    ne, ns, nst, nu, nsim, nev = (C.c_int64(0) for _ in range(6))
    cb, keep = _wrap_cb(py_eval)
    err = lib().c4o_selfplay_reuse(C.byref(cfg), C.c_int(V), _p(uniforms, C.c_double), cb, None, C.c_float(eps), None if eta is None else _p(eta, C.c_float),
                                   C.c_int(int(greedy_from)), _p(ep_slot, C.c_int32), _p(ep_len, C.c_int32), _p(ep_step, C.c_int32),
                                   _p(ep_out, C.c_int8), _p(s0, C.c_uint64), _p(s1, C.c_uint64), _p(sp, C.c_uint8),
                                   _p(sc, C.c_int32), C.c_int64(max_samples), C.byref(ne), C.byref(ns), C.byref(nst), C.byref(nu),
                                   C.byref(nsim), C.byref(nev), _p(st, C.c_int64))
    if err:
        raise RuntimeError(f"c4o_selfplay_reuse error {err}")
    n_ep, n_s = ne.value, ns.value
    return (SelfPlayResult(ep_slot[:n_ep], ep_len[:n_ep], ep_step[:n_ep], ep_out[:n_ep], s0[:n_s], s1[:n_s], sp[:n_s], sc[:n_s], nst.value,
                           nu.value, nsim.value, nev.value), _stats(st))
