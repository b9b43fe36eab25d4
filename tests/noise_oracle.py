"""TEST INFRASTRUCTURE — ctypes wrapper of tests/native/c4_noise_oracle.c: the C oracle (oracle/c4_oracle.c, included unchanged)
plus the library's opt-in root noise and greedy cutoff.  Built on first use with gcc into a temporary directory (keyed by the
sources' contents), so the tests never write into the tree."""
from __future__ import annotations

import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

from oracle.c4oracle import SelfPlayResult, _Cfg, _p, _wrap_cb

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SRC = os.path.join(ROOT, "tests", "native", "c4_noise_oracle.c")
DEPS = (SRC, os.path.join(ROOT, "oracle", "c4_oracle.c"))

_lib = None


def lib() -> C.CDLL:
    """gcc -O2 -ffp-contract=off (every fp32 / fp64 operation rounds on its own, as in the oracle and the kernels)."""
    global _lib
    if _lib is None:
        h = hashlib.sha256(b"".join(open(p, "rb").read() for p in DEPS)).hexdigest()[:16]
        path = os.path.join(tempfile.gettempdir(), f"c4_noise_oracle_{os.getuid()}_{h}.so")
        if not os.path.exists(path):
            tmp = f"{path}.{os.getpid()}.tmp"
            subprocess.run(["gcc", "-O2", "-ffp-contract=off", "-fopenmp", "-shared", "-fPIC", "-std=gnu11", "-o", tmp, SRC, "-lm"],
                           check=True)
            os.replace(tmp, path)
        _lib = C.CDLL(path)
    return _lib


def search_noise(bb0, bb1, player, S, eps, eta, c_puct=1.0, eval_kind=1, py_eval=None):
    """`oracle.c4oracle.search` with root noise: simulation 1, the fp32 mixing with `eta` [E, 7] and fraction `eps`,
    simulations 2..S."""
    E = len(bb0)
    bb0 = np.ascontiguousarray(bb0, np.uint64); bb1 = np.ascontiguousarray(bb1, np.uint64)
    player = np.ascontiguousarray(player, np.uint8)
    eta = np.ascontiguousarray(eta, np.float32).reshape(E, 7)
    cN = np.zeros((E, 7), np.int32); cW = np.zeros((E, 7), np.float64); cP = np.zeros((E, 7), np.float32)
    rW = np.zeros(E, np.float64); rN = np.zeros(E, np.int32); lg = np.zeros(E, np.uint8)
    nev = C.c_int64(0)
    cb, keep = _wrap_cb(py_eval)
    err = lib().c4o_search_noise(C.c_int(E), _p(bb0, C.c_uint64), _p(bb1, C.c_uint64), _p(player, C.c_uint8), C.c_int(S),
                                 C.c_double(c_puct), C.c_int(eval_kind), cb, None, C.c_float(eps), _p(eta, C.c_float),
                                 _p(cN, C.c_int32), _p(cW, C.c_double), _p(cP, C.c_float), _p(rW, C.c_double), _p(rN, C.c_int32),
                                 _p(lg, C.c_uint8), C.byref(nev))
    if err:
        raise RuntimeError(f"c4o_search_noise error {err}")
    return dict(child_N=cN, child_W=cW, child_P=cP, root_W=rW, root_N=rN, legal=lg, n_evals=nev.value)


def selfplay_noise(E, S, uniforms, eps, eta, greedy_from=-1, quota=None, c_puct=1.0, eval_kind=1, init=(0, 0, 0),
                   py_eval=None) -> SelfPlayResult:
    """`oracle.c4oracle.selfplay` with root noise (fraction `eps`, `eta` [steps, E, 7]: the noise of every move step's search)
    and the greedy cutoff (plies >= `greedy_from` play the most visited root child; negative = off)."""
    quota = E if quota is None else quota
    uniforms = np.ascontiguousarray(uniforms, np.float64).reshape(-1, E)
    max_steps = uniforms.shape[0]
    eta = np.ascontiguousarray(eta, np.float32).reshape(max_steps, E, 7)
    n_ep_cap = int(min(quota, E * max_steps // 7 + E))  # a game lasts at least 7 plies
    max_samples = n_ep_cap * 42
    quota = int(min(quota, 2**31 - 1))
    ep_slot = np.zeros(n_ep_cap, np.int32); ep_len = np.zeros(n_ep_cap, np.int32); ep_step = np.zeros(n_ep_cap, np.int32)
    ep_out = np.zeros((n_ep_cap, 2), np.int8)
    cfg = _Cfg(E, S, eval_kind, init[2], quota, max_steps, c_puct, init[0], init[1])
    s0 = np.zeros(max_samples, np.uint64); s1 = np.zeros(max_samples, np.uint64); sp = np.zeros(max_samples, np.uint8)
    sc = np.zeros((max_samples, 7), np.int32)
    ne, ns, nst, nu, nsim, nev = (C.c_int64(0) for _ in range(6))
    cb, keep = _wrap_cb(py_eval)
    err = lib().c4o_selfplay_noise(C.byref(cfg), _p(uniforms, C.c_double), cb, None, C.c_float(eps), _p(eta, C.c_float),
                                   C.c_int(int(greedy_from)), _p(ep_slot, C.c_int32), _p(ep_len, C.c_int32), _p(ep_step, C.c_int32),
                                   _p(ep_out, C.c_int8), _p(s0, C.c_uint64), _p(s1, C.c_uint64), _p(sp, C.c_uint8),
                                   _p(sc, C.c_int32), C.c_int64(max_samples), C.byref(ne), C.byref(ns), C.byref(nst), C.byref(nu),
                                   C.byref(nsim), C.byref(nev))
    if err:
        raise RuntimeError(f"c4o_selfplay_noise error {err}")
    n_ep, n_s = ne.value, ns.value
    return SelfPlayResult(ep_slot[:n_ep], ep_len[:n_ep], ep_step[:n_ep], ep_out[:n_ep], s0[:n_s], s1[:n_s], sp[:n_s],
                          sc[:n_s], nst.value, nu.value, nsim.value, nev.value)
