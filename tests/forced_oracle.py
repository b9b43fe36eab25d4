"""TEST INFRASTRUCTURE — ctypes wrapper of tests/native/c4_forced_oracle.c: the cap oracle (tests/native/c4_cap_oracle.c, which
includes the reuse and noise oracles and oracle/c4_oracle.c; all unchanged) plus the library's opt-in forced playouts and policy
target pruning, and a numpy restatement of the pruning.  Built on first use with gcc into a temporary directory (keyed by the
sources' contents), so the tests never write into the tree."""
from __future__ import annotations

import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

from cap_oracle import STATS
from oracle.c4oracle import SelfPlayResult, _Cfg, _p, _wrap_cb

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SRC = os.path.join(ROOT, "tests", "native", "c4_forced_oracle.c")
DEPS = (SRC, os.path.join(ROOT, "tests", "native", "c4_cap_oracle.c"), os.path.join(ROOT, "tests", "native", "c4_reuse_oracle.c"),
        os.path.join(ROOT, "tests", "native", "c4_noise_oracle.c"), os.path.join(ROOT, "oracle", "c4_oracle.c"))
FORCED_STATS = ("forced_selections", "forced_searches", "visits_pruned", "children_zeroed")

_lib = None


def lib() -> C.CDLL:
    """gcc -O2 -ffp-contract=off (every fp32 / fp64 operation rounds on its own, as in the oracle and the kernels)."""
    global _lib
    if _lib is None:
        h = hashlib.sha256(b"".join(open(p, "rb").read() for p in DEPS)).hexdigest()[:16]
        path = os.path.join(tempfile.gettempdir(), f"c4_forced_oracle_{os.getuid()}_{h}.so")
        if not os.path.exists(path):
            tmp = f"{path}.{os.getpid()}.tmp"
            subprocess.run(["gcc", "-O2", "-ffp-contract=off", "-fopenmp", "-shared", "-fPIC", "-std=gnu11", "-o", tmp, SRC, "-lm"],
                           check=True)
            os.replace(tmp, path)
        _lib = C.CDLL(path)
    return _lib


def prune_c(N, W, P, legal, root_N, c_puct, k):
    """c4o_prune: N' [n, 7] and (visits pruned, children zeroed)."""
    N = np.ascontiguousarray(N, np.int32)
    n = N.shape[0]
    out = np.zeros((n, 7), np.int32)
    st = np.zeros(2, np.int64)
    lib().c4o_prune(C.c_int(n), _p(N, C.c_int32), _p(np.ascontiguousarray(W, np.float64), C.c_double),
                    _p(np.ascontiguousarray(P, np.float32), C.c_float), _p(np.ascontiguousarray(legal, np.uint8), C.c_uint8),
                    _p(np.ascontiguousarray(root_N, np.int32), C.c_int32), C.c_double(c_puct), C.c_double(k), _p(out, C.c_int32),
                    _p(st, C.c_int64))
    return out, (int(st[0]), int(st[1]))


def n_forced(P, root_N, k):
    """n_f [n, 7]: the least n >= 0 with RN(n * n) >= RN(RN(k * P) * (N_root - 1)) (numpy fp64, one rounding per operation)."""
    thr = (np.float64(k) * np.asarray(P, np.float32).astype(np.float64)) * (np.asarray(root_N, np.float64)[:, None] - 1.0)
    nf = np.ceil(np.sqrt(np.maximum(thr, 0.0))).astype(np.int64)
    nf = np.where((nf - 1).astype(np.float64) ** 2 >= thr, nf - 1, nf)
    nf = np.maximum(nf, 0)
    return np.where(nf.astype(np.float64) ** 2 < thr, nf + 1, nf)


def prune_np(N, W, P, legal, root_N, c_puct, k):
    """The pruning rule of include/az_engine.h in numpy fp64, vectorised over roots (one visit at a time for all of them)."""
    N = np.asarray(N, np.int64)
    W = np.asarray(W, np.float64)
    Pd = np.asarray(P, np.float32).astype(np.float64)
    root_N = np.asarray(root_N, np.int64)
    lg = ((np.asarray(legal, np.int64)[:, None] >> np.arange(7)) & 1).astype(bool)
    out = N.copy()
    active = (root_N > 1) & (k != 0.0)
    rows = np.arange(len(N))
    bc = np.argmax(np.where(lg, N, -1), axis=1)  # first maximum
    sq = np.sqrt(root_N.astype(np.float64))
    nb, wb, pb = N[rows, bc], W[rows, bc], Pd[rows, bc]
    with np.errstate(divide="ignore", invalid="ignore"):
        qb = np.where(wb == 0.0, 0.0, wb / np.maximum(nb, 1))
        s_star = qb + ((np.float64(c_puct) * pb) * sq) / (1.0 + nb)
        q = np.where(W == 0.0, 0.0, W / np.maximum(N, 1))
    x = (np.float64(c_puct) * Pd) * sq[:, None]
    nf = n_forced(P, root_N, k)
    cand = lg & (N > 0) & (np.arange(7)[None, :] != bc[:, None]) & active[:, None]
    while True:
        with np.errstate(divide="ignore", invalid="ignore"):
            score = q + x / out.astype(np.float64)
        step = cand & (N - out < nf) & (out > 0) & (score < s_star[:, None])
        if not step.any():
            break
        out = out - step
    out = np.where(cand & (out == 1), 0, out)
    return out.astype(np.int32)


def selfplay_forced(E, S, k, uniforms, full=None, fast_sims=None, V=0, visit_budget=False, eps=0.0, eta=None, greedy_from=-1, quota=None,
                    c_puct=1.0, eval_kind=1, init=(0, 0, 0), py_eval=None) -> tuple[SelfPlayResult, dict]:
    """Self-play with forced playouts of parameter k on the full searches (`full` [steps, E], None = every search full: no cap),
    their pruned counts as samples and moves, and otherwise the arguments of `cap_oracle.selfplay_cap`.  -> (result, dict(the
    counters of FORCED_STATS, samples_dropped, the reuse stats, last_counts = [E, 7] the counts the last move step recorded))."""
    quota = E if quota is None else quota
    uniforms = np.ascontiguousarray(uniforms, np.float64).reshape(-1, E)
    max_steps = uniforms.shape[0]
    full = np.ones((max_steps, E), np.uint8) if full is None else np.ascontiguousarray(full, np.uint8).reshape(max_steps, E)
    fast_sims = S if fast_sims is None else fast_sims
    eta = None if eta is None else np.ascontiguousarray(eta, np.float32).reshape(max_steps, E, 7)
    n_ep_cap = int(min(quota, E * max_steps // 7 + E))
    max_samples = n_ep_cap * 42
    quota = int(min(quota, 2**31 - 1))
    ep_slot = np.zeros(n_ep_cap, np.int32); ep_len = np.zeros(n_ep_cap, np.int32); ep_step = np.zeros(n_ep_cap, np.int32)
    ep_out = np.zeros((n_ep_cap, 2), np.int8)
    cfg = _Cfg(E, S, eval_kind, init[2], quota, max_steps, c_puct, init[0], init[1])
    s0 = np.zeros(max_samples, np.uint64); s1 = np.zeros(max_samples, np.uint64); sp = np.zeros(max_samples, np.uint8)
    sc = np.zeros((max_samples, 7), np.int32)
    st = np.zeros(len(STATS), np.int64)
    fst = np.zeros(len(FORCED_STATS), np.int64)
    last = np.zeros((E, 7), np.int32)
    ne, ns, nst, nu, nsim, nev, ndrop = (C.c_int64(0) for _ in range(7))
    cb, keep = _wrap_cb(py_eval)
    err = lib().c4o_selfplay_forced(C.byref(cfg), C.c_double(k), C.c_int(V), C.c_int(fast_sims), C.c_int(1 if visit_budget else 0),
                                    _p(full, C.c_uint8), _p(uniforms, C.c_double), cb, None, C.c_float(eps),
                                    None if eta is None else _p(eta, C.c_float), C.c_int(int(greedy_from)), _p(ep_slot, C.c_int32),
                                    _p(ep_len, C.c_int32), _p(ep_step, C.c_int32), _p(ep_out, C.c_int8), _p(s0, C.c_uint64),
                                    _p(s1, C.c_uint64), _p(sp, C.c_uint8), _p(sc, C.c_int32), C.c_int64(max_samples), C.byref(ne),
                                    C.byref(ns), C.byref(nst), C.byref(nu), C.byref(nsim), C.byref(nev), C.byref(ndrop), _p(st, C.c_int64),
                                    _p(fst, C.c_int64), _p(last, C.c_int32))
    if err:
        raise RuntimeError(f"c4o_selfplay_forced error {err}")
    n_ep, n_s = ne.value, ns.value
    extra = {k_: int(v) for k_, v in zip(STATS, st)}
    extra.update({k_: int(v) for k_, v in zip(FORCED_STATS, fst)})
    extra["samples_dropped"] = ndrop.value
    extra["last_counts"] = last
    return (SelfPlayResult(ep_slot[:n_ep], ep_len[:n_ep], ep_step[:n_ep], ep_out[:n_ep], s0[:n_s], s1[:n_s], sp[:n_s], sc[:n_s],
                           nst.value, nu.value, nsim.value, nev.value), extra)
