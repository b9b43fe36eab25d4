"""TEST INFRASTRUCTURE — ctypes wrapper of tests/native/c4_cap_oracle.c: the reuse oracle (tests/native/c4_reuse_oracle.c, which
includes the noise oracle and oracle/c4_oracle.c; all unchanged) plus the library's opt-in playout cap randomization, and a numpy
restatement of the engine's full / fast draw.  Built on first use with gcc into a temporary directory (keyed by the sources'
contents), so the tests never write into the tree."""
from __future__ import annotations

import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

from oracle.c4oracle import SelfPlayResult, _Cfg, _p, _wrap_cb

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SRC = os.path.join(ROOT, "tests", "native", "c4_cap_oracle.c")
DEPS = (SRC, os.path.join(ROOT, "tests", "native", "c4_reuse_oracle.c"), os.path.join(ROOT, "tests", "native", "c4_noise_oracle.c"),
        os.path.join(ROOT, "oracle", "c4_oracle.c"))
STATS = ("retained", "fresh", "dropped", "nodes", "visits", "max_used")

_lib = None


def lib() -> C.CDLL:
    """gcc -O2 -ffp-contract=off (every fp32 / fp64 operation rounds on its own, as in the oracle and the kernels)."""
    global _lib
    if _lib is None:
        h = hashlib.sha256(b"".join(open(p, "rb").read() for p in DEPS)).hexdigest()[:16]
        path = os.path.join(tempfile.gettempdir(), f"c4_cap_oracle_{os.getuid()}_{h}.so")
        if not os.path.exists(path):
            tmp = f"{path}.{os.getpid()}.tmp"
            subprocess.run(["gcc", "-O2", "-ffp-contract=off", "-fopenmp", "-shared", "-fPIC", "-std=gnu11", "-o", tmp, SRC, "-lm"],
                           check=True)
            os.replace(tmp, path)
        _lib = C.CDLL(path)
    return _lib


def _philox4x32_10(c0, c1, c2, c3, k0, k1):
    """Philox4x32-10 on uint32 arrays (numpy, vectorised over the counters)"""
    m = np.uint64(0xFFFFFFFF)
    c0, c1, c2, c3 = (np.asarray(x, np.uint64) for x in (c0, c1, c2, c3))
    k0, k1 = np.uint64(k0), np.uint64(k1)
    for _ in range(10):
        p0 = np.uint64(0xD2511F53) * c0
        p1 = np.uint64(0xCD9E8D57) * c2
        c0, c1, c2, c3 = (p1 >> np.uint64(32)) ^ c1 ^ k0, p1 & m, (p0 >> np.uint64(32)) ^ c3 ^ k1, p0 & m
        k0 = (k0 + np.uint64(0x9E3779B9)) & m
        k1 = (k1 + np.uint64(0xBB67AE85)) & m
    return c0, c1, c2, c3


def draw_full(seed: int, slot_offset: int, n: int, step: int, p_full: float) -> np.ndarray:
    """The engine's full / fast flags (u8 [n]) of global slots slot_offset .. slot_offset + n - 1 at move step `step`."""
    g = np.arange(slot_offset, slot_offset + n, dtype=np.uint64)
    seed = int(seed) & (2**64 - 1)
    x, _, _, _ = _philox4x32_10(g & np.uint64(0xFFFFFFFF), g >> np.uint64(32), np.full(n, step, np.uint64),
                                np.full(n, 0xC0000000, np.uint64), seed & 0xFFFFFFFF, seed >> 32)
    u = (x.astype(np.float64) + 0.5) * 2.0**-32
    return (u < np.float64(np.float32(p_full))).astype(np.uint8)


def draw_full_c(seed: int, slot_offset: int, n: int, step: int, p_full: float) -> np.ndarray:
    out = np.zeros(n, np.uint8)
    lib().c4o_cap_draw(C.c_uint64(int(seed) & (2**64 - 1)), C.c_int64(slot_offset), C.c_int(n), C.c_uint32(step), C.c_float(p_full),
                       _p(out, C.c_uint8))
    return out


def selfplay_cap(E, S, fast_sims, full, uniforms, V=0, visit_budget=False, eps=0.0, eta=None, greedy_from=-1, quota=None,
                 c_puct=1.0, eval_kind=1, init=(0, 0, 0), py_eval=None) -> tuple[SelfPlayResult, dict]:
    """Self-play with the playout cap: `full` [steps, E] the flags of every search (1 = full: S new simulations, else fast_sims),
    subtree reuse under max_root_visits V (0 = off), `visit_budget`, root noise (`eta` [steps, E, 7], None = off) on the full
    searches, the greedy cutoff.  -> (result with only the full searches' samples, dict(samples_dropped=..., the reuse stats,
    last_counts = [E, 7] root visit counts by column that the last move step's search left))."""
    quota = E if quota is None else quota
    uniforms = np.ascontiguousarray(uniforms, np.float64).reshape(-1, E)
    max_steps = uniforms.shape[0]
    full = np.ascontiguousarray(full, np.uint8).reshape(max_steps, E)
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
    last = np.zeros((E, 7), np.int32)
    ne, ns, nst, nu, nsim, nev, ndrop = (C.c_int64(0) for _ in range(7))
    cb, keep = _wrap_cb(py_eval)
    err = lib().c4o_selfplay_cap(C.byref(cfg), C.c_int(V), C.c_int(fast_sims), C.c_int(1 if visit_budget else 0), _p(full, C.c_uint8),
                                 _p(uniforms, C.c_double), cb, None, C.c_float(eps), None if eta is None else _p(eta, C.c_float),
                                 C.c_int(int(greedy_from)), _p(ep_slot, C.c_int32), _p(ep_len, C.c_int32), _p(ep_step, C.c_int32),
                                 _p(ep_out, C.c_int8), _p(s0, C.c_uint64), _p(s1, C.c_uint64), _p(sp, C.c_uint8), _p(sc, C.c_int32),
                                 C.c_int64(max_samples), C.byref(ne), C.byref(ns), C.byref(nst), C.byref(nu), C.byref(nsim),
                                 C.byref(nev), C.byref(ndrop), _p(st, C.c_int64), _p(last, C.c_int32))
    if err:
        raise RuntimeError(f"c4o_selfplay_cap error {err}")
    n_ep, n_s = ne.value, ns.value
    extra = {k: int(v) for k, v in zip(STATS, st)}
    extra["samples_dropped"] = ndrop.value
    extra["last_counts"] = last
    return (SelfPlayResult(ep_slot[:n_ep], ep_len[:n_ep], ep_step[:n_ep], ep_out[:n_ep], s0[:n_s], s1[:n_s], sp[:n_s], sc[:n_s],
                           nst.value, nu.value, nsim.value, nev.value), extra)
