"""Python handle on the CUDA engine (include/az_engine.h).  PyTorch is used only for device
memory, streams and host<->device copies; every computation on the path is a kernel of
libaz_engine.so.  No fallback exists: constructing an `Engine` without a B200 raises.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass

import numpy as np
import torch

from . import _lib
from ._lib import AzCapStats, AzConfig, AzEvalCacheStats, AzPlayoutCap, AzReuseStats, AzRootNoise, AzStats

EVAL_UNIFORM = 1
EVAL_HASH = 2
LAYOUT_GRID_F32 = 0
LAYOUT_PLANES_F32 = 1
LAYOUT_PLANES_BF16 = 2
LAYOUT_PLANES_BF16_NHWC = 3
POLICY_LOGITS = 0
POLICY_PRIORS = 1
LEAF_EVAL, LEAF_TERMINAL, LEAF_IDLE, LEAF_SERVED = 0, 1, 2, 3
TREE_ROOT_ENDED = 3

_LAYOUT_SHAPE = {
    LAYOUT_GRID_F32: ((6, 7), torch.float32),
    LAYOUT_PLANES_F32: ((3, 6, 7), torch.float32),
    LAYOUT_PLANES_BF16: ((3, 6, 7), torch.bfloat16),
    LAYOUT_PLANES_BF16_NHWC: ((6, 7, 8), torch.bfloat16),
}


def _ptr(t: torch.Tensor | None, allow_pinned: bool = False) -> int | None:
    if t is None:
        return None
    ok = t.is_cuda or (allow_pinned and t.is_pinned())  # page-locked host memory is device-addressable (UVA): zero-copy
    assert ok and t.is_contiguous(), "engine buffers must be contiguous CUDA tensors" + (" or pinned host tensors" if allow_pinned else "")
    return t.data_ptr()


def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


@dataclass
class EpisodeBatch:
    """Finished games as flat host arrays (the device ring drained once).

    Episode i owns samples [ep_offset[i], ep_offset[i] + ep_len[i]).  Policy target of a sample =
    s_counts / (root visits - 1) = s_counts over their sum (`Node.improved_policy`, node.py:23-29; S - 1 unless the root kept
    its subtree, `Engine.set_subtree_reuse`); value target = ep_outcome of its episode
    (`Episode.backpropagate_outcome`, episode.py:52-54).  Sorted in the reference's yield order (step, slot).
    """

    ep_slot: np.ndarray
    ep_step: np.ndarray
    ep_len: np.ndarray
    ep_offset: np.ndarray
    ep_outcome: np.ndarray  # [n,2] int8
    s_bb0: np.ndarray
    s_bb1: np.ndarray
    s_player: np.ndarray
    s_counts: np.ndarray  # [m,7] int32

    def __len__(self) -> int:
        return int(self.ep_slot.shape[0])

    @property
    def num_samples(self) -> int:
        return int(self.ep_len.sum())


class Engine:
    """E game slots, each with a tree arena sized for S simulations per move."""

    def __init__(self, num_games: int, num_simulations: int, c_puct: float = 1.0, device: int | None = None,
                 lanes_per_tree: int = 0, hot_nodes: int | None = None):
        self.lib = _lib.load()
        if not torch.cuda.is_available():
            raise RuntimeError("alphazero_implementation_b200 needs a CUDA device (B200, sm_100a); there is no CPU path")
        self.device_index = torch.cuda.current_device() if device is None else int(device)
        self.device = torch.device("cuda", self.device_index)
        self.num_games = int(num_games)
        self.num_simulations = int(num_simulations)
        self.c_puct = float(c_puct)
        cfg = AzConfig(6, 7, 4, self.num_games, self.num_simulations, self.device_index, int(lanes_per_tree),
                       0 if hot_nodes is None else int(hot_nodes) + 1, self.c_puct)
        h = C.c_void_p()
        rc = self.lib.az_create(C.byref(cfg), C.byref(h))
        if rc != 0:
            raise RuntimeError(f"az_create failed ({rc}): {self.lib.az_last_error(None).decode()}")
        self.h = h
        self.n_active = self.num_games
        self.leaf_compaction = False
        self.leaf_compaction_fused = False
        self.eval_cache_log2 = 0
        self.root_noise = None  # (alpha, fraction, seed, slot_offset) while noise is configured
        self.greedy_from = -1
        self.symmetric_eval = False
        self.subtree_reuse = 0  # max_root_visits, 0 = off
        self.playout_cap = None  # (fast_sims, p_full, seed, slot_offset, visit_budget) while the playout cap is on
        self.tree_capacity = self.lib.az_tree_capacity(self.h)

    # -- plumbing --------------------------------------------------------------------------------
    def _check(self, rc: int, what: str):
        if rc != 0:
            raise RuntimeError(f"{what} failed ({rc}): {self.lib.az_last_error(self.h).decode()}")

    def close(self):
        if getattr(self, "h", None):
            self.lib.az_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _dev(self, x, dtype) -> torch.Tensor:
        if isinstance(x, torch.Tensor):
            return x.to(device=self.device, dtype=dtype, non_blocking=True).contiguous()
        a = np.ascontiguousarray(x)
        if a.dtype == np.uint64:
            a = a.view(np.int64)
        return torch.from_numpy(a).to(device=self.device, dtype=dtype, non_blocking=True)

    def empty(self, shape, dtype) -> torch.Tensor:
        return torch.empty(shape, dtype=dtype, device=self.device)

    @property
    def device_bytes(self) -> int:
        return int(self.lib.az_device_bytes(self.h))

    @property
    def launch_count(self) -> int:
        return int(self.lib.az_launch_count(self.h))

    # -- rules -----------------------------------------------------------------------------------
    def env_step(self, bb0, bb1, player, col):
        """`Action.sample_next_state()` on a batch -> dict of device tensors."""
        bb0 = self._dev(bb0, torch.int64); bb1 = self._dev(bb1, torch.int64)
        player = self._dev(player, torch.uint8); col = self._dev(col, torch.uint8)
        n = bb0.numel()
        out = dict(bb0=self.empty(n, torch.int64), bb1=self.empty(n, torch.int64), player=self.empty(n, torch.uint8),
                   legal=self.empty(n, torch.uint8), ended=self.empty(n, torch.uint8), reward=self.empty((n, 2), torch.int8),
                   status=self.empty(n, torch.uint8))
        self._check(self.lib.az_env_step(self.h, _ptr(bb0), _ptr(bb1), _ptr(player), _ptr(col), n, _ptr(out["bb0"]),
                                         _ptr(out["bb1"]), _ptr(out["player"]), _ptr(out["legal"]), _ptr(out["ended"]),
                                         _ptr(out["reward"]), _ptr(out["status"]), _stream()), "az_env_step")
        return out

    def state_info(self, bb0, bb1, player=None):
        bb0 = self._dev(bb0, torch.int64); bb1 = self._dev(bb1, torch.int64)
        n = bb0.numel()
        out = dict(legal=self.empty(n, torch.uint8), ended=self.empty(n, torch.uint8), reward=self.empty((n, 2), torch.int8))
        self._check(self.lib.az_state_info(self.h, _ptr(bb0), _ptr(bb1), None, n, _ptr(out["legal"]), _ptr(out["ended"]),
                                           _ptr(out["reward"]), _stream()), "az_state_info")
        return out

    def mirror_states(self, bb0, bb1, flags=None, out: tuple[torch.Tensor, torch.Tensor] | None = None):
        """Left-right mirror of the positions (`az_mirror_states`): column c goes to column 6 - c in both bitboards; with `flags`
        (u8 per position) only the rows whose flag is non-zero, the others are copied.  `out` = (bb0, bb1) int64 device tensors,
        which may be the inputs themselves.  -> (bb0, bb1)"""
        bb0 = self._dev(bb0, torch.int64); bb1 = self._dev(bb1, torch.int64)
        flags = None if flags is None else self._dev(flags, torch.uint8)
        n = bb0.numel()
        o0, o1 = out if out is not None else (self.empty(n, torch.int64), self.empty(n, torch.int64))
        self._check(self.lib.az_mirror_states(self.h, _ptr(bb0), _ptr(bb1), _ptr(flags), n, _ptr(o0), _ptr(o1), _stream()),
                    "az_mirror_states")
        return o0, o1

    def masked_softmax(self, logits: torch.Tensor, legal) -> torch.Tensor:
        logits = self._dev(logits, torch.float32).reshape(-1, 7)
        legal = self._dev(legal, torch.uint8)
        out = self.empty(logits.shape, torch.float32)
        self._check(self.lib.az_masked_softmax(self.h, _ptr(logits), _ptr(legal), logits.shape[0], _ptr(out), _stream()),
                    "az_masked_softmax")
        return out

    def encode_states(self, bb0, bb1, player, layout: int, out: torch.Tensor | None = None) -> torch.Tensor:
        bb0 = self._dev(bb0, torch.int64); bb1 = self._dev(bb1, torch.int64); player = self._dev(player, torch.uint8)
        n = bb0.numel()
        shape, dtype = _LAYOUT_SHAPE[layout]
        if out is None:
            out = self.empty((n, *shape), dtype)
        self._check(self.lib.az_encode_states(self.h, _ptr(bb0), _ptr(bb1), _ptr(player), n, _ptr(out), layout, _stream()),
                    "az_encode_states")
        return out

    # -- roots -----------------------------------------------------------------------------------
    def reset_games(self, init_bb0: int = 0, init_bb1: int = 0, init_player: int = 0):
        self._check(self.lib.az_reset_games(self.h, int(init_bb0), int(init_bb1), int(init_player), _stream()), "az_reset_games")
        self.n_active = self.num_games

    def set_roots(self, bb0, bb1, player):
        bb0 = self._dev(bb0, torch.int64); bb1 = self._dev(bb1, torch.int64); player = self._dev(player, torch.uint8)
        n = bb0.numel()
        self._check(self.lib.az_set_roots(self.h, _ptr(bb0), _ptr(bb1), _ptr(player), n, _stream()), "az_set_roots")
        self.n_active = n

    # -- search ----------------------------------------------------------------------------------
    def set_leaf_compaction(self, on: bool, fused: bool = False):
        """Every selection also writes the list of the slots that wait for an evaluation (the ResNet / CNN kernels walk it): in one
        more launch, ascending - or, `fused`, inside `expand_backup_select` itself, in the order the warps finished."""
        mode = (2 if fused else 1) if on else 0
        self._check(self.lib.az_set_leaf_compaction(self.h, mode), "az_set_leaf_compaction")
        self.leaf_compaction = bool(on)
        self.leaf_compaction_fused = mode == 2

    def set_eval_cache(self, log2_entries: int | None):
        """Evaluation cache of the leaves (`az_set_eval_cache`, active while leaf compaction is on): 2^log2_entries entries of 64
        bytes, 0 = off.  None = sized for this engine: about one entry per simulation of a move step (at least 2^10, at most 2^24 =
        1 GiB), so that the positions of the current and the previous move step fit at under half load.  Only for evaluators whose
        output row is a pure function of the position; call it before a CUDA graph of the search is captured."""
        if log2_entries is None:
            log2_entries = min(24, max(10, (self.num_games * self.num_simulations - 1).bit_length()))
        self._check(self.lib.az_set_eval_cache(self.h, int(log2_entries)), "az_set_eval_cache")
        self.eval_cache_log2 = int(log2_entries)

    def bump_eval_epoch(self):
        """Cached evaluations stop matching (the evaluator's weights changed)."""
        self._check(self.lib.az_bump_eval_epoch(self.h, _stream()), "az_bump_eval_epoch")

    def eval_cache_stats(self) -> dict:
        """rows (leaves the evaluator computed), hits, followers (leaves that reused another tree's row of the same selection),
        failed_claims, evictions - totals since creation / `reset_stats`."""
        st = AzEvalCacheStats()
        self._check(self.lib.az_get_eval_cache_stats(self.h, C.byref(st), _stream()), "az_get_eval_cache_stats")
        return {n: int(getattr(st, n)) for n, _ in AzEvalCacheStats._fields_}

    def set_root_noise(self, alpha: float | None, fraction: float = 0.25, seed: int = 0, slot_offset: int = 0):
        """Dirichlet noise on the root priors (`az_set_root_noise`); `alpha=None` turns it off.  Resets the draw counter: the
        n-th `apply_root_noise` after this call draws the same eta for the same (seed, slot_offset + slot)."""
        if alpha is None:
            self._check(self.lib.az_set_root_noise(self.h, None), "az_set_root_noise")
            self.root_noise = None
            return
        cfg = AzRootNoise(float(alpha), float(fraction), int(seed) & (2**64 - 1), int(slot_offset))
        self._check(self.lib.az_set_root_noise(self.h, C.byref(cfg)), "az_set_root_noise")
        self.root_noise = (float(alpha), float(fraction), int(seed), int(slot_offset))

    def apply_root_noise(self):
        """Mix fresh noise into the root priors of every active tree: exactly once per search, after its first simulation."""
        self._check(self.lib.az_apply_root_noise(self.h, _stream()), "az_apply_root_noise")

    def root_noise_values(self, out: torch.Tensor | None = None) -> torch.Tensor:
        """eta [num_games, 7] f32 of the last `apply_root_noise` (0 on illegal columns and for the trees it skipped)."""
        if out is None:
            out = self.empty((self.num_games, 7), torch.float32)
        self._check(self.lib.az_root_noise_values(self.h, _ptr(out), _stream()), "az_root_noise_values")
        return out

    def set_greedy_from(self, plies: int | None):
        """From ply `plies` of every game on, the move step plays the most visited root child (lowest column on ties) instead of
        sampling; None or negative = off."""
        plies = -1 if plies is None or plies < 0 else int(plies)
        self._check(self.lib.az_set_greedy_from(self.h, plies), "az_set_greedy_from")
        self.greedy_from = plies

    def set_symmetric_eval(self, on: bool):
        """Symmetric leaf evaluation (`az_set_symmetric_eval`): every non-terminal leaf is evaluated in its canonical orientation
        (the smaller of it and its left-right mirror) and a mirrored leaf's priors are stored with the columns reversed.  Network and
        `predict` evaluators only; call it before a CUDA graph of the search is captured."""
        self._check(self.lib.az_set_symmetric_eval(self.h, 1 if on else 0), "az_set_symmetric_eval")
        self.symmetric_eval = bool(on)

    def leaf_mirror(self) -> torch.Tensor | None:
        """u8 [num_games] view of the engine's flags: 1 where the last selection's leaf is the mirror of the position reached;
        None when that selection ran with symmetric evaluation off."""
        p = C.c_void_p()
        self._check(self.lib.az_leaf_mirror(self.h, C.byref(p)), "az_leaf_mirror")
        if not p.value:
            return None

        class _Raw:
            def __init__(self, ptr, n):
                self.__cuda_array_interface__ = dict(shape=(n,), typestr="|u1", data=(ptr, False), version=2)

        return torch.as_tensor(_Raw(p.value, self.num_games), device=self.device)

    def set_subtree_reuse(self, max_root_visits: int | None):
        """Subtree reuse (`az_set_subtree_reuse`): after each self-play move (and `advance_roots`) the played child becomes the root
        and keeps its subtree with all its statistics when it is expanded and N(child) + num_simulations <= max_root_visits; every
        search still runs num_simulations new simulations.  None / 0 = off (the default).  Sizes the trees for 1 + 7 max_root_visits
        nodes (`tree_capacity`) and resets every tree to a fresh root (positions and game logs are kept).  Call it before a CUDA
        graph of the search is captured."""
        v = 0 if max_root_visits is None else int(max_root_visits)
        self._check(self.lib.az_set_subtree_reuse(self.h, v), "az_set_subtree_reuse")
        self.subtree_reuse = v
        self.tree_capacity = self.lib.az_tree_capacity(self.h)

    def advance_roots(self, cols) -> torch.Tensor:
        """Play column `cols[t]` on every active root and keep that child's subtree under the reuse rule (`az_advance_roots`; subtree
        reuse must be on).  -> u8 status per root: 0 played, 1 illegal column (the slot is left as it was).  A move that ends the game
        leaves that position as a finished root (`TREE_ROOT_ENDED`)."""
        cols = self._dev(cols, torch.uint8)
        assert cols.numel() >= self.n_active
        status = self.empty(self.n_active, torch.uint8)
        self._check(self.lib.az_advance_roots(self.h, _ptr(cols), _ptr(status), _stream()), "az_advance_roots")
        return status

    def reuse_stats(self) -> dict:
        """Moves whose played child's subtree was retained, that went to a never-expanded child (fresh) or were dropped
        (N(child) + num_simulations > max_root_visits), and the retained nodes and root visits - totals since creation /
        `reset_stats`."""
        st = AzReuseStats()
        self._check(self.lib.az_get_reuse_stats(self.h, C.byref(st), _stream()), "az_get_reuse_stats")
        return {n: int(getattr(st, n)) for n, _ in AzReuseStats._fields_}

    def set_playout_cap(self, fast_sims: int | None, p_full: float = 0.25, seed: int = 0, slot_offset: int = 0,
                        visit_budget: bool = False):
        """Playout cap randomization (`az_set_playout_cap`, KataGo): each self-play search (after `reset_games` and every
        `sample_moves`) is full with probability `p_full` (num_simulations new simulations) or fast (`fast_sims`); a tree that has run
        its share is idle for the rest of the move step.  Only full searches become samples of the finished games (an episode may
        then have none).  Fast searches get no root noise.  `visit_budget`: a search tops the root up to that many visits instead
        (at least one new simulation; for subtree reuse).  The draw is a function of (seed, slot_offset + slot, move step) alone.
        `fast_sims=None` = off (the default).  Call it before a CUDA graph of the search is captured."""
        if fast_sims is None:
            self._check(self.lib.az_set_playout_cap(self.h, None), "az_set_playout_cap")
            self.playout_cap = None
            return
        cfg = AzPlayoutCap(int(fast_sims), float(p_full), int(seed) & (2**64 - 1), int(slot_offset), 1 if visit_budget else 0)
        self._check(self.lib.az_set_playout_cap(self.h, C.byref(cfg)), "az_set_playout_cap")
        self.playout_cap = (int(fast_sims), float(p_full), int(seed), int(slot_offset), bool(visit_budget))

    def search_budgets(self) -> tuple[torch.Tensor, torch.Tensor]:
        """The playout cap's current draw -> (budget int64 [num_games]: the root visit count at which each tree stops, full u8
        [num_games]: 1 = full search)."""
        b = self.empty(self.num_games, torch.int32)
        f = self.empty(self.num_games, torch.uint8)
        self._check(self.lib.az_search_budgets(self.h, _ptr(b), _ptr(f), _stream()), "az_search_budgets")
        return b.to(torch.int64) & 0xFFFFFFFF, f

    def cap_stats(self) -> dict:
        """Self-play searches by kind (full / fast), samples of finished games recorded / dropped, and the new simulations run -
        totals since creation / `reset_stats`."""
        st = AzCapStats()
        self._check(self.lib.az_get_cap_stats(self.h, C.byref(st), _stream()), "az_get_cap_stats")
        return {n: int(getattr(st, n)) for n, _ in AzCapStats._fields_}

    def run_simulations(self, num_sims: int, eval_kind: int):
        self._check(self.lib.az_run_simulations(self.h, int(num_sims), int(eval_kind), _stream()), "az_run_simulations")

    def select_leaves(self):
        self._check(self.lib.az_select_leaves(self.h, _stream()), "az_select_leaves")

    def gather_leaves(self, layout: int, out: torch.Tensor | None = None) -> torch.Tensor:
        """Pack the leaves' planes into `out`: a device batch, or a PINNED host batch the kernel writes straight into (for an
        evaluator that lives on the host; synchronise the stream before reading it)."""
        shape, dtype = _LAYOUT_SHAPE[layout]
        if out is None:
            out = self.empty((self.n_active, *shape), dtype)
        self._check(self.lib.az_gather_leaves(self.h, _ptr(out, allow_pinned=True), layout, _stream()), "az_gather_leaves")
        return out

    def expand_backup(self, policy: torch.Tensor, values: torch.Tensor, policy_kind: int = POLICY_LOGITS):
        assert policy.dtype == torch.float32 and values.dtype == torch.float32
        assert policy.shape[0] >= self.n_active and policy.shape[-1] == 7 and values.shape[-1] == 2
        self._check(self.lib.az_expand_backup(self.h, _ptr(policy, allow_pinned=True), _ptr(values, allow_pinned=True), policy_kind, _stream()),
                    "az_expand_backup")

    def expand_backup_select(self, policy: torch.Tensor, values: torch.Tensor, policy_kind: int = POLICY_LOGITS):
        """`expand_backup` of this simulation and `select_leaves` of the next one in one launch."""
        assert policy.dtype == torch.float32 and values.dtype == torch.float32
        assert policy.shape[0] >= self.n_active and policy.shape[-1] == 7 and values.shape[-1] == 2
        self._check(self.lib.az_expand_backup_select(self.h, _ptr(policy, allow_pinned=True), _ptr(values, allow_pinned=True), policy_kind,
                                                     _stream()), "az_expand_backup_select")

    def leaf_compact(self):
        """The engine's list of the slots whose leaf waits for an evaluation and its length (`az_leaf_compact`), as views of the
        device arrays - `None` when the last selection ran without compaction."""
        lst, cnt = C.c_void_p(), C.c_void_p()
        self._check(self.lib.az_leaf_compact(self.h, C.byref(lst), C.byref(cnt)), "az_leaf_compact")
        if not lst.value or not cnt.value:
            return None

        class _Raw:
            def __init__(self, ptr, n):
                self.__cuda_array_interface__ = dict(shape=(n,), typestr="<i4", data=(ptr, False), version=2)

        return torch.as_tensor(_Raw(lst.value, self.num_games), device=self.device), torch.as_tensor(_Raw(cnt.value, 4), device=self.device)

    def leaf_info(self):
        n = self.n_active
        out = dict(bb0=self.empty(n, torch.int64), bb1=self.empty(n, torch.int64), player=self.empty(n, torch.uint8),
                   legal=self.empty(n, torch.uint8), status=self.empty(n, torch.uint8))
        self._check(self.lib.az_leaf_info(self.h, _ptr(out["bb0"]), _ptr(out["bb1"]), _ptr(out["player"]), _ptr(out["legal"]),
                                          _ptr(out["status"]), _stream()), "az_leaf_info")
        return out

    # -- results ---------------------------------------------------------------------------------
    def root_stats(self, out: dict | None = None):
        n = self.n_active
        if out is None:
            out = dict(child_N=self.empty((n, 7), torch.int32), child_W=self.empty((n, 7), torch.float64),
                       child_P=self.empty((n, 7), torch.float32), root_W=self.empty(n, torch.float64),
                       root_N=self.empty(n, torch.int32), legal=self.empty(n, torch.uint8), err=self.empty(n, torch.int32))
        self._check(self.lib.az_root_stats(self.h, _ptr(out.get("child_N")), _ptr(out.get("child_W")), _ptr(out.get("child_P")),
                                           _ptr(out.get("root_W")), _ptr(out.get("root_N")), _ptr(out.get("legal")),
                                           _ptr(out.get("err")), _stream()), "az_root_stats")
        return out

    def export_tree(self, slot: int):
        cap = self.tree_capacity
        W = self.empty(cap, torch.float64); N = self.empty(cap, torch.int32); P = self.empty(cap, torch.float32)
        CB = self.empty(cap, torch.int32)
        used = C.c_int32(0)
        self._check(self.lib.az_export_tree(self.h, int(slot), _ptr(W), _ptr(N), _ptr(P), _ptr(CB), C.byref(used)), "az_export_tree")
        u = used.value
        return dict(W=W[:u].cpu().numpy(), N=N[:u].cpu().numpy(), P=P[:u].cpu().numpy(), first_child=CB[:u].cpu().numpy(), used=u)

    # -- self-play -------------------------------------------------------------------------------
    def sample_moves(self, uniforms: torch.Tensor, finished: torch.Tensor | None = None):
        assert uniforms.dtype == torch.float64 and uniforms.numel() >= self.n_active
        self._check(self.lib.az_sample_moves(self.h, _ptr(uniforms), _ptr(finished), _stream()), "az_sample_moves")

    def run_move_step(self, num_sims: int, evaluator: int, uniforms: torch.Tensor, finished: torch.Tensor | None = None):
        """`run_simulations` + `sample_moves` in one launch (built-in evaluators): one self-play move step."""
        assert uniforms.dtype == torch.float64 and uniforms.numel() >= self.n_active
        self._check(self.lib.az_run_move_step(self.h, int(num_sims), int(evaluator), _ptr(uniforms), _ptr(finished), _stream()),
                    "az_run_move_step")

    def episode_counts(self) -> tuple[int, int]:
        ne, ns = C.c_int64(0), C.c_int64(0)
        self._check(self.lib.az_episode_counts(self.h, C.byref(ne), C.byref(ns), _stream()), "az_episode_counts")
        return ne.value, ns.value

    def alloc_drain_buffers(self) -> dict:
        """Device buffers that hold a full ring (2 E + 64 episodes of at most 42 samples): pass them to `drain_episodes_device`
        to drain without allocating (the caching allocator's occasional cudaMalloc is a host-side stall of tens of ms)."""
        ce = 2 * self.num_games + 64
        cs = ce * 42
        return dict(ep_slot=self.empty(ce, torch.int32), ep_step=self.empty(ce, torch.int32), ep_len=self.empty(ce, torch.int32),
                    ep_offset=self.empty(ce, torch.int64), ep_outcome=self.empty((ce, 2), torch.int8),
                    s_bb0=self.empty(cs, torch.int64), s_bb1=self.empty(cs, torch.int64), s_player=self.empty(cs, torch.uint8),
                    s_counts=self.empty((cs, 7), torch.int32))

    def drain_episodes_device(self, buffers: dict | None = None):
        """Ring -> device tensors (ring order, unsorted): fresh ones, or views of `buffers` (`alloc_drain_buffers`).  Used by the
        NCCL all-gather."""
        ne, ns = self.episode_counts()
        if buffers is not None:
            d = {k: (v[:ne] if k.startswith("ep_") else v[:ns]) for k, v in buffers.items()}
        else:
            d = dict(ep_slot=self.empty(ne, torch.int32), ep_step=self.empty(ne, torch.int32), ep_len=self.empty(ne, torch.int32),
                     ep_offset=self.empty(ne, torch.int64), ep_outcome=self.empty((ne, 2), torch.int8),
                     s_bb0=self.empty(ns, torch.int64), s_bb1=self.empty(ns, torch.int64), s_player=self.empty(ns, torch.uint8),
                     s_counts=self.empty((ns, 7), torch.int32))
        one, ons = C.c_int64(0), C.c_int64(0)
        self._check(self.lib.az_drain_episodes(self.h, ne, ns, _ptr(d["ep_slot"]), _ptr(d["ep_step"]), _ptr(d["ep_len"]),
                                               _ptr(d["ep_offset"]), _ptr(d["ep_outcome"]), _ptr(d["s_bb0"]), _ptr(d["s_bb1"]),
                                               _ptr(d["s_player"]), _ptr(d["s_counts"]), C.byref(one), C.byref(ons), _stream()),
                    "az_drain_episodes")
        assert one.value == ne and ons.value == ns
        return d

    # double-buffered ring: read one step's episodes on a copy stream while the next step runs
    def swap_episode_ring(self) -> int:
        prev = C.c_int32(0)
        self._check(self.lib.az_swap_episode_ring(self.h, C.byref(prev), _stream()), "az_swap_episode_ring")
        return prev.value

    def read_ring_to_host(self, ring: int, host: "PinnedEpisodeBuffers", stream: torch.cuda.Stream) -> EpisodeBatch | None:
        """Counters, then exactly-sized copies of ring `ring` into pinned host memory, all on `stream`."""
        ne, ns = C.c_int64(0), C.c_int64(0)
        self._check(self.lib.az_ring_counts(self.h, ring, C.byref(ne), C.byref(ns), stream.cuda_stream), "az_ring_counts")
        ne, ns = ne.value, ns.value
        if ne == 0:
            return None
        host.reserve(ne, ns)
        t = host.t
        self._check(self.lib.az_read_episode_ring(self.h, ring, ne, ns, t["ep_slot"].data_ptr(), t["ep_step"].data_ptr(),
                                                  t["ep_len"].data_ptr(), t["ep_offset"].data_ptr(), t["ep_outcome"].data_ptr(),
                                                  t["s_bb0"].data_ptr(), t["s_bb1"].data_ptr(), t["s_player"].data_ptr(),
                                                  t["s_counts"].data_ptr(), stream.cuda_stream), "az_read_episode_ring")
        stream.synchronize()
        d = {k: (v[:ne] if k.startswith("ep_") else v[:ns]).numpy() for k, v in t.items()}
        return sort_episode_batch(d)  # fancy indexing copies out of the pinned buffers

    def drain_episodes(self) -> EpisodeBatch:
        """Ring -> host, sorted into the reference's yield order (move step, then slot)."""
        d = {k: v.cpu().numpy() for k, v in self.drain_episodes_device().items()}
        return sort_episode_batch(d)

    # -- instrumentation -------------------------------------------------------------------------
    def stats(self) -> dict:
        st = AzStats()
        self._check(self.lib.az_get_stats(self.h, C.byref(st), _stream()), "az_get_stats")
        return {n: int(getattr(st, n)) for n, _ in AzStats._fields_}

    def selftest_division(self, n: int = 1 << 26, seed: int = 1) -> int:
        bad = C.c_int64(-1)
        self._check(self.lib.az_selftest_division(self.h, int(n), int(seed), C.byref(bad)), "az_selftest_division")
        return bad.value

    def reset_stats(self):
        self._check(self.lib.az_reset_stats(self.h, _stream()), "az_reset_stats")


class PinnedEpisodeBuffers:
    """Page-locked host staging for one ring read; grows geometrically."""

    _SPEC = dict(ep_slot=(torch.int32, ()), ep_step=(torch.int32, ()), ep_len=(torch.int32, ()), ep_offset=(torch.int64, ()),
                 ep_outcome=(torch.int8, (2,)), s_bb0=(torch.int64, ()), s_bb1=(torch.int64, ()), s_player=(torch.uint8, ()),
                 s_counts=(torch.int32, (7,)))

    def __init__(self):
        self.ne = self.ns = 0
        self.t: dict[str, torch.Tensor] = {}

    def reserve(self, ne: int, ns: int):
        if ne <= self.ne and ns <= self.ns:
            return
        self.ne, self.ns = max(2 * ne, self.ne, 64), max(2 * ns, self.ns, 1024)
        for k, (dt, tail) in self._SPEC.items():
            n = self.ne if k.startswith("ep_") else self.ns
            self.t[k] = torch.empty((n, *tail), dtype=dt).pin_memory()

    @property
    def nbytes(self) -> int:
        return sum(v.numel() * v.element_size() for v in self.t.values())


def sort_episode_batch(d: dict) -> EpisodeBatch:
    """Order episodes by (step, slot) and make their samples contiguous in that order."""
    order = np.lexsort((d["ep_slot"], d["ep_step"]))
    ep_len = d["ep_len"][order].astype(np.int32)
    old_off = d["ep_offset"][order]
    new_off = np.zeros(len(order), np.int64)
    if len(order):
        new_off[1:] = np.cumsum(ep_len[:-1])
    # sample i of the sorted batch comes from old position i + (old offset - new offset of its episode)
    idx = (np.arange(int(ep_len.sum()), dtype=np.int64) + np.repeat(old_off - new_off, ep_len)) if len(order) else np.zeros(0, np.int64)
    return EpisodeBatch(
        ep_slot=d["ep_slot"][order], ep_step=d["ep_step"][order], ep_len=ep_len, ep_offset=new_off,
        ep_outcome=d["ep_outcome"][order], s_bb0=d["s_bb0"][idx].view(np.uint64), s_bb1=d["s_bb1"][idx].view(np.uint64),
        s_player=d["s_player"][idx], s_counts=d["s_counts"][idx],
    )
