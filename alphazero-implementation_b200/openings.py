"""Opening positions of self-play and arena games (`Engine.set_openings`; the rule is in include/az_engine.h).

Every game the engine plays starts from one position unless told otherwise.  With `Openings` each game starts from a position of a
set, or from the `reset_games` position, followed by a seeded number of random plies that neither win nor fill the board.  An
arena between deterministic agents then plays different games, and self-play visits more positions.
"""
from __future__ import annotations

from dataclasses import dataclass

import numpy as np

MAX_PLIES = 40


@dataclass(frozen=True, eq=False)
class Openings:
    """Where self-play games start.  The game of global slot g that starts at move step s takes a base position - entry i of
    `positions` drawn from (seed, g, s), or the `reset_games` position when `positions` is None - and plays r random plies,
    min_plies <= r <= max_plies, each drawn uniformly among the columns whose drop neither completes four nor fills the board.
    The random plies are not samples: a game's first sample is its opening.  `positions`: a list of `State`s or a (bb0, bb1,
    player) array triple.  `slot_offset` is the global index of the engine's first game, so sharded self-play draws what the
    unsharded run draws.  Off (None) by default."""

    positions: object = None
    min_plies: int = 0
    max_plies: int = 0
    seed: int = 0
    slot_offset: int = 0


def position_arrays(positions) -> tuple[np.ndarray, np.ndarray, np.ndarray]:
    """A list of `State`s or a (bb0, bb1, player) triple -> (bb0 uint64, bb1 uint64, player uint8) numpy arrays."""
    if isinstance(positions, tuple) and len(positions) == 3:
        bb0, bb1, pl = positions
        bb0, bb1, pl = (np.asarray(x.cpu() if hasattr(x, "cpu") else x) for x in (bb0, bb1, pl))
    else:
        positions = list(positions)
        bb0 = np.array([s.bb0 for s in positions], np.uint64)
        bb1 = np.array([s.bb1 for s in positions], np.uint64)
        pl = np.array([s.player for s in positions], np.uint8)
    bb0 = np.ascontiguousarray(bb0).astype(np.int64).view(np.uint64) if bb0.dtype != np.uint64 else np.ascontiguousarray(bb0)
    bb1 = np.ascontiguousarray(bb1).astype(np.int64).view(np.uint64) if bb1.dtype != np.uint64 else np.ascontiguousarray(bb1)
    if not (bb0.ndim == bb1.ndim == np.ndim(pl) == 1 and len(bb0) == len(bb1) == len(pl)):
        raise ValueError("positions: three 1-D arrays of equal length")
    return bb0, bb1, np.ascontiguousarray(pl, np.uint8)


def distinct_openings(k: int, plies: int, seed: int = 0, base=None, engine=None) -> tuple[np.ndarray, np.ndarray, np.ndarray]:
    """k openings of exactly `plies` random plies from `base` (a `State`; None = the empty board), pairwise distinct also up to the
    left-right mirror: the openings of slots 0, 1, 2, ... at move step 0 under `Openings([base], plies, plies, seed)`, keeping the
    first of each mirror-canonical form (`Engine.mirror_states`) until k are found.  -> (bb0, bb1, player) arrays in draw order,
    ready for `Openings(positions=...)` or an `Arena`.  `engine`: an `Engine` to draw with (its opening configuration is restored);
    None = a temporary one.  ValueError when the draws do not reach k distinct openings (few exist for small `plies`)."""
    from .engine import Engine

    if not 0 <= plies <= MAX_PLIES:
        raise ValueError(f"plies must be in [0, {MAX_PLIES}]")
    base = (np.zeros(1, np.uint64), np.zeros(1, np.uint64), np.zeros(1, np.uint8)) if base is None else [base]
    own = engine is None
    eng = Engine(1, 1) if own else engine
    keys: set = set()
    out: list = []
    try:
        saved = eng.openings
        eng.set_openings(Openings(base, plies, plies, seed))
        batch = max(1024, 4 * k)
        for first in range(0, 64 * batch, batch):
            o0, o1, pl = eng.opening_positions(first, batch, 0)
            m0, m1 = eng.mirror_states(o0, o1)
            o0, o1, m0, m1 = (x.cpu().numpy().view(np.uint64) for x in (o0, o1, m0, m1))
            pl = pl.cpu().numpy()
            mirrored = (m0 < o0) | ((m0 == o0) & (m1 < o1))
            c0, c1 = np.where(mirrored, m0, o0), np.where(mirrored, m1, o1)
            for i in range(batch):
                key = (int(c0[i]), int(c1[i]), int(pl[i]))
                if key not in keys:
                    keys.add(key)
                    out.append((o0[i], o1[i], pl[i]))
            if len(out) >= k:
                break
        eng.set_openings(saved)
    finally:
        if own:
            eng.close()
    if len(out) < k:
        raise ValueError(f"only {len(out)} distinct {plies}-ply openings found, {k} asked for")
    out = out[:k]
    return (np.array([o[0] for o in out], np.uint64), np.array([o[1] for o in out], np.uint64), np.array([o[2] for o in out], np.uint8))
