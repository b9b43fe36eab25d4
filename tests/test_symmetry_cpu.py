"""The host helpers of Connect4's left-right mirror symmetry (game.mirror_bitboards / canonical_bitboards) on positions played
by the oracle's rules: the mirror is the column flip of the grid, an involution, keeps the rules' verdicts, and the canonical
form is the same for a position and its mirror.  No GPU."""
import numpy as np

from alphazero_implementation_b200.game import bitboards_to_grid, canonical_bitboards, mirror_bitboards


def _positions(oracle, n, seed, max_plies=42):
    """n positions after 0..max_plies random legal moves (ended ones included: the game stops where it ended)."""
    rng = np.random.RandomState(seed)
    bb0, bb1, pl = np.zeros(n, np.uint64), np.zeros(n, np.uint64), np.zeros(n, np.uint8)
    target = rng.randint(0, max_plies + 1, size=n)
    for ply in range(max_plies):
        info = oracle.state_info(bb0, bb1, pl)
        go = np.nonzero((target > ply) & (info["ended"] == 0))[0]
        if not len(go):
            break
        legal = info["legal"][go]
        cols = np.array([rng.choice([c for c in range(7) if (m >> c) & 1]) for m in legal], np.uint8)
        nxt = oracle.env_step(bb0[go], bb1[go], pl[go], cols)
        bb0[go], bb1[go], pl[go] = nxt["bb0"], nxt["bb1"], nxt["player"]
    return bb0, bb1, pl


def _reverse7(m):
    m = np.asarray(m, np.uint8)
    return sum(((m >> c) & 1) << (6 - c) for c in range(7)).astype(np.uint8)


def test_mirror_is_the_column_flip_and_an_involution(oracle):
    bb0, bb1, _ = _positions(oracle, 3000, seed=1)
    m0, m1 = mirror_bitboards(bb0, bb1)
    for i in range(0, 3000, 7):
        assert np.array_equal(bitboards_to_grid(int(m0[i]), int(m1[i])), bitboards_to_grid(int(bb0[i]), int(bb1[i]))[:, ::-1])
    b0, b1 = mirror_bitboards(m0, m1)
    assert np.array_equal(b0, bb0) and np.array_equal(b1, bb1)
    assert not ((m0 | m1) & ~np.uint64(0xFDFBF7EFDFBF)).any()  # guard bits stay empty


def test_canonical_form(oracle):
    bb0, bb1, _ = _positions(oracle, 3000, seed=2)
    c0, c1, mir = canonical_bitboards(bb0, bb1)
    m0, m1 = mirror_bitboards(bb0, bb1)
    k0, k1, kmir = canonical_bitboards(m0, m1)
    assert np.array_equal(c0, k0) and np.array_equal(c1, k1)  # a position and its mirror share their canonical form
    d0, d1, dmir = canonical_bitboards(c0, c1)
    assert np.array_equal(d0, c0) and np.array_equal(d1, c1) and not dmir.any()  # idempotent
    # the smaller of the two, bb0 first; flagged exactly when the mirror was taken
    smaller = (m0 < bb0) | ((m0 == bb0) & (m1 < bb1))
    assert np.array_equal(mir, smaller)
    assert np.array_equal(c0, np.where(mir, m0, bb0)) and np.array_equal(c1, np.where(mir, m1, bb1))
    pal = (m0 == bb0) & (m1 == bb1)
    assert pal.any() and not mir[pal].any() and not kmir[pal].any()  # palindromes (the empty board at least) are not flagged
    assert mir.any() and kmir[~pal & ~mir].all()


def test_rules_of_the_mirror(oracle):
    bb0, bb1, pl = _positions(oracle, 4000, seed=3)
    m0, m1 = mirror_bitboards(bb0, bb1)
    a, b = oracle.state_info(bb0, bb1, pl), oracle.state_info(m0, m1, pl)
    assert a["ended"].any() and (a["ended"] == 0).any()
    assert np.array_equal(b["legal"], _reverse7(a["legal"]))
    assert np.array_equal(b["ended"], a["ended"]) and np.array_equal(b["reward"], a["reward"])
