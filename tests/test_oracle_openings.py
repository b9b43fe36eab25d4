"""Opening positions (az_set_openings): the C restatement of the rule (tests/native/c4_openings_oracle.c) against a plain-Python one
on thousands of games, the random plies are legal and never end the game, the degenerate cases, and the self-play oracle built on it:
the mode off is c4o_selfplay_forced, and with it on every game's first sample is its opening.  CPU only."""
import numpy as np
import pytest

import forced_oracle
import openings_oracle as oo

# a drawn full board (no four for either side) with the top stone of column 3 taken away: the one legal drop fills the board
FULL0, FULL1 = 0xD1A0B1665334, 0x2C5B46898C8B
TOP3 = 1 << (7 * 3 + 5)
NO_MOVE = (FULL0 & ~TOP3, FULL1 & ~TOP3, 0)
SET = (np.array([0, 1 << 21, 0, NO_MOVE[0]], np.uint64), np.array([0, 1 << 14, 1 << 21, NO_MOVE[1]], np.uint64),
       np.array([0, 0, 0, 1], np.uint8))

CONFIGS = [dict(min_plies=0, max_plies=8, seed=1), dict(min_plies=4, max_plies=4, seed=2**63 + 12345),
           dict(positions=SET, min_plies=2, max_plies=6, seed=7), dict(min_plies=30, max_plies=40, seed=3),
           dict(min_plies=0, max_plies=3, seed=9, init=(1 << 21, 1 << 22, 0))]


def _pairs(n, seed):
    rs = np.random.RandomState(seed)
    g = np.concatenate([np.arange(n // 2), rs.randint(0, 2**62, n - n // 2, dtype=np.int64)]).astype(np.int64)
    s = rs.randint(0, 5000, n).astype(np.int64)
    return g, s


@pytest.mark.parametrize("cfg", CONFIGS, ids=range(len(CONFIGS)))
def test_oracle_is_the_python_rule(cfg):
    g, s = _pairs(600, 11)
    for gi, si in zip(g.tolist(), s.tolist()):
        (b0, b1, pl), cols = oo.opening_py(gi, si, **cfg)
        c0, c1, cp = oo.openings_c(gi, 1, si, **cfg)
        assert (int(c0[0]), int(c1[0]), int(cp[0])) == (b0, b1, pl), (gi, si)


@pytest.mark.parametrize("cfg", CONFIGS, ids=range(len(CONFIGS)))
def test_random_plies_are_legal_and_never_end_the_game(cfg):
    """Replayed from the base, each column is legal and leaves a game that has not ended; an opening shorter than its draw stops
    only where no such column exists."""
    o0, o1, op = oo.openings_c(0, 200, 17, **cfg)
    lengths = []
    for i in range(200):
        (b0, b1, pl), cols = oo.opening_py(i, 17, **cfg)
        x0 = oo._x(cfg.get("seed", 0), i, 17, 0)
        pos = cfg.get("positions")
        if pos is None:
            c = cfg.get("init", (0, 0, 0))
        else:
            j = (x0[0] * len(pos[0])) >> 32
            c = (int(pos[0][j]), int(pos[1][j]), int(pos[2][j]))
        r = cfg["min_plies"] + ((x0[1] * (cfg["max_plies"] - cfg["min_plies"] + 1)) >> 32)
        for col in cols:
            nxt = oo.drop(*c, col)
            assert nxt is not None and not oo.ended(nxt[0], nxt[1])
            c = nxt
        assert c == (b0, b1, pl) == (int(o0[i]), int(o1[i]), int(op[i]))
        assert len(cols) <= r
        if len(cols) < r:
            assert all(oo.drop(*c, k) is None or oo.ended(*oo.drop(*c, k)[:2]) for k in range(7))
        lengths.append(len(cols))
    assert max(lengths) > 0


def test_zero_plies_give_the_base():
    o0, o1, op = oo.openings_c(0, 256, 3, min_plies=0, max_plies=0, seed=4, init=(1 << 21, 1 << 14, 0))
    assert (o0 == 1 << 21).all() and (o1 == 1 << 14).all() and (op == 0).all()
    o0, o1, op = oo.openings_c(0, 4096, 3, positions=SET, min_plies=0, max_plies=0, seed=4)
    got = set(zip(o0.tolist(), o1.tolist(), op.tolist()))
    assert got == set(zip(SET[0].tolist(), SET[1].tolist(), SET[2].tolist()))


def test_base_without_a_non_ending_move_stops_early():
    assert not oo.ended(NO_MOVE[0], NO_MOVE[1])
    assert oo.drop(*NO_MOVE, 3) is not None and oo.ended(*oo.drop(*NO_MOVE, 3)[:2])
    pos = tuple(np.array([x]) for x in NO_MOVE)
    o0, o1, op = oo.openings_c(0, 64, 0, positions=(pos[0].astype(np.uint64), pos[1].astype(np.uint64), pos[2].astype(np.uint8)),
                               min_plies=1, max_plies=40, seed=8)
    assert (o0 == NO_MOVE[0]).all() and (o1 == NO_MOVE[1]).all() and (op == NO_MOVE[2]).all()


EP_FIELDS = ("ep_slot", "ep_step", "ep_len", "ep_outcome", "s_bb0", "s_bb1", "s_player", "s_counts")


def test_selfplay_oracle_off_is_the_forced_oracle():
    E, S, steps = 96, 24, 30
    u = np.random.RandomState(3).random_sample((steps, E))
    a, _ = oo.selfplay_openings(E, S, u, min_plies=0, max_plies=6, seed=5, off=True, quota=E * steps, eval_kind=2)
    b, _ = forced_oracle.selfplay_forced(E, S, 0.0, u, quota=E * steps, eval_kind=2)
    for f in EP_FIELDS:
        assert np.array_equal(getattr(a, f), getattr(b, f)), f


@pytest.mark.parametrize("positions", [None, tuple(x[:3] for x in SET)])
def test_selfplay_oracle_first_sample_is_the_opening(positions):
    E, S, steps, off = 96, 24, 40, 1000
    u = np.random.RandomState(4).random_sample((steps, E))
    kw = dict(positions=positions, min_plies=0, max_plies=6, seed=6)
    r, _ = oo.selfplay_openings(E, S, u, slot_offset=off, quota=E * steps, eval_kind=2, **kw)
    assert len(r.ep_slot) > E
    start = np.cumsum(r.ep_len) - r.ep_len
    for i in range(len(r.ep_slot)):
        s = int(r.ep_step[i] - r.ep_len[i] + 1)
        o0, o1, op = oo.openings_c(off + int(r.ep_slot[i]), 1, s, **kw)
        j = start[i]
        assert (r.s_bb0[j], r.s_bb1[j], r.s_player[j]) == (o0[0], o1[0], op[0])
    assert len({(int(r.s_bb0[j]), int(r.s_bb1[j])) for j in start}) > len(r.ep_slot) // 4
