"""CPU: the noise oracle's entry points (tests/native/c4_noise_oracle.c: c4o_search_noise, c4o_selfplay_noise) - the yardstick the GPU tests
of the library's noise hold it against.  Noise off (fraction 0, cutoff past the last ply) is plain c4o_selfplay bit for bit; the
mixing is the fp32 formula; past the cutoff every move is the first maximum of the recorded visit counts."""
import numpy as np
import pytest

import noise_oracle

FIELDS = ("ep_slot", "ep_len", "ep_step", "ep_outcome", "s_bb0", "s_bb1", "s_player", "s_counts")


def random_positions(oracle, n, plies, seed):
    """n positions reached by `plies` random legal moves from the empty board (games that end early stay where they ended)."""
    rng = np.random.RandomState(seed)
    b0 = np.zeros(n, np.uint64); b1 = np.zeros(n, np.uint64); pl = np.zeros(n, np.uint8)
    for _ in range(plies):
        info = oracle.state_info(b0, b1, pl)
        live = (info["ended"] == 0) & (info["legal"] != 0)
        if not live.any():
            break
        col = np.array([rng.choice([c for c in range(7) if (m >> c) & 1]) if ok else 0 for m, ok in zip(info["legal"], live)], np.uint8)
        nxt = oracle.env_step(b0, b1, pl, col)
        ok = live & (nxt["ended"] == 0)
        b0 = np.where(ok, nxt["bb0"], b0); b1 = np.where(ok, nxt["bb1"], b1); pl = np.where(ok, nxt["player"], pl)
    return b0, b1, pl


def played_column(bb0, bb1, nbb0, nbb1):
    diff = int((int(nbb0) | int(nbb1)) ^ (int(bb0) | int(bb1)))
    assert diff and diff & (diff - 1) == 0
    return (diff.bit_length() - 1) // 7  # bit index = column * 7 + row


@pytest.mark.parametrize("eval_kind", [1, 2])
def test_selfplay_noise_off_is_selfplay(oracle, eval_kind):
    E, S, steps = 48, 40, 70
    u = np.random.RandomState(3).random_sample((steps, E))
    eta = np.random.RandomState(4).dirichlet(np.ones(7), size=(steps, E)).astype(np.float32)
    ref = oracle.selfplay(E, S, u, eval_kind=eval_kind)
    got = noise_oracle.selfplay_noise(E, S, u, 0.0, eta, greedy_from=42, eval_kind=eval_kind)
    assert len(ref.ep_slot) == E
    for f in FIELDS:
        assert np.array_equal(getattr(ref, f), getattr(got, f)), f
    assert (ref.n_steps, ref.n_uniforms_used, ref.n_sims, ref.n_evals) == (got.n_steps, got.n_uniforms_used, got.n_sims, got.n_evals)


@pytest.mark.parametrize("eps", [0.25, 1.0, 0.1])
def test_search_noise_mixes_in_fp32(oracle, eps):
    E, S = 96, 30
    b0, b1, pl = random_positions(oracle, E, 9, seed=5)
    info = oracle.state_info(b0, b1, pl)
    keep = info["ended"] == 0
    b0, b1, pl = b0[keep], b1[keep], pl[keep]
    E = len(b0)
    legal = oracle.state_info(b0, b1, pl)["legal"]
    rng = np.random.RandomState(6)
    eta = np.zeros((E, 7), np.float32)
    for i in range(E):
        cols = [c for c in range(7) if (legal[i] >> c) & 1]
        eta[i, cols] = rng.dirichlet(np.full(len(cols), 0.3)).astype(np.float32)
    before = oracle.search(b0, b1, pl, 1, eval_kind=2)  # simulation 1 expands the root with the evaluator's priors
    got = noise_oracle.search_noise(b0, b1, pl, S, eps, eta, eval_kind=2)
    e32 = np.float32(eps)
    want = (np.float32(1) - e32) * before["child_P"] + e32 * eta  # float32 arrays: one rounding per operation
    want = np.where(before["child_P"] > 0, want, np.float32(0))
    assert want.dtype == np.float32
    assert np.array_equal(got["child_P"].view(np.uint32), want.view(np.uint32))
    assert (got["root_N"] == S).all() and (got["child_N"].sum(1) == S - 1).all()
    # the noise changes the search: some visit distribution differs from the noiseless one
    plain = oracle.search(b0, b1, pl, S, eval_kind=2)
    assert (plain["child_N"] != got["child_N"]).any()


@pytest.mark.parametrize("greedy_from", [0, 6, 12])
def test_cutoff_plays_the_first_argmax(oracle, greedy_from):
    E, S, steps = 40, 30, 80
    u = np.random.RandomState(8).random_sample((steps, E))
    eta = np.random.RandomState(9).dirichlet(np.ones(7), size=(steps, E)).astype(np.float32)
    r = noise_oracle.selfplay_noise(E, S, u, 0.25, eta, greedy_from=greedy_from, eval_kind=2)
    assert len(r.ep_slot) == E
    sampled_off_argmax = 0
    off = 0
    for e in range(len(r.ep_slot)):
        n = int(r.ep_len[e])
        for k in range(n - 1):  # the last move is not recorded as a position
            i = off + k
            col = played_column(r.s_bb0[i], r.s_bb1[i], r.s_bb0[i + 1], r.s_bb1[i + 1])
            first_max = int(np.argmax(r.s_counts[i]))
            if k >= greedy_from:
                assert col == first_max, (e, k)
            elif col != first_max:
                sampled_off_argmax += 1
        off += n
    if greedy_from > 0:
        assert sampled_off_argmax > 0  # before the cutoff the moves are still sampled
