"""CPU: the cap oracle (tests/native/c4_cap_oracle.c: c4o_selfplay_cap, c4o_cap_draw) - the yardstick the GPU tests of the
library's playout cap randomization hold it against.  Every search full is the plain / noise / reuse oracle bit for bit; every
search fast with fast_sims = S plays the same games with every sample dropped; the numpy restatement of the engine's draw is the
C one."""
import numpy as np
import pytest

import cap_oracle
import noise_oracle
import reuse_oracle

FIELDS = ("ep_slot", "ep_len", "ep_step", "ep_outcome", "s_bb0", "s_bb1", "s_player", "s_counts")
GAME_FIELDS = ("ep_slot", "ep_step", "ep_outcome")


@pytest.mark.parametrize("eval_kind", [1, 2])
def test_all_full_is_selfplay(oracle, eval_kind):
    E, S, steps = 48, 40, 70
    u = np.random.RandomState(3).random_sample((steps, E))
    ref = oracle.selfplay(E, S, u, eval_kind=eval_kind)
    got, extra = cap_oracle.selfplay_cap(E, S, 7, np.ones((steps, E), np.uint8), u, eval_kind=eval_kind)
    assert len(ref.ep_slot) == E
    for f in FIELDS:
        assert np.array_equal(getattr(ref, f), getattr(got, f)), f
    assert (ref.n_steps, ref.n_uniforms_used, ref.n_sims, ref.n_evals) == (got.n_steps, got.n_uniforms_used, got.n_sims, got.n_evals)
    assert extra["samples_dropped"] == 0


@pytest.mark.parametrize("greedy_from", [-1, 8])
def test_all_full_is_noise_oracle(greedy_from):
    E, S, steps = 40, 30, 80
    u = np.random.RandomState(8).random_sample((steps, E))
    eta = np.random.RandomState(9).dirichlet(np.ones(7), size=(steps, E)).astype(np.float32)
    ref = noise_oracle.selfplay_noise(E, S, u, 0.25, eta, greedy_from=greedy_from, eval_kind=2)
    got, _ = cap_oracle.selfplay_cap(E, S, 5, np.ones((steps, E), np.uint8), u, eps=0.25, eta=eta, greedy_from=greedy_from, eval_kind=2)
    for f in FIELDS:
        assert np.array_equal(getattr(ref, f), getattr(got, f)), f
    assert (ref.n_sims, ref.n_evals) == (got.n_sims, got.n_evals)


def test_all_full_is_reuse_oracle():
    E, S, V, steps = 32, 30, 120, 80
    u = np.random.RandomState(10).random_sample((steps, E))
    ref, rst = reuse_oracle.selfplay_reuse(E, S, V, u, eval_kind=2)
    got, extra = cap_oracle.selfplay_cap(E, S, 4, np.ones((steps, E), np.uint8), u, V=V, eval_kind=2)
    for f in FIELDS:
        assert np.array_equal(getattr(ref, f), getattr(got, f)), f
    assert rst["retained"] > 0 and all(rst[k] == extra[k] for k in rst)


@pytest.mark.parametrize("eval_kind", [1, 2])
def test_all_fast_at_full_size_drops_every_sample(oracle, eval_kind):
    E, S, steps = 48, 40, 70
    u = np.random.RandomState(4).random_sample((steps, E))
    ref = oracle.selfplay(E, S, u, eval_kind=eval_kind)
    got, extra = cap_oracle.selfplay_cap(E, S, S, np.zeros((steps, E), np.uint8), u, eval_kind=eval_kind)
    for f in GAME_FIELDS:
        assert np.array_equal(getattr(ref, f), getattr(got, f)), f
    assert (got.ep_len == 0).all() and len(got.s_bb0) == 0
    assert extra["samples_dropped"] == int(ref.ep_len.sum())
    assert (ref.n_sims, ref.n_evals) == (got.n_sims, got.n_evals)


def test_mixed_budgets_keep_the_full_samples():
    """A fast search is a shorter search: its counts sum to fast_sims - 1; the recorded samples are exactly the full plies."""
    E, S, F, steps = 40, 50, 10, 90
    u = np.random.RandomState(11).random_sample((steps, E))
    full = (np.random.RandomState(12).random_sample((steps, E)) < 0.3).astype(np.uint8)
    got, extra = cap_oracle.selfplay_cap(E, S, F, full, u, eval_kind=2)
    assert (got.s_counts.sum(1) == S - 1).all()
    # the same games with every search recorded (all flags 1 would change the games): compare against fast_sims = S per flag 0
    assert got.n_sims == int(np.where(full[:got.n_steps], S, F).sum())
    assert extra["samples_dropped"] > 0 and got.ep_len.sum() > 0


def test_visit_budget_without_reuse_is_the_plain_cap():
    E, S, F, steps = 32, 40, 8, 80
    u = np.random.RandomState(13).random_sample((steps, E))
    full = (np.random.RandomState(14).random_sample((steps, E)) < 0.5).astype(np.uint8)
    a, ea = cap_oracle.selfplay_cap(E, S, F, full, u, eval_kind=2)
    b, eb = cap_oracle.selfplay_cap(E, S, F, full, u, visit_budget=True, eval_kind=2)
    for f in FIELDS:
        assert np.array_equal(getattr(a, f), getattr(b, f)), f
    assert a.n_sims == b.n_sims and np.array_equal(ea.pop("last_counts"), eb.pop("last_counts")) and ea == eb


def test_visit_budget_with_reuse_runs_fewer_simulations():
    E, S, V, steps = 32, 40, 160, 80
    u = np.random.RandomState(15).random_sample((steps, E))
    full = np.ones((steps, E), np.uint8)
    a, ea = cap_oracle.selfplay_cap(E, S, S, full, u, V=V, eval_kind=2)
    b, eb = cap_oracle.selfplay_cap(E, S, S, full, u, V=V, visit_budget=True, eval_kind=2)
    assert ea["retained"] > 0 and eb["retained"] > 0
    assert b.n_sims < a.n_sims
    # a search ends with max(S, N_start + 1) root visits: the recorded counts sum to at least S - 1
    assert (b.s_counts.sum(1) >= S - 1).all()


@pytest.mark.parametrize("seed,offset,step,p", [(0, 0, 0, 0.25), (12345678901234567, 7, 3, 0.1), (2**64 - 1, 2**40 + 5, 1000, 0.9),
                                                (99, 1 << 33, 2**32 - 1, 1.0), (5, 3, 9, 0.0)])
def test_numpy_draw_is_the_c_draw(seed, offset, step, p):
    n = 4096
    a = cap_oracle.draw_full(seed, offset, n, step, p)
    b = cap_oracle.draw_full_c(seed, offset, n, step, p)
    assert np.array_equal(a, b)
    if 0.0 < p < 1.0:
        k = int(a.sum())
        assert abs(k - n * p) < 6 * np.sqrt(n * p * (1 - p))
    else:
        assert (a == (1 if p == 1.0 else 0)).all()
