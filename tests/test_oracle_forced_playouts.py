"""CPU: the forced-playouts oracle (tests/native/c4_forced_oracle.c: c4o_selfplay_forced, c4o_prune) - the yardstick the GPU tests of
the library's forced playouts and policy target pruning hold it against.  k = 0 is the cap / noise / reuse / plain oracle bit for bit;
the numpy restatement of the pruning is the C one, on random and adversarial root statistics; pruned counts keep the rule's
invariants."""
import numpy as np
import pytest

import cap_oracle
import forced_oracle
import noise_oracle
import reuse_oracle

FIELDS = ("ep_slot", "ep_len", "ep_step", "ep_outcome", "s_bb0", "s_bb1", "s_player", "s_counts")


def _same(ref, got):
    for f in FIELDS:
        assert np.array_equal(getattr(ref, f), getattr(got, f)), f
    assert (ref.n_steps, ref.n_uniforms_used, ref.n_sims, ref.n_evals) == (got.n_steps, got.n_uniforms_used, got.n_sims, got.n_evals)


@pytest.mark.parametrize("eval_kind", [1, 2])
def test_k0_is_the_plain_oracle(oracle, eval_kind):
    E, S, steps = 48, 40, 70
    u = np.random.RandomState(3).random_sample((steps, E))
    ref = oracle.selfplay(E, S, u, eval_kind=eval_kind)
    got, extra = forced_oracle.selfplay_forced(E, S, 0.0, u, eval_kind=eval_kind)
    _same(ref, got)
    assert extra["forced_selections"] == 0 and extra["visits_pruned"] == 0 and extra["children_zeroed"] == 0
    assert extra["forced_searches"] == got.n_uniforms_used


@pytest.mark.parametrize("greedy_from", [-1, 8])
def test_k0_is_the_noise_oracle(greedy_from):
    E, S, steps = 40, 30, 80
    u = np.random.RandomState(8).random_sample((steps, E))
    eta = np.random.RandomState(9).dirichlet(np.ones(7), size=(steps, E)).astype(np.float32)
    ref = noise_oracle.selfplay_noise(E, S, u, 0.25, eta, greedy_from=greedy_from, eval_kind=2)
    got, _ = forced_oracle.selfplay_forced(E, S, 0.0, u, eps=0.25, eta=eta, greedy_from=greedy_from, eval_kind=2)
    _same(ref, got)


def test_k0_is_the_reuse_oracle():
    E, S, V, steps = 32, 30, 120, 80
    u = np.random.RandomState(10).random_sample((steps, E))
    ref, rst = reuse_oracle.selfplay_reuse(E, S, V, u, eval_kind=2)
    got, extra = forced_oracle.selfplay_forced(E, S, 0.0, u, V=V, eval_kind=2)
    _same(ref, got)
    assert rst["retained"] > 0 and all(rst[k] == extra[k] for k in rst)


@pytest.mark.parametrize("visit_budget", [False, True])
def test_k0_is_the_cap_oracle(visit_budget):
    E, S, F, V, steps = 32, 40, 8, 160, 80
    u = np.random.RandomState(13).random_sample((steps, E))
    full = (np.random.RandomState(14).random_sample((steps, E)) < 0.5).astype(np.uint8)
    eta = np.random.RandomState(15).dirichlet(np.ones(7), size=(steps, E)).astype(np.float32)
    ref, re_ = cap_oracle.selfplay_cap(E, S, F, full, u, V=V, visit_budget=visit_budget, eps=0.25, eta=eta, greedy_from=10, eval_kind=2)
    got, ge = forced_oracle.selfplay_forced(E, S, 0.0, u, full=full, fast_sims=F, V=V, visit_budget=visit_budget, eps=0.25, eta=eta,
                                            greedy_from=10, eval_kind=2)
    _same(ref, got)
    assert np.array_equal(re_["last_counts"], ge["last_counts"]) and re_["samples_dropped"] == ge["samples_dropped"]


def _random_roots(rs, n, S=800):
    """root statistics of the shape a search leaves: counts summing to N_root - 1 over the legal columns, means in [-1, 1]"""
    legal = rs.randint(1, 128, n).astype(np.uint8)
    lg = ((legal[:, None] >> np.arange(7)) & 1).astype(bool)
    P = np.where(lg, rs.dirichlet(np.ones(7) * 0.5, n), 0).astype(np.float32)
    root_N = rs.randint(1, S + 1, n).astype(np.int32)
    w = np.where(lg, rs.dirichlet(np.ones(7) * 0.3, n), 0)
    w = w / w.sum(1, keepdims=True)
    N = np.zeros((n, 7), np.int32)
    for i in range(n):
        N[i] = rs.multinomial(root_N[i] - 1, w[i])
    W = np.where(N > 0, N * rs.uniform(-1, 1, (n, 7)), 0.0)
    W = np.round(W * 128) / 128  # dyadic, like the hash evaluator's values
    return N, W, P, legal, root_N


def _adversarial_roots():
    rows = []
    def add(N, W, P, legal, root_N):
        rows.append((np.array(N, np.int32), np.array(W, np.float64), np.array(P, np.float32), legal, root_N))
    add([5, 5, 3, 0, 0, 0, 0], [1.0, -1.0, 0.5, 0, 0, 0, 0], [0.2, 0.3, 0.1, 0.1, 0.1, 0.1, 0.1], 0x7F, 14)  # tie for c*
    add([0] * 7, [0.0] * 7, [1 / 7] * 7, 0x7F, 1)                                                       # M = 0
    add([0, 0, 0, 9, 0, 0, 0], [0, 0, 0, 2.0, 0, 0, 0], [0, 0, 0, 1.0, 0, 0, 0], 0x08, 10)               # one legal column
    add([6, 1, 1, 1, 0, 0, 0], [1.0, 0.0, -0.5, 0.25, 0, 0, 0], [0.5, 0.0, 0.0, 0.5, 0, 0, 0], 0x0F, 10)  # P = 0, N = 1
    add([3, 20, 2, 1, 1, 1, 1], [0.0, 5.0, 0.0, 0.0, 1.0, -1.0, 0.0], [0.05, 0.05, 0.6, 0.1, 0.1, 0.05, 0.05], 0x7F, 30)  # n_f > N
    add([1, 1, 1, 1, 1, 1, 1], [0.0] * 7, [1 / 7] * 7, 0x7F, 8)                                           # all ones: c* = column 0
    add([40, 0, 2, 0, 0, 0, 0], [-30.0, 0, 1.5, 0, 0, 0, 0], [0.01, 0.0, 0.99, 0, 0, 0, 0], 0x05, 43)     # c* with a bad mean
    N, W, P, legal, root_N = (np.stack([r[i] for r in rows]) if i < 3 else np.array([r[i] for r in rows]) for i in range(5))
    return N, W, P, legal.astype(np.uint8), root_N.astype(np.int32)


def _invariants(N, W, P, legal, root_N, c_puct, k, Np):
    n_f = forced_oracle.n_forced(P, root_N, k)
    lg = ((legal[:, None].astype(np.int64) >> np.arange(7)) & 1).astype(bool)
    bc = np.argmax(np.where(lg, N, -1), axis=1)
    rows = np.arange(len(N))
    active = (root_N > 1) & (k != 0)
    assert (Np[rows, bc] == N[rows, bc]).all()
    assert ((Np >= 0) & (Np <= N)).all()
    off = np.ones_like(lg)
    off[rows, bc] = False
    assert not ((Np == 1) & off & active[:, None]).any()
    one_to_zero = (Np == 0) & (N - Np <= n_f + 1)  # the bound, then the last visit by the 1 -> 0 step
    assert ((N - Np <= n_f) | one_to_zero | ~active[:, None]).all()
    assert (Np[~active] == N[~active]).all()
    # no remaining child could lose one more visit: the bound, N' = 0 or the score stops it
    sq = np.sqrt(root_N.astype(np.float64))
    Pd = P.astype(np.float64)
    q = np.where(W == 0.0, 0.0, W / np.maximum(N, 1))
    qb = q[rows, bc]
    s_star = qb + ((c_puct * Pd[rows, bc]) * sq) / (1.0 + N[rows, bc])
    with np.errstate(divide="ignore", invalid="ignore"):
        score = q + ((c_puct * Pd) * sq[:, None]) / Np
    could = lg & off & active[:, None] & (N > 0) & (Np > 1) & (N - Np < n_f) & (score < s_star[:, None])
    assert not could.any()


@pytest.mark.parametrize("k", [0.0, 0.5, 2.0, 7.5, 1024.0])
@pytest.mark.parametrize("c_puct", [1.0, 1.25])
def test_numpy_pruning_is_the_c_pruning(k, c_puct):
    rs = np.random.RandomState(int(k * 10) + int(c_puct * 100))
    for N, W, P, legal, root_N in (_random_roots(rs, 4000), _random_roots(rs, 2000, S=40), _adversarial_roots()):
        a = forced_oracle.prune_np(N, W, P, legal, root_N, c_puct, k)
        b, (pruned, zeroed) = forced_oracle.prune_c(N, W, P, legal, root_N, c_puct, k)
        assert np.array_equal(a, b)
        assert pruned == int((N - b).sum()) and zeroed == int(((N > 0) & (b == 0)).sum())
        _invariants(N, W, P, legal, root_N, c_puct, k, b)
        if k == 0.0:
            assert np.array_equal(b, N)


def test_adversarial_cases_do_what_the_rule_says():
    N, W, P, legal, root_N = _adversarial_roots()
    b, _ = forced_oracle.prune_c(N, W, P, legal, root_N, 1.0, 2.0)
    assert b[0, 0] == 5 and b[0, 1] <= 5          # tie for c*: the lowest column keeps its count
    assert np.array_equal(b[1], N[1])              # M = 0: untouched
    assert np.array_equal(b[2], N[2])              # one legal column: c* alone
    assert b[3, 1] == 0 and b[3, 2] == 0           # P = 0, N = 1: no forced visits, but 1 -> 0
    assert (b[5, 1:] == 0).all() and b[5, 0] == 1  # all ones: c* is column 0, the others go to 0


def test_forcing_spreads_visits_and_pruning_takes_them_back():
    E, S, steps = 48, 60, 60
    u = np.random.RandomState(21).random_sample((steps, E))
    eta = np.random.RandomState(22).dirichlet(np.ones(7) * 0.3, size=(steps, E)).astype(np.float32)
    plain, _ = forced_oracle.selfplay_forced(E, S, 0.0, u, eps=0.25, eta=eta, eval_kind=2)
    got, extra = forced_oracle.selfplay_forced(E, S, 2.0, u, eps=0.25, eta=eta, eval_kind=2)
    assert extra["forced_selections"] > 0 and extra["visits_pruned"] > 0 and extra["children_zeroed"] > 0
    assert extra["forced_searches"] == got.n_uniforms_used
    sums = got.s_counts.sum(1)
    assert (sums <= S - 1).all() and (sums > 0).all() and (sums < S - 1).any()
    assert not np.array_equal(plain.s_counts, got.s_counts)
