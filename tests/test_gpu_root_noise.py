"""GPU: AlphaZero's self-play exploration - Dirichlet noise on the root priors (k_root_noise, az_apply_root_noise) and the greedy
cutoff of the move step (az_set_greedy_from).  The noise has the Dirichlet law, is a pure function of (seed, global slot, draw,
column), is mixed in fp32 exactly, is the identity at fraction 0, and the searches around it match the C oracle fed the noise the
engine drew - on the built-in evaluators and with ResNet 4x64 in the loop, evaluation cache and CUDA graph on or off."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

import alphazero_implementation_b200 as az  # noqa: E402
from alphazero_implementation_b200.engine import POLICY_LOGITS, Engine  # noqa: E402
import noise_oracle  # noqa: E402

EP_FIELDS = ("ep_slot", "ep_step", "ep_len", "ep_outcome", "s_bb0", "s_bb1", "s_player", "s_counts")


# ---- helpers -------------------------------------------------------------------------------------------------------------------
def full_columns(cols):
    """A position whose columns `cols` are full (stones alternate up every column: no four in a line while no four neighbouring
    columns are filled), player 0 to move: 7 - len(cols) legal columns."""
    b0 = b1 = 0
    for c in cols:
        for r in range(6):
            if r % 2 == 0:
                b0 |= 1 << (c * 7 + r)
            else:
                b1 |= 1 << (c * 7 + r)
    return b0, b1


FULL = {7: (), 6: (0,), 5: (0, 3), 4: (0, 3, 6), 3: (0, 2, 4, 6), 2: (0, 1, 3, 4, 6), 1: (0, 1, 2, 4, 5, 6)}


def random_positions(oracle, n, seed, max_plies=26):
    """n non-terminal positions after 0..max_plies random legal moves."""
    rng = np.random.RandomState(seed)
    bb0, bb1, pl = np.zeros(n, np.uint64), np.zeros(n, np.uint64), np.zeros(n, np.uint8)
    target = rng.randint(0, max_plies + 1, size=n)
    legal = np.full(n, 0x7F, np.uint8)
    for ply in range(max_plies):
        go = np.nonzero(target > ply)[0]
        if not len(go):
            break
        r = rng.random_sample(len(go))
        cols = np.zeros(len(go), np.uint8)
        for j, i in enumerate(go):
            opts = [c for c in range(7) if (legal[i] >> c) & 1]
            cols[j] = opts[int(r[j] * len(opts))]
        nxt = oracle.env_step(bb0[go], bb1[go], pl[go], cols)
        ok = (nxt["status"] == 0) & (nxt["ended"] == 0)
        keep = go[ok]
        bb0[keep], bb1[keep], pl[keep], legal[keep] = nxt["bb0"][ok], nxt["bb1"][ok], nxt["player"][ok], nxt["legal"][ok]
        target[go[~ok]] = 0
    return bb0, bb1, pl


def draw_eta(E, alpha, seed=1, slot_offset=0, pos=(0, 0), draws=1, lanes=0):
    """eta of `draws` consecutive searches (one simulation, the noise) on E copies of position `pos`."""
    eng = Engine(num_games=E, num_simulations=2, lanes_per_tree=lanes)
    eng.set_root_noise(alpha, 0.25, seed, slot_offset)
    out = []
    for _ in range(draws):
        eng.set_roots(np.full(E, pos[0], np.uint64), np.full(E, pos[1], np.uint64), np.zeros(E, np.uint8))
        eng.run_simulations(1, 1)
        eng.apply_root_noise()
        out.append(eng.root_noise_values().cpu().numpy())
    eng.close()
    return out


def flatten(parts):
    eps = []
    for b in parts:
        for e in range(len(b)):
            o, n = int(b.ep_offset[e]), int(b.ep_len[e])
            eps.append(dict(slot=int(b.ep_slot[e]), step=int(b.ep_step[e]), outcome=b.ep_outcome[e].tolist(),
                            bb0=b.s_bb0[o:o + n].tolist(), bb1=b.s_bb1[o:o + n].tolist(), player=b.s_player[o:o + n].tolist(),
                            counts=b.s_counts[o:o + n].tolist()))
    return eps


# ---- 1. distribution -----------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("alpha", [0.3, 1.0])
def test_eta_is_dirichlet(alpha):
    from scipy import stats

    E = 16384
    for k, cols in FULL.items():
        (eta,) = draw_eta(E, alpha, seed=2024, pos=full_columns(cols))
        legal = [c for c in range(7) if c not in cols]
        assert np.all(np.isfinite(eta))
        assert np.all(eta[:, list(cols)] == 0)
        assert np.abs(eta.sum(1, dtype=np.float64) - 1).max() < 1e-6
        if k == 1:
            assert np.all(eta[:, legal[0]] == 1)
            continue
        for c in legal:  # marginal of Dirichlet(alpha x k) = Beta(alpha, (k - 1) alpha)
            p = stats.kstest(eta[:, c].astype(np.float64), "beta", args=(alpha, (k - 1) * alpha)).pvalue
            assert p > 1e-4, (k, c, p)


def test_small_alpha_does_not_underflow():
    (eta,) = draw_eta(16384, 0.03, seed=5)
    assert np.all(np.isfinite(eta)) and np.all(eta >= 0)
    assert np.abs(eta.sum(1, dtype=np.float64) - 1).max() < 1e-6
    assert (eta.max(1) > 0.5).mean() > 0.9  # at alpha = 0.03 nearly all the mass goes to one column


def test_no_correlation_between_slots_or_draws():
    a, b = draw_eta(16384, 1.0, seed=9, draws=2)
    r_slots = np.corrcoef(a[:-1].ravel(), a[1:].ravel())[0, 1]
    r_draws = np.corrcoef(a.ravel(), b.ravel())[0, 1]
    assert abs(r_slots) < 0.02 and abs(r_draws) < 0.02, (r_slots, r_draws)


# ---- 2. determinism and shards -------------------------------------------------------------------------------------------------
def test_eta_is_a_function_of_seed_slot_and_draw():
    E = 4096
    a = draw_eta(E, 0.5, seed=77, draws=2)
    b = draw_eta(E, 0.5, seed=77, draws=2, lanes=32)
    c = draw_eta(E, 0.5, seed=78, draws=1)
    assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1])
    assert not np.array_equal(a[0], a[1])
    assert (a[0] != c[0]).all(axis=1).mean() > 0.99
    lo, hi = 1000, 3000
    part = draw_eta(hi - lo, 0.5, seed=77, slot_offset=lo, draws=2)
    assert np.array_equal(part[0], a[0][lo:hi]) and np.array_equal(part[1], a[1][lo:hi])


def _play_sharded(lo, hi, u, S, steps):
    eng = Engine(num_games=hi - lo, num_simulations=S)
    eng.reset_games()
    eng.set_root_noise(0.5, 0.25, 31, slot_offset=lo)
    eng.set_greedy_from(8)
    out = {}
    for s in range(steps):
        eng.run_simulations(1, 2)
        eng.apply_root_noise()
        eng.run_move_step(S - 1, 2, torch.from_numpy(np.ascontiguousarray(u[s, lo:hi])).cuda())
        if s % 8 == 7 or s == steps - 1:
            b = eng.drain_episodes()
            for e in range(len(b)):
                o, n = int(b.ep_offset[e]), int(b.ep_len[e])
                out[(int(b.ep_step[e]), int(b.ep_slot[e]) + lo)] = (b.ep_outcome[e].tolist(), b.s_bb0[o:o + n].tolist(),
                                                                   b.s_bb1[o:o + n].tolist(), b.s_counts[o:o + n].tolist())
    eng.close()
    return out


def test_sharded_selfplay_with_noise_equals_unsharded():
    from alphazero_implementation_b200.distributed import shard_range

    E, S, steps = 1000, 64, 45
    u = np.random.RandomState(11).random_sample((steps, E))
    full = _play_sharded(0, E, u, S, steps)
    assert full == _play_sharded(0, E, u, S, steps)  # the same seed plays the same games
    merged = {}
    for r in range(2):
        merged.update(_play_sharded(*shard_range(E, r, 2), u, S, steps))
    assert len(full) > E // 2 and full.keys() == merged.keys()
    for k in full:
        assert full[k] == merged[k], k


# ---- 3. exact mixing -----------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("fraction", [0.25, 0.6])
def test_mixing_is_the_fp32_formula(oracle, fraction):
    E = 4096
    bb0, bb1, pl = random_positions(oracle, E, seed=3)
    eng = Engine(num_games=E, num_simulations=8)
    eng.set_root_noise(0.3, fraction, 5)
    eng.set_roots(bb0, bb1, pl)
    eng.run_simulations(1, 2)
    before = eng.root_stats()["child_P"].cpu().numpy()
    eng.apply_root_noise()
    after = eng.root_stats()["child_P"].cpu().numpy()
    eta = eng.root_noise_values().cpu().numpy()
    f = np.float32(fraction)
    want = (np.float32(1) - f) * before + f * eta
    want[before == 0] = 0
    assert np.array_equal(after.view(np.uint32), want.view(np.uint32))
    assert (after != before).any()
    eng.run_simulations(7, 2)  # the rest of the search reads the mixed priors
    assert np.array_equal(eng.root_stats()["child_P"].cpu().numpy().view(np.uint32), want.view(np.uint32))


def test_apply_is_valid_once_after_one_simulation():
    eng = Engine(num_games=64, num_simulations=8)
    with pytest.raises(RuntimeError):
        eng.apply_root_noise()  # not configured
    eng.set_root_noise(1.0, 0.25, 0)
    eng.reset_games()
    with pytest.raises(RuntimeError):
        eng.apply_root_noise()  # no simulation yet
    eng.run_simulations(1, 1)
    eng.apply_root_noise()
    with pytest.raises(RuntimeError):
        eng.apply_root_noise()  # twice
    eng.run_simulations(1, 1)
    with pytest.raises(RuntimeError):
        eng.apply_root_noise()
    for bad in (dict(alpha=0.0), dict(alpha=float("nan")), dict(alpha=1.0, fraction=1.5), dict(alpha=1.0, slot_offset=-1)):
        with pytest.raises(RuntimeError):
            eng.set_root_noise(**bad)
    eng.close()


# ---- 4. fraction 0 is the identity, 5. against the oracle (built-in evaluators) --------------------------------------------------
def _builtin_selfplay(noise, E=2048, S=100, steps=30, lanes=0):
    search = az.AlphaZeroSearch(model=az.HashEvaluator(), num_simulations=S, lanes_per_tree=lanes, root_noise=noise)
    eng = search.engine_for(E, exact=True)
    eng.reset_games()
    u = torch.from_numpy(np.random.RandomState(4).random_sample((steps, E))).cuda()
    parts = []
    for s in range(steps):
        search.simulate_and_move(eng, u[s])  # built-in evaluator: the fused move step
        if s % 8 == 7 or s == steps - 1:
            parts.append(eng.drain_episodes())
    st = eng.stats()
    roots = np.zeros(E, np.uint64)
    eng.set_roots(roots, roots, np.zeros(E, np.uint8))
    search.simulate(eng)
    rs = {k: v.cpu().numpy() for k, v in eng.root_stats().items()}
    search.close()
    return flatten(parts), st, rs


def test_fraction_zero_is_noise_off_builtin():
    off = _builtin_selfplay(None)
    on = _builtin_selfplay(az.RootNoise(alpha=0.3, fraction=0.0, seed=1))
    assert len(off[0]) > 1000 and off[0] == on[0] and off[1] == on[1]
    for k in off[2]:
        assert np.array_equal(off[2][k], on[2][k]), k
    noisy = _builtin_selfplay(az.RootNoise(alpha=0.3, fraction=0.25, seed=1))
    assert noisy[0] != off[0]


@pytest.mark.parametrize("kind,lanes,fused", [(1, 8, False), (2, 8, True), (2, 32, False), (1, 32, True)])
def test_selfplay_with_noise_and_cutoff_vs_oracle(oracle, kind, lanes, fused):
    E, S, eps, greedy = 4096, 200, 0.25, 10
    u2 = np.random.RandomState(E + S + kind).random_sample((60, E))
    eng = Engine(num_games=E, num_simulations=S, lanes_per_tree=lanes)
    eng.reset_games()
    eng.set_root_noise(1.0, eps, 1234 + kind)
    eng.set_greedy_from(greedy)
    etas, parts, count = [], [], 0
    for step in range(u2.shape[0]):
        eng.run_simulations(1, kind)
        eng.apply_root_noise()
        etas.append(eng.root_noise_values().cpu().numpy())
        u = torch.from_numpy(u2[step]).cuda()
        if fused:  # k_run_sims, then k_sample_moves<greedy>
            eng.run_move_step(S - 1, kind, u)
        else:
            eng.run_simulations(S - 1, kind)
            eng.sample_moves(u)
        ne, _ = eng.episode_counts()
        if ne:
            parts.append(eng.drain_episodes())
            count += ne
            if count >= E:
                break
    steps = step + 1
    stats = eng.stats()
    eng.close()
    ref = noise_oracle.selfplay_noise(E, S, u2[:steps], eps, np.stack(etas), greedy_from=greedy, eval_kind=kind)
    got = flatten(parts)[:E]
    assert len(got) == E == len(ref.ep_slot) and steps == ref.n_steps
    assert [g["slot"] for g in got] == ref.ep_slot.tolist() and [g["step"] for g in got] == ref.ep_step.tolist()
    assert [g["outcome"] for g in got] == ref.ep_outcome.tolist()
    assert [len(g["bb0"]) for g in got] == ref.ep_len.tolist()
    assert (np.concatenate([np.array(g["bb0"], np.uint64) for g in got]) == ref.s_bb0).all()
    assert (np.concatenate([np.array(g["bb1"], np.uint64) for g in got]) == ref.s_bb1).all()
    assert (np.concatenate([np.array(g["player"], np.uint8) for g in got]) == ref.s_player).all()
    assert (np.concatenate([np.array(g["counts"], np.int32) for g in got]) == ref.s_counts).all()
    assert stats["simulations"] == ref.n_sims and stats["evaluations"] == ref.n_evals


# ---- 4 / 6. network in the loop ------------------------------------------------------------------------------------------------
NE, NS, NSTEPS = 2048, 800, 12


def _resnet(seed=0):
    torch.manual_seed(seed)
    m = az.ResNet(num_res_blocks=4, num_channels=64)
    with torch.no_grad():
        for mod in m.modules():
            if isinstance(mod, torch.nn.BatchNorm2d):
                mod.running_mean.uniform_(-0.5, 0.5)
                mod.running_var.uniform_(0.5, 2.0)
    return m.eval()


def _net_selfplay(noise, cache=True, graph=True, greedy=None):
    search = az.AlphaZeroSearch(model=_resnet(), num_simulations=NS, inference_dtype=torch.bfloat16, eval_cache=cache,
                                use_cuda_graph=graph, root_noise=noise)
    eng = search.engine_for(NE, exact=True)
    eng.reset_games()
    eng.set_greedy_from(greedy)
    u = torch.from_numpy(np.random.RandomState(5).random_sample((NSTEPS, NE))).cuda()
    roots, episodes = [], []
    for step in range(NSTEPS):
        search.simulate(eng)
        roots.append({k: v.cpu().numpy() for k, v in eng.root_stats().items()})
        eng.sample_moves(u[step])
        b = eng.drain_episodes()
        episodes.append({f: np.asarray(getattr(b, f)).copy() for f in EP_FIELDS})
    out = dict(roots=roots, episodes=episodes, stats=eng.stats(), cache=eng.eval_cache_stats(), kernel=search.evaluator_name,
               log2=eng.eval_cache_log2)
    search.close()
    return out


def _same(a, b):
    if a["stats"] != b["stats"]:
        return False
    for ra, rb in zip(a["roots"], b["roots"]):
        if any(not np.array_equal(ra[k], rb[k]) for k in ra):
            return False
    for ea, eb in zip(a["episodes"], b["episodes"]):
        if any(not np.array_equal(ea[k], eb[k]) for k in ea):
            return False
    return True


@pytest.fixture(scope="module")
def net_plain():
    return _net_selfplay(None)


def test_fraction_zero_is_noise_off_network(net_plain):
    on = _net_selfplay(az.RootNoise(alpha=1.0, fraction=0.0, seed=3))
    assert net_plain["kernel"] == "k_resnet_wide" and net_plain["log2"] > 0
    assert _same(net_plain, on)


def test_network_noise_cache_and_graph_change_no_bit(net_plain):
    noise = az.RootNoise(alpha=1.0, fraction=0.25, seed=3)
    ref = _net_selfplay(noise, cache=True, graph=True, greedy=6)
    assert ref["log2"] > 0 and ref["cache"]["hits"] > 0
    assert not _same(ref, net_plain)  # the noise changes the games
    for kw in (dict(cache=False, graph=True), dict(cache=True, graph=False)):
        other = _net_selfplay(noise, greedy=6, **kw)
        assert _same(ref, other), kw
        if not kw["cache"]:
            assert other["log2"] == 0 and other["cache"]["hits"] == 0


class KernelEvaluator:
    """`predict` for the oracle: the production kernels applied to the given positions (a helper engine whose roots are the
    positions: the first selection returns the root; expansion stores the legal-only softmax priors)."""

    def __init__(self, net, cap=64):
        self.net, self.cap = net, cap
        self.eng = Engine(num_games=cap, num_simulations=1)

    def __call__(self, bb0, bb1, player, legal):
        n = len(bb0)
        assert n <= self.cap
        e = self.eng
        e.set_roots(bb0, bb1, player)
        e.select_leaves()
        logits, values = self.net.forward_leaves(e)
        e.expand_backup(logits, values, POLICY_LOGITS)
        return e.root_stats()["child_P"][:n].cpu().numpy(), values[:n].cpu().numpy()


def test_network_trees_with_noise_vs_oracle(oracle):
    eps = 0.25
    search = az.AlphaZeroSearch(model=_resnet(), num_simulations=NS, inference_dtype=torch.bfloat16,
                                root_noise=az.RootNoise(alpha=0.5, fraction=eps, seed=8))
    bb0, bb1, pl = random_positions(oracle, NE, seed=12)
    eng = search.engine_for(NE)
    eng.set_roots(bb0, bb1, pl)
    search.simulate(eng)
    got = {k: v.cpu().numpy() for k, v in eng.root_stats().items()}
    eta = eng.root_noise_values().cpu().numpy()
    assert (got["root_N"] == NS).all() and (np.abs(eta.sum(1) - 1) < 1e-6).all()
    idx = np.random.RandomState(5).choice(NE, 16, replace=False)
    ref = noise_oracle.search_noise(bb0[idx], bb1[idx], pl[idx], NS, eps, eta[idx], py_eval=KernelEvaluator(search._net))
    for k in ("child_N", "root_N", "child_W", "root_W", "child_P"):
        assert np.array_equal(got[k][idx], ref[k]), k
    search.close()


# ---- 7. launch count, 8. trainer -----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("spec", ["builtin", "builtin_greedy", "basic"])
def test_launches_per_move_step_with_noise(spec):
    S, E = 24, 256
    model = az.BasicNN() if spec == "basic" else az.UniformEvaluator()
    search = az.AlphaZeroSearch(model=model, num_simulations=S, use_cuda_graph=False, root_noise=az.RootNoise(seed=1))
    eng = search.engine_for(E, exact=True)
    eng.reset_games()
    eng.set_greedy_from(4 if spec == "builtin_greedy" else None)
    u = torch.from_numpy(np.random.RandomState(0).random_sample((3, E))).cuda()
    search.simulate_and_move(eng, u[0])  # first step: one-off allocations (the packed batch of the gather)
    for s in (1, 2):
        n0 = eng.launch_count
        search.simulate_and_move(eng, u[s])
        assert eng.launch_count - n0 == search.launches_per_move_step(), spec
    expect = {"builtin": 3, "builtin_greedy": 4, "basic": 2 * S + 4}[spec]
    assert search.launches_per_move_step() == expect
    search.close()


def test_trainer_with_noise_and_cutoff():
    from alphazero_implementation_b200.trainer import Trainer

    torch.manual_seed(0)
    np.random.seed(0)
    tr = Trainer(az.BasicNN())
    hist = tr.train(num_iterations=2, episodes_per_iter=32, simulations_per_episode=32, epochs_per_iter=1,
                    initial_state=az.Config(6, 7, 4).sample_initial_state(), buffer_size=64,
                    root_noise=az.RootNoise(alpha=1.0, fraction=0.25, seed=4), sampling_moves=6)
    assert len(hist) == 2 and hist[0]["episodes"] == 32 and hist[1]["episodes"] == 64
    assert hist[0]["samples"] >= 32 * 7 and hist[1]["loss"] is not None
