"""GPU: mirror-symmetric self-play (az_set_symmetric_eval, az_mirror_states, AlphaZeroSearch(symmetric=True), mirror augmentation).

With the mode on the search evaluates f_sym(x) = f(canon(x)) with the policy columns reversed when canon(x) is the mirror of x.
The trees it builds are bit-exact with the oracle's when the oracle's `predict` callback computes f_sym on the host (canonical
form, the same kernels with the mode off, reversed priors); the evaluation cache stays exact; a position and its mirror share one
evaluator row."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

import alphazero_implementation_b200 as az  # noqa: E402
from alphazero_implementation_b200.engine import LEAF_EVAL, LEAF_IDLE, LEAF_SERVED, LEAF_TERMINAL, POLICY_LOGITS, Engine  # noqa: E402
from alphazero_implementation_b200.game import canonical_bitboards, mirror_bitboards  # noqa: E402
import noise_oracle  # noqa: E402
from test_gpu_config3 import KernelEvaluator, random_positions  # noqa: E402

EP_FIELDS = ("ep_slot", "ep_step", "ep_len", "ep_outcome", "s_bb0", "s_bb1", "s_player", "s_counts")
BOARD = np.uint64(0xFDFBF7EFDFBF)


def _resnet(seed=0):
    torch.manual_seed(seed)
    m = az.ResNet(num_res_blocks=4, num_channels=64)
    with torch.no_grad():  # random BatchNorm statistics: priors and values differ between a position and its mirror
        for mod in m.modules():
            if isinstance(mod, torch.nn.BatchNorm2d):
                mod.running_mean.uniform_(-0.5, 0.5)
                mod.running_var.uniform_(0.5, 2.0)
    return m.eval()


def _reverse7(m):
    m = np.asarray(m, np.uint8)
    return sum(((m >> c) & 1) << (6 - c) for c in range(7)).astype(np.uint8)


class SymmetricEvaluator:
    """f_sym on the host for the oracle: canonicalise, evaluate the canonical positions with `inner` (kernels of an engine whose
    mode is off), reverse the prior columns of the mirrored rows."""

    def __init__(self, inner):
        self.inner, self.calls = inner, 0

    def __call__(self, bb0, bb1, player, legal):
        self.calls += 1
        c0, c1, mir = canonical_bitboards(bb0, bb1)
        pri, val = self.inner(c0, c1, player, np.where(mir, _reverse7(legal), legal))
        pri = np.where(mir[:, None], pri[:, ::-1], pri)
        return np.ascontiguousarray(pri, np.float32), np.ascontiguousarray(val, np.float32)


def _random_boards(rng, n):
    """n random (not necessarily reachable) boards: disjoint stone sets inside the 42 cells"""
    occ = rng.randint(0, 2**63, size=n, dtype=np.int64).view(np.uint64) & BOARD
    side = rng.randint(0, 2**63, size=n, dtype=np.int64).view(np.uint64)
    return occ & side, occ & ~side


# ---- 1. az_mirror_states ------------------------------------------------------------------------------------------------------
def test_mirror_states_kernel():
    eng = Engine(num_games=1, num_simulations=1)
    rng = np.random.RandomState(0)
    n = (1 << 20) + 3  # the 4-position vector path and the scalar tail
    b0, b1 = _random_boards(rng, n)
    m0, m1 = mirror_bitboards(b0, b1)
    d0, d1 = eng._dev(b0, torch.int64), eng._dev(b1, torch.int64)
    o0, o1 = eng.mirror_states(d0, d1)
    assert np.array_equal(o0.cpu().numpy().view(np.uint64), m0) and np.array_equal(o1.cpu().numpy().view(np.uint64), m1)
    flags = (rng.random_sample(n) < 0.5).astype(np.uint8) * rng.randint(1, 256, size=n).astype(np.uint8)
    want0, want1 = np.where(flags != 0, m0, b0), np.where(flags != 0, m1, b1)
    o0, o1 = eng.mirror_states(d0, d1, torch.from_numpy(flags).cuda())
    assert np.array_equal(o0.cpu().numpy().view(np.uint64), want0) and np.array_equal(o1.cpu().numpy().view(np.uint64), want1)
    # in place, on a view whose start is 8 bytes off the 16-byte alignment (scalar kernel only)
    f = torch.from_numpy(flags).cuda()
    v0, v1, fv = d0[1:], d1[1:], f[1:]
    eng.mirror_states(v0, v1, fv, out=(v0, v1))
    assert np.array_equal(d0[1:].cpu().numpy().view(np.uint64), want0[1:]) and np.array_equal(d1[1:].cpu().numpy().view(np.uint64), want1[1:])
    eng.mirror_states(d0, d1, f, out=(d0, d1))  # in place, vector path: row 0 flips once, rows >= 1 flip back
    assert np.array_equal(d0[1:].cpu().numpy().view(np.uint64), b0[1:]) and int(d0[0]) == int(want0[0].view(np.int64))


def test_mirror_states_keep_the_rules(oracle):
    eng = Engine(num_games=1, num_simulations=1)
    bb0, bb1, pl, _ = random_positions(oracle, 16384, seed=4, max_plies=40)
    o0, o1 = eng.mirror_states(bb0, bb1)
    a, b = eng.state_info(bb0, bb1), eng.state_info(o0, o1)
    assert np.array_equal(b["legal"].cpu().numpy(), _reverse7(a["legal"].cpu().numpy()))
    assert torch.equal(a["ended"], b["ended"]) and torch.equal(a["reward"], b["reward"])


# ---- 2. trees bit-exact with the oracle fed f_sym -------------------------------------------------------------------------------
@pytest.mark.parametrize("spec", ["resnet4x64", "basic"])
def test_symmetric_trees_bit_exact_with_oracle(oracle, spec):
    E, S, n_check = 16384, 800, 24
    model = _resnet() if spec == "resnet4x64" else (torch.manual_seed(0), az.BasicNN())[1]
    search = az.AlphaZeroSearch(model=model, num_simulations=S, inference_dtype=torch.bfloat16, symmetric=True)
    bb0, bb1, pl, _ = random_positions(oracle, E, seed=11)
    eng = search.engine_for(E)
    eng.set_roots(bb0, bb1, pl)
    search.simulate(eng)  # graph-replayed (evaluator, k_expand_select<SYM>) with compaction; the cache where the net allows it
    assert eng.symmetric_eval and (spec != "resnet4x64" or eng.eval_cache_log2 > 0)
    got = {k: v.cpu().numpy() for k, v in eng.root_stats().items()}
    assert (got["root_N"] == S).all()
    idx = np.random.RandomState(5).choice(E, n_check, replace=False)
    ev = SymmetricEvaluator(KernelEvaluator(search._net))
    ref = oracle.search(bb0[idx], bb1[idx], pl[idx], S, py_eval=ev)
    assert ev.calls == S
    for k in ("child_N", "root_N", "child_W", "root_W", "child_P"):
        assert np.array_equal(got[k][idx], ref[k]), k
    search.close()


# ---- 3. leaf arrays ----------------------------------------------------------------------------------------------------------
def test_leaf_arrays_hold_canonical_leaves(oracle):
    """With uniform priors (zero logits) a tree does not depend on the mode: the same leaves are reached with the mode on and
    off, and the mode-on engine reports them in canonical form."""
    E, K = 4096, 24
    bb0, bb1, pl, _ = random_positions(oracle, E, seed=7, max_plies=36)
    bb0[:2], bb1[:2], pl[:2] = [0xF, 0xF << 42], [0x7 << 7, 0x7 << 35], [1, 1]  # a won position and its mirror: IDLE slots
    engs = [Engine(num_games=E, num_simulations=K) for _ in range(2)]
    engs[1].set_symmetric_eval(True)
    zero_p, zero_v = torch.zeros((E, 7), device="cuda"), torch.zeros((E, 2), device="cuda")
    seen = {LEAF_EVAL: 0, LEAF_TERMINAL: 0, LEAF_IDLE: 0}
    for e in engs:
        e.set_roots(bb0, bb1, pl)
    for _ in range(K):
        off, on = [], []
        for e, out in zip(engs, (off, on)):
            e.select_leaves()
            out.append({k: v.cpu().numpy() for k, v in e.leaf_info().items()})
        assert engs[0].leaf_mirror() is None
        mir = engs[1].leaf_mirror().cpu().numpy()
        a, b = off[0], on[0]
        st = a["status"]
        assert np.array_equal(st, b["status"]) and np.array_equal(a["player"], b["player"])
        live = (st == LEAF_EVAL) | (st == LEAF_SERVED)
        c0, c1, cm = canonical_bitboards(a["bb0"].view(np.uint64), a["bb1"].view(np.uint64))
        assert np.array_equal(b["bb0"].view(np.uint64)[live], c0[live]) and np.array_equal(b["bb1"].view(np.uint64)[live], c1[live])
        assert np.array_equal(mir[live], cm[live].astype(np.uint8))
        assert np.array_equal(b["legal"][live], np.where(cm, _reverse7(a["legal"]), a["legal"])[live])
        rest = ~live & (st == LEAF_TERMINAL)
        assert np.array_equal(b["bb0"][rest], a["bb0"][rest]) and np.array_equal(b["bb1"][rest], a["bb1"][rest])
        assert not mir[~live].any()
        for s in seen:
            seen[s] += int((st == s).sum())
        for e in engs:
            e.expand_backup(zero_p, zero_v, POLICY_LOGITS)
    assert all(v > 0 for v in seen.values()), seen
    so, sn = engs[0].root_stats(), engs[1].root_stats()
    for k in ("child_N", "child_W", "child_P", "root_W", "root_N"):
        assert torch.equal(so[k], sn[k]), k


# ---- 4. mirror consistency ---------------------------------------------------------------------------------------------------
def _roots_and_mirrors(oracle, n, seed):
    bb0, bb1, pl, _ = random_positions(oracle, 4 * n, seed=seed)
    c0, c1, _ = canonical_bitboards(bb0, bb1)
    m0, m1 = mirror_bitboards(bb0, bb1)
    keep = ~((m0 == bb0) & (m1 == bb1))  # no palindromes
    _, first = np.unique(np.stack([c0, c1], 1)[keep], axis=0, return_index=True)  # distinct canonical forms
    sel = np.nonzero(keep)[0][np.sort(first)][:n]
    assert len(sel) == n
    b0, b1, p = bb0[sel], bb1[sel], pl[sel]
    n0, n1 = mirror_bitboards(b0, b1)
    return np.concatenate([b0, n0]), np.concatenate([b1, n1]), np.concatenate([p, p])


@pytest.mark.parametrize("symmetric", [True, False])
def test_root_priors_of_a_position_and_its_mirror(oracle, symmetric):
    n = 1024
    bb0, bb1, pl = _roots_and_mirrors(oracle, n, seed=8)
    search = az.AlphaZeroSearch(model=_resnet(), num_simulations=8, inference_dtype=torch.bfloat16, symmetric=symmetric)
    eng = search.engine_for(2 * n)
    eng.set_roots(bb0, bb1, pl)
    search.simulate(eng)
    P = eng.root_stats()["child_P"].cpu().numpy()
    same = np.array([np.array_equal(P[i], P[n + i][::-1]) for i in range(n)])
    if symmetric:
        assert same.all()
    else:
        assert not same.all()  # the test has power: the random net is not symmetric by itself
    search.close()


# ---- 5. the cache stays exact ------------------------------------------------------------------------------------------------
def _selfplay(E, S, steps, cache=True, graph=True, noise=None, greedy=None):
    search = az.AlphaZeroSearch(model=_resnet(), num_simulations=S, inference_dtype=torch.bfloat16, eval_cache=cache,
                                use_cuda_graph=graph, symmetric=True, root_noise=noise)
    eng = search.engine_for(E, exact=True)
    eng.reset_games()
    eng.set_greedy_from(greedy)
    u = torch.from_numpy(np.random.RandomState(5).random_sample((steps, E))).cuda()
    roots, episodes, etas = [], [], []
    for step in range(steps):
        search.simulate(eng)
        roots.append({k: v.cpu().numpy() for k, v in eng.root_stats().items()})
        if noise is not None:
            etas.append(eng.root_noise_values().cpu().numpy())
        eng.sample_moves(u[step])
        b = eng.drain_episodes()
        episodes.append({f: np.asarray(getattr(b, f)).copy() for f in EP_FIELDS})
    out = dict(roots=roots, episodes=episodes, etas=etas, stats=eng.stats(), cache=eng.eval_cache_stats(), log2=eng.eval_cache_log2,
               kernel=search.evaluator_name)
    search.close()
    return out


def _assert_same(a, b):
    assert a["stats"] == b["stats"]
    for ra, rb in zip(a["roots"], b["roots"]):
        for k in ra:
            assert np.array_equal(ra[k], rb[k]), k
    for ea, eb in zip(a["episodes"], b["episodes"]):
        for k in ea:
            assert np.array_equal(ea[k], eb[k]), k
    for x, y in zip(a["etas"], b["etas"]):
        assert np.array_equal(x, y)


def test_cache_exact_under_symmetry():
    E, S, steps = 2048, 800, 12
    on = _selfplay(E, S, steps)
    assert on["kernel"] == "k_resnet_wide" and on["log2"] > 0 and on["cache"]["hits"] > 0
    assert on["cache"]["rows"] + on["cache"]["hits"] + on["cache"]["followers"] == on["stats"]["evaluations"]
    off = _selfplay(E, S, steps, cache=False)
    assert off["log2"] == 0
    _assert_same(on, off)
    _assert_same(on, _selfplay(E, S, steps, cache=False, graph=False))
    tiny = _selfplay(E, S, steps, cache=10)
    assert tiny["log2"] == 10 and tiny["cache"]["evictions"] > 0
    _assert_same(on, tiny)


# ---- 6. twins share rows -----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("symmetric", [True, False])
def test_twins_share_one_row(oracle, symmetric):
    n = 4096
    bb0, bb1, pl = _roots_and_mirrors(oracle, n, seed=9)
    search = az.AlphaZeroSearch(model=_resnet(), num_simulations=1, inference_dtype=torch.bfloat16, eval_cache=22,
                                symmetric=symmetric, use_cuda_graph=False)
    eng = search.engine_for(2 * n, exact=True)
    eng.set_roots(bb0, bb1, pl)
    search.simulate(eng)  # one selection: every leaf is its root
    c = eng.eval_cache_stats()
    assert eng.stats()["evaluations"] == 2 * n and c["hits"] == 0
    if symmetric:
        print(f"twins: rows {c['rows']} followers {c['followers']} failed claims {c['failed_claims']}")
        assert c["rows"] == n + c["failed_claims"] and c["followers"] == n - c["failed_claims"]
        assert c["failed_claims"] <= n // 20
    else:
        assert c["rows"] == 2 * n and c["followers"] == 0
    search.close()


# ---- 7. exploration together with symmetry -----------------------------------------------------------------------------------
def test_noise_and_greedy_cutoff_with_symmetry(oracle):
    eps, NE, NS = 0.25, 2048, 200
    noise = az.RootNoise(alpha=0.5, fraction=eps, seed=8)
    search = az.AlphaZeroSearch(model=_resnet(), num_simulations=NS, inference_dtype=torch.bfloat16, root_noise=noise, symmetric=True)
    bb0, bb1, pl, _ = random_positions(oracle, NE, seed=12)
    eng = search.engine_for(NE)
    eng.set_roots(bb0, bb1, pl)
    search.simulate(eng)
    got = {k: v.cpu().numpy() for k, v in eng.root_stats().items()}
    eta = eng.root_noise_values().cpu().numpy()
    idx = np.random.RandomState(5).choice(NE, 16, replace=False)
    ref = noise_oracle.search_noise(bb0[idx], bb1[idx], pl[idx], NS, eps, eta[idx], py_eval=SymmetricEvaluator(KernelEvaluator(search._net)))
    for k in ("child_N", "root_N", "child_W", "root_W", "child_P"):
        assert np.array_equal(got[k][idx], ref[k]), k
    search.close()
    # self-play with noise, the greedy cutoff and the mode on: cache and graph change no bit
    a = _selfplay(512, 200, 10, noise=noise, greedy=4)
    _assert_same(a, _selfplay(512, 200, 10, cache=False, graph=False, noise=noise, greedy=4))


# ---- 8. predict path ---------------------------------------------------------------------------------------------------------
class RecordingHash:
    """a user `predict` evaluator (HashEvaluator's pseudo-random priors: not symmetric) that records the positions it is given"""

    def __init__(self):
        self.inner, self.seen = az.HashEvaluator(), []

    def get_inference_clone(self):
        return self

    def predict(self, states):
        self.seen.append(np.array([[s.bb0, s.bb1] for s in states], np.uint64))
        return self.inner.predict(states)


def _hash_arrays(bb0, bb1, player, legal):
    from alphazero_implementation_b200.game import states_from_arrays

    states = states_from_arrays(bb0, bb1, player, legal=legal, ended=np.zeros(len(bb0), bool), reward=np.zeros((len(bb0), 2), np.int8))
    pols, vals = az.HashEvaluator().predict(states)
    pri = np.zeros((len(bb0), 7), np.float32)
    for i, p in enumerate(pols):
        for act, v in p.items():
            pri[i, act.column] = v
    return pri, np.array(vals, np.float32)


def test_predict_path_sees_canonical_states(oracle):
    E, S = 64, 50
    model = RecordingHash()
    search = az.AlphaZeroSearch(model=model, num_simulations=S, symmetric=True)
    bb0, bb1, pl, _ = random_positions(oracle, E, seed=13)
    eng = search.engine_for(E)
    eng.set_roots(bb0, bb1, pl)
    search.simulate(eng)
    seen = np.concatenate(model.seen)
    _, _, mir = canonical_bitboards(seen[:, 0], seen[:, 1])
    assert len(seen) > E and not mir.any()
    got = {k: v.cpu().numpy() for k, v in eng.root_stats().items()}
    ref = oracle.search(bb0, bb1, pl, S, py_eval=SymmetricEvaluator(_hash_arrays))
    for k in ("child_N", "root_N", "child_W", "root_W", "child_P"):
        assert np.array_equal(got[k], ref[k]), k
    search.close()


# ---- 9. guards ---------------------------------------------------------------------------------------------------------------
def test_guards():
    with pytest.raises(ValueError):
        az.AlphaZeroSearch(model=az.UniformEvaluator(), num_simulations=8, symmetric=True)
    eng = Engine(num_games=64, num_simulations=16)
    eng.reset_games()
    eng.set_symmetric_eval(True)
    u = torch.zeros(64, dtype=torch.float64, device="cuda")
    with pytest.raises(RuntimeError, match=r"\(-4\)"):
        eng.run_simulations(4, 1)
    with pytest.raises(RuntimeError, match=r"\(-4\)"):
        eng.run_move_step(4, 1, u)
    eng.select_leaves()
    with pytest.raises(RuntimeError, match=r"\(-4\)"):
        eng.set_symmetric_eval(False)
    eng.expand_backup(torch.zeros((64, 7), device="cuda"), torch.zeros((64, 2), device="cuda"))
    eng.set_symmetric_eval(False)
    eng.run_simulations(4, 1)


def test_launches_per_move_step_unchanged():
    S, E = 24, 256
    counts = []
    for sym in (False, True):
        torch.manual_seed(0)
        search = az.AlphaZeroSearch(model=az.BasicNN(), num_simulations=S, use_cuda_graph=False, symmetric=sym)
        eng = search.engine_for(E, exact=True)
        eng.reset_games()
        u = torch.from_numpy(np.random.RandomState(0).random_sample((3, E))).cuda()
        search.simulate_and_move(eng, u[0])
        for s in (1, 2):
            n0 = eng.launch_count
            search.simulate_and_move(eng, u[s])
            assert eng.launch_count - n0 == search.launches_per_move_step()
        counts.append(search.launches_per_move_step())
        search.close()
    assert counts[0] == counts[1]


# ---- 10. training ------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def replay():
    from alphazero_implementation_b200.replay import ReplayBuffer

    gen = az.EpisodeGenerator(model=az.HashEvaluator(), num_simulations=24, num_episodes=64,
                              game_initial_state=az.Config().sample_initial_state())
    np.random.seed(3)
    rb = ReplayBuffer(buffer_size=64, num_simulations=24)
    for batch in gen.generate_batches(quota=64):
        rb.extend(batch)
    return rb


def _expected(rb, j, f, layout):
    """minibatch of samples j (replay-set indices), rows with f set in their mirror image"""
    bb0, bb1, pl, policy, value = rb.tensors()
    j, f = j.cuda(), f.cuda().bool()
    m0, m1 = mirror_bitboards(bb0[j].cpu().numpy().view(np.uint64), bb1[j].cpu().numpy().view(np.uint64))
    b0 = torch.where(f, torch.from_numpy(m0.view(np.int64)).cuda(), bb0[j])
    b1 = torch.where(f, torch.from_numpy(m1.view(np.int64)).cuda(), bb1[j])
    x = az.game.rules_engine().encode_states(b0, b1, pl[j], layout)
    pol = torch.where(f[:, None], policy[j].flip(1), policy[j])
    return x, pol, value[j], f


def test_replay_batches_mirror(replay):
    from alphazero_implementation_b200.engine import LAYOUT_GRID_F32

    n = replay.num_samples
    g = torch.Generator().manual_seed(7)
    perm = torch.randperm(n, generator=g)
    flags = torch.randint(0, 2, (n,), generator=g, dtype=torch.uint8)
    x, pol, val = next(iter(replay.batches(LAYOUT_GRID_F32, batch_size=64, generator=torch.Generator().manual_seed(7), mirror=True)))
    ex, epol, evl, f = _expected(replay, perm[:64], flags[:64], LAYOUT_GRID_F32)  # flags drawn per position of the shuffled set
    assert 0 < int(f.sum()) < 64
    assert torch.equal(x, ex) and torch.equal(pol, epol) and torch.equal(val, evl)
    x0, pol0, _ = next(iter(replay.batches(LAYOUT_GRID_F32, batch_size=64, generator=torch.Generator().manual_seed(7))))
    assert torch.equal(x0[~f], x[~f]) and not torch.equal(x0[f], x[f]) and torch.equal(pol0[~f], pol[~f])


def test_graphed_training_mirror_augment(replay):
    from alphazero_implementation_b200.trainer import _GraphedTraining

    dev = torch.device("cuda", torch.cuda.current_device())
    results = []
    for use_graph in (False, True):
        torch.manual_seed(11)
        model = az.BasicNN().cuda().train()
        opt = model.configure_optimizers()
        for group in opt.param_groups:
            group["capturable"] = True
        steps = _GraphedTraining(model, opt, batch_size=32, precision="32-true", device=dev, mirror_augment=True)
        first = []
        if not use_graph:  # the inputs of the first optimiser step: flagged rows mirrored, the others untouched
            orig = model.training_step

            def rec(batch, i):
                if not first:
                    first.append([t.detach().clone() for t in batch])
                return orig(batch, i)

            model.training_step = rec
        loss_sum, n = steps.run(replay, epochs=2, generator=torch.Generator().manual_seed(5), use_graph=use_graph)
        assert (steps.replays > 0) == use_graph
        if first:
            g = torch.Generator().manual_seed(5)
            perm = torch.randperm(replay.num_samples, generator=g)
            flags = torch.randint(0, 2, (replay.num_samples,), generator=g, dtype=torch.uint8)
            ex, epol, evl, f = _expected(replay, perm[:32], flags[perm[:32]], model.input_layout)  # flags drawn per sample
            assert 0 < int(f.sum()) < 32
            assert torch.equal(first[0][0], ex) and torch.equal(first[0][1], epol) and torch.equal(first[0][2], evl)
        results.append((float(loss_sum), [p.detach().clone() for p in model.parameters()]))
    (l0, w0), (l1, w1) = results
    assert l0 == pytest.approx(l1, rel=1e-5)
    for a, b in zip(w0, w1):
        assert torch.allclose(a, b, atol=1e-6, rtol=1e-5)


def test_trainer_symmetric_with_mirror_augment():
    from alphazero_implementation_b200.trainer import Trainer

    torch.manual_seed(0)
    np.random.seed(0)
    tr = Trainer(az.BasicNN())
    hist = tr.train(num_iterations=2, episodes_per_iter=32, simulations_per_episode=32, epochs_per_iter=1,
                    initial_state=az.Config(6, 7, 4).sample_initial_state(), buffer_size=64, symmetric=True, mirror_augment=True)
    assert len(hist) == 2 and hist[1]["episodes"] == 64
    assert all(h["loss"] is not None and np.isfinite(h["loss"]) for h in hist)
