"""GPU: subtree reuse (az_set_subtree_reuse, k_reroot, k_sample_moves<GREEDY, REUSE>, az_advance_roots).  A retained tree is the
reuse oracle's compacted tree field for field and the played child's subtree of the tree before the move; self-play with reuse is
bit-exact against tests/native/c4_reuse_oracle.c on the built-in evaluators (noise, greedy cutoff, 8 / 32 lanes, trees too large
for the shared-memory prefix); V = S is reuse off; with ResNet 4x64 in the loop the evaluation cache, the CUDA graph and symmetric
evaluation change no bit and sampled trees match the oracle fed the kernels' outputs."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

import alphazero_implementation_b200 as az  # noqa: E402
from alphazero_implementation_b200.engine import POLICY_LOGITS, TREE_ROOT_ENDED, Engine  # noqa: E402
import reuse_oracle  # noqa: E402

EP_FIELDS = ("ep_slot", "ep_step", "ep_len", "ep_outcome", "s_bb0", "s_bb1", "s_player", "s_counts")
TREE_FIELDS = ("W", "N", "P", "first_child")


def random_positions(oracle, n, seed, max_plies=20):
    """n non-terminal positions after 0..max_plies random legal moves."""
    rng = np.random.RandomState(seed)
    bb0, bb1, pl = np.zeros(n, np.uint64), np.zeros(n, np.uint64), np.zeros(n, np.uint8)
    target = rng.randint(0, max_plies + 1, size=n)
    legal = np.full(n, 0x7F, np.uint8)
    for ply in range(max_plies):
        go = np.nonzero(target > ply)[0]
        if not len(go):
            break
        cols = np.array([rng.choice([c for c in range(7) if (legal[i] >> c) & 1]) for i in go], np.uint8)
        nxt = oracle.env_step(bb0[go], bb1[go], pl[go], cols)
        ok = (nxt["status"] == 0) & (nxt["ended"] == 0)
        keep = go[ok]
        bb0[keep], bb1[keep], pl[keep], legal[keep] = nxt["bb0"][ok], nxt["bb1"][ok], nxt["player"][ok], nxt["legal"][ok]
        target[go[~ok]] = 0
    return bb0, bb1, pl


def legal_cols(b0, b1):
    occ = int(b0) | int(b1)
    return [c for c in range(7) if not (occ >> (7 * c + 5)) & 1]


def export(eng, slot, cap):
    t = eng.export_tree(slot)
    out = {k: np.zeros(cap, dt) for k, dt in (("W", np.float64), ("N", np.uint32), ("P", np.float32), ("first_child", np.uint32))}
    for k in TREE_FIELDS:
        out[k][:t["used"]] = t[k].view(out[k].dtype)
    return out, t["used"]


def node_map(node, path=()):
    """{column path: (N, W, P)} of a materialised `Node` tree"""
    out = {path: (node.visit_count, node.value_sum, np.float32(node.prior))}
    for a, ch in node.children.items():
        out.update(node_map(ch, path + (a.column,)))
    return out


def tree_map(t, i, b0, b1, pl, idx=0, path=()):
    out = {path: (int(t["N"][i][idx]), float(t["W"][i][idx]), np.float32(t["P"][i][idx]))}
    cb = int(t["first_child"][i][idx])
    if cb:
        occ = int(b0) | int(b1)
        for j, c in enumerate(legal_cols(b0, b1)):
            col = occ >> (7 * c) & 0x7F
            bit = ((col + 1) & ~col) << (7 * c)
            nb = (int(b0) | bit, int(b1), 1) if pl == 0 else (int(b0), int(b1) | bit, 0)
            out.update(tree_map(t, i, *nb, cb + j, path + (c,)))
    return out


# ---- 1. advance_roots ----------------------------------------------------------------------------------------------------------
def test_advance_roots_vs_oracle_and_materialized_tree(oracle):
    E, S, V = 4096, 200, 400
    bb0, bb1, pl = random_positions(oracle, E, seed=21)
    rng = np.random.RandomState(3)
    cols = np.array([rng.choice(legal_cols(bb0[i], bb1[i])) for i in range(E)], np.uint8)
    cols[rng.choice(E, 64, replace=False)] = 7  # illegal: the slot stays as it was
    for i in range(E):  # a few full columns, illegal too
        if len(legal_cols(bb0[i], bb1[i])) < 7 and i % 17 == 0:
            cols[i] = [c for c in range(7) if c not in legal_cols(bb0[i], bb1[i])][0]
    # slot 1: a move that wins - three stones of player 0 in column 0, player 0 to move
    bb0[1], bb1[1], pl[1], cols[1] = np.uint64(0b111), np.uint64(0b111 << 7), 0, 0
    eng = Engine(num_games=E, num_simulations=S)
    eng.set_subtree_reuse(V)
    cap = eng.tree_capacity
    assert cap == (1 + 7 * V + 7) & ~7
    eng.set_roots(bb0, bb1, pl)
    eng.run_simulations(S, 2)
    eng.reset_stats()
    status = eng.advance_roots(cols).cpu().numpy()
    st = eng.reuse_stats()
    err = eng.root_stats()["err"].cpu().numpy()
    got = [export(eng, i, cap) for i in range(E)]
    eng.close()
    ref_st = None
    for lo in range(0, E, 1024):
        ref = reuse_oracle.advance_reuse(bb0, bb1, pl, S, cols, S, V, export_slots=np.arange(lo, lo + 1024), eval_kind=2)
        ref_st = ref["stats"]
        assert np.array_equal(status[lo:lo + 1024], ref["status"][lo:lo + 1024])
        for k in range(1024):
            t, used = got[lo + k]
            assert used == ref["used"][k], lo + k
            for f in TREE_FIELDS:
                assert t[f].tobytes() == ref[f][k].tobytes(), (lo + k, f)
    assert err[1] == TREE_ROOT_ENDED and status[1] == 0 and got[1][1] == 1
    assert (status == 1).sum() >= 64
    assert {k: st[k] for k in ("retained", "fresh", "dropped", "nodes", "visits")} == \
        {k: ref_st[k] for k in ("retained", "fresh", "dropped", "nodes", "visits")}
    ended = int((err == TREE_ROOT_ENDED).sum())  # recycled, not counted
    assert st["retained"] > E // 2 and st["retained"] + st["fresh"] + st["dropped"] == int((status == 0).sum()) - ended

    # the retained tree is the played child's subtree of the tree materialize="full" built before the move
    search = az.AlphaZeroSearch(model=az.HashEvaluator(), num_simulations=S)
    idx = [i for i in range(2, 400) if status[i] == 0][:6]
    nodes = [az.Node(az.State(az.Config(6, 7, 4), int(bb0[i]), int(bb1[i]), int(pl[i]))) for i in idx]
    search.run_simulations(nodes, materialize="full")
    for i, nd in zip(idx, nodes):
        full = node_map(nd)
        c = int(cols[i])
        sub = {p[1:]: v for p, v in full.items() if p[:1] == (c,)}
        t = got[i][0]
        child = nd.children[next(a for a in nd.children if a.column == c)]
        after = tree_map({k: [t[k]] for k in TREE_FIELDS}, 0, child.state.bb0, child.state.bb1, child.state.player)
        if got[i][1] == 1:
            continue  # fresh or dropped
        r = sub.pop(())
        assert after.pop(()) == (r[0], r[1], np.float32(0))
        assert after == sub
    search.close()


def test_advance_roots_unexpanded_child_and_root():
    eng = Engine(num_games=2, num_simulations=8)
    eng.set_subtree_reuse(16)
    eng.set_roots(np.zeros(2, np.uint64), np.zeros(2, np.uint64), np.zeros(2, np.uint8))
    eng.run_simulations(2, 1)  # the root and the child of column 0 (uniform priors, first maximum) are expanded
    assert eng.root_stats()["child_N"].cpu().numpy()[0].tolist() == [1, 0, 0, 0, 0, 0, 0]
    eng.reset_stats()
    assert eng.advance_roots(torch.tensor([3, 3], dtype=torch.uint8)).cpu().tolist() == [0, 0]  # never expanded: fresh
    assert eng.reuse_stats() == dict(retained=0, fresh=2, dropped=0, nodes=0, visits=0)
    for slot in range(2):
        t = eng.export_tree(slot)
        assert t["used"] == 1 and t["N"][0] == 0 and t["first_child"][0] == 0
    # a root that was never searched just takes the new position
    assert eng.advance_roots(torch.tensor([2, 4], dtype=torch.uint8)).cpu().tolist() == [0, 0]
    assert eng.reuse_stats()["fresh"] == 2
    eng.run_simulations(8, 1)
    assert eng.root_stats()["root_N"].cpu().tolist() == [8, 8]
    eng.close()


# ---- 2 / 3. self-play with the built-in evaluators -----------------------------------------------------------------------------
def _flatten(parts):
    return {f: np.concatenate([np.asarray(getattr(b, f)) for b in parts]) for f in EP_FIELDS}


def _builtin_selfplay(E, S, V, kind, lanes, noise, greedy, fused, steps=60, quota=None):
    u2 = np.random.RandomState(E + S + kind).random_sample((steps, E))
    eng = Engine(num_games=E, num_simulations=S, lanes_per_tree=lanes)
    if V:
        eng.set_subtree_reuse(V)
    eng.reset_games()
    if noise:
        eng.set_root_noise(1.0, 0.25, 99 + kind)
    eng.set_greedy_from(greedy)
    etas, parts, count = [], [], 0
    quota = E if quota is None else quota
    for step in range(steps):
        u = torch.from_numpy(u2[step]).cuda()
        n = S
        if noise:
            eng.run_simulations(1, kind)
            eng.apply_root_noise()
            etas.append(eng.root_noise_values().cpu().numpy())
            n = S - 1
        if fused:
            eng.run_move_step(n, kind, u)
        else:
            eng.run_simulations(n, kind)
            eng.sample_moves(u)
        ne, _ = eng.episode_counts()
        if ne:
            parts.append(eng.drain_episodes())
            count += ne
            if count >= quota:
                break
    out = dict(ep=_flatten(parts), steps=step + 1, u=u2, eta=np.stack(etas) if noise else None, stats=eng.stats(),
               reuse=eng.reuse_stats(), cap=eng.tree_capacity)
    eng.close()
    return out


@pytest.mark.parametrize("kind,lanes,noise,greedy,fused,E,V", [
    (1, 8, False, None, True, 4096, 800),
    (2, 8, True, 10, False, 4096, 800),
    (2, 32, False, 8, True, 4096, 800),
    (1, 32, True, None, True, 4096, 400),
    (2, 8, False, None, True, 1024, 9400),  # 1 + 7 V > 65535 nodes: no shared-memory prefix (K = 0)
])
def test_selfplay_with_reuse_vs_oracle(oracle, kind, lanes, noise, greedy, fused, E, V):
    S = 200
    got = _builtin_selfplay(E, S, V, kind, lanes, noise, greedy, fused)
    if V > 9362:
        assert got["cap"] > 65535
    ref, ref_st = reuse_oracle.selfplay_reuse(E, S, V, got["u"][:got["steps"]], 0.25 if noise else 0.0, got["eta"],
                                              greedy_from=-1 if greedy is None else greedy, eval_kind=kind)
    ep = got["ep"]
    ne = len(ref.ep_slot)
    assert ne == E and got["steps"] == ref.n_steps
    ns = int(ref.ep_len.sum())
    for f, r in (("ep_slot", ref.ep_slot), ("ep_step", ref.ep_step), ("ep_len", ref.ep_len), ("ep_outcome", ref.ep_outcome)):
        assert np.array_equal(ep[f][:ne], r), f
    for f, r in (("s_bb0", ref.s_bb0), ("s_bb1", ref.s_bb1), ("s_player", ref.s_player), ("s_counts", ref.s_counts)):
        assert np.array_equal(ep[f][:ns].view(r.dtype) if f.startswith("s_bb") else ep[f][:ns], r), f
    assert got["stats"]["simulations"] == ref.n_sims and got["stats"]["evaluations"] == ref.n_evals
    assert got["reuse"]["retained"] > 0 and ref_st["max_used"] <= 1 + 7 * V
    assert (ref.s_counts.sum(1) > S - 1).any()


@pytest.mark.parametrize("fused", [True, False])
def test_v_equal_s_is_reuse_off(fused):
    off = _builtin_selfplay(4096, 200, 0, 2, 8, False, None, fused, steps=30, quota=10**9)
    same = _builtin_selfplay(4096, 200, 200, 2, 8, False, None, fused, steps=30, quota=10**9)
    for f in EP_FIELDS:
        assert off["ep"][f].tobytes() == same["ep"][f].tobytes(), f
    assert off["stats"] == same["stats"]
    assert same["reuse"]["retained"] == 0 and same["reuse"]["dropped"] > 0


# ---- 4. ResNet 4x64 in the loop ------------------------------------------------------------------------------------------------
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


def _net_selfplay(reuse=True, cache=True, graph=True, symmetric=False):
    search = az.AlphaZeroSearch(model=_resnet(), num_simulations=NS, inference_dtype=torch.bfloat16, eval_cache=cache,
                                use_cuda_graph=graph, symmetric=symmetric, subtree_reuse=reuse)
    eng = search.engine_for(NE, exact=True)
    eng.reset_games()
    u = torch.from_numpy(np.random.RandomState(5).random_sample((NSTEPS, NE))).cuda()
    episodes, samples = [], 0
    for step in range(NSTEPS):
        search.simulate_and_move(eng, u[step])
        b = eng.drain_episodes()
        episodes.append({f: np.asarray(getattr(b, f)).copy() for f in EP_FIELDS})
    roots = {k: v.cpu().numpy() for k, v in eng.root_stats().items()}
    out = dict(roots=roots, episodes=episodes, stats=eng.stats(), reuse=eng.reuse_stats(), cache=eng.eval_cache_stats(),
               kernel=search.evaluator_name, log2=eng.eval_cache_log2)
    search.close()
    return out


def _same(a, b):
    return (a["stats"] == b["stats"] and a["reuse"] == b["reuse"] and all(np.array_equal(a["roots"][k], b["roots"][k]) for k in a["roots"])
            and all(np.array_equal(ea[k], eb[k]) for ea, eb in zip(a["episodes"], b["episodes"]) for k in ea))


@pytest.mark.parametrize("symmetric", [False, True])
def test_network_reuse_cache_and_graph_change_no_bit(symmetric):
    ref = _net_selfplay(symmetric=symmetric)
    assert ref["kernel"] == "k_resnet_wide" and ref["log2"] > 0 and ref["cache"]["hits"] > 0
    assert ref["reuse"]["retained"] > NE
    assert any((ep["s_counts"].sum(1) > NS - 1).any() for ep in ref["episodes"])  # roots that kept their subtree
    for kw in (dict(cache=False), dict(graph=False)):
        other = _net_selfplay(symmetric=symmetric, **kw)
        assert _same(ref, other), kw
    if not symmetric:
        assert not _same(ref, _net_selfplay(reuse=False))


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


def test_network_reused_trees_vs_oracle(oracle):
    V = 4 * NS
    search = az.AlphaZeroSearch(model=_resnet(), num_simulations=NS, inference_dtype=torch.bfloat16)
    bb0, bb1, pl = random_positions(oracle, NE, seed=13, max_plies=12)
    cols = np.array([legal_cols(bb0[i], bb1[i])[i % len(legal_cols(bb0[i], bb1[i]))] for i in range(NE)], np.uint8)
    eng = search.engine_for(NE)
    eng.set_subtree_reuse(V)
    eng.set_roots(bb0, bb1, pl)
    search.simulate(eng)
    assert (eng.advance_roots(cols).cpu().numpy() == 0).all()
    assert eng.reuse_stats()["retained"] > NE // 2
    search.simulate(eng)
    idx = np.random.RandomState(5).choice(NE, 12, replace=False)
    got = [export(eng, int(i), eng.tree_capacity) for i in idx]
    ref = reuse_oracle.advance_reuse(bb0[idx], bb1[idx], pl[idx], NS, cols[idx], NS, V, S2=NS, py_eval=KernelEvaluator(search._net))
    for k in range(len(idx)):
        assert got[k][1] == ref["used"][k]
        for f in TREE_FIELDS:
            assert got[k][0][f].tobytes() == ref[f][k].tobytes(), (k, f)
    search.close()


# ---- 5 / 6 / 7. tables, guards, launch counts, trainer -------------------------------------------------------------------------
def test_division_selftest_over_the_enlarged_tables():
    eng = Engine(num_games=64, num_simulations=200)
    eng.set_subtree_reuse(9400)
    assert eng.selftest_division(1 << 24, seed=3) == 0
    eng.close()


def test_guards():
    eng = Engine(num_games=64, num_simulations=32)
    cap0 = eng.tree_capacity
    with pytest.raises(RuntimeError, match=r"\(-1\)"):
        eng.set_subtree_reuse(31)
    with pytest.raises(RuntimeError, match=r"\(-1\)"):
        eng.set_subtree_reuse(1 << 17)
    with pytest.raises(RuntimeError, match=r"\(-4\)"):
        eng.advance_roots(torch.zeros(64, dtype=torch.uint8))  # reuse off
    eng.reset_games()
    eng.select_leaves()
    with pytest.raises(RuntimeError, match=r"\(-4\)"):
        eng.set_subtree_reuse(64)
    eng.expand_backup(torch.zeros(64, 7, device="cuda"), torch.zeros(64, 2, device="cuda"))
    eng.set_subtree_reuse(64)
    assert eng.tree_capacity == (1 + 7 * 64 + 7) & ~7
    eng.set_subtree_reuse(None)
    assert eng.tree_capacity == cap0
    eng.close()


@pytest.mark.parametrize("spec", ["builtin", "builtin_greedy", "builtin_noise", "basic"])
def test_launches_per_move_step_with_reuse(spec):
    S, E = 24, 256
    model = az.BasicNN() if spec == "basic" else az.UniformEvaluator()
    search = az.AlphaZeroSearch(model=model, num_simulations=S, use_cuda_graph=False, subtree_reuse=True,
                                root_noise=az.RootNoise(seed=1) if spec == "builtin_noise" else None)
    eng = search.engine_for(E, exact=True)
    eng.reset_games()
    eng.set_greedy_from(4 if spec == "builtin_greedy" else None)
    u = torch.from_numpy(np.random.RandomState(0).random_sample((3, E))).cuda()
    search.simulate_and_move(eng, u[0])  # first step: one-off allocations and the reuse setting
    for s in (1, 2):
        n0 = eng.launch_count
        search.simulate_and_move(eng, u[s])
        assert eng.launch_count - n0 == search.launches_per_move_step(), spec
    expect = {"builtin": 3, "builtin_greedy": 3, "builtin_noise": 5, "basic": 2 * S + 3}[spec]
    assert search.launches_per_move_step() == expect
    assert eng.subtree_reuse == 4 * S and eng.reuse_stats()["retained"] > 0
    search.close()


def test_trainer_with_reuse():
    from alphazero_implementation_b200.trainer import Trainer

    torch.manual_seed(0)
    np.random.seed(0)
    tr = Trainer(az.BasicNN())
    hist = tr.train(num_iterations=2, episodes_per_iter=32, simulations_per_episode=32, epochs_per_iter=1,
                    initial_state=az.Config(6, 7, 4).sample_initial_state(), buffer_size=64, subtree_reuse=True)
    assert len(hist) == 2 and hist[0]["episodes"] == 32 and hist[1]["episodes"] == 64
    assert hist[0]["samples"] >= 32 * 7 and hist[1]["loss"] is not None
