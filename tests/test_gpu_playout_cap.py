"""GPU: playout cap randomization (az_set_playout_cap: k_cap_draw, the BUDGET builds of k_select / k_expand_select / k_run_sims /
k_sample_moves / k_root_noise).  The engine's full / fast flags are the host restatement of the draw bit for bit; every search
stops at exactly N_start + n_t root visits and stopped trees are never evaluated; self-play is bit-exact against
tests/native/c4_cap_oracle.c fed the engine's flags (and eta) on the built-in evaluators, with reuse and the total-visit budget too;
with ResNet 4x64 in the loop the evaluation cache and the CUDA graph change no bit; p_full = 1 is the mode off; the guards hold."""
import ctypes as C

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

import alphazero_implementation_b200 as az  # noqa: E402
from alphazero_implementation_b200.engine import LEAF_IDLE, POLICY_LOGITS, Engine  # noqa: E402
import cap_oracle  # noqa: E402

AZ_E_INVALID, AZ_E_STATE = -1, -4
EP_FIELDS = ("ep_slot", "ep_step", "ep_len", "ep_outcome", "s_bb0", "s_bb1", "s_player", "s_counts")


def budgets(eng):
    b, f = eng.search_budgets()
    return b.cpu().numpy(), f.cpu().numpy()


def root_n(eng):
    return eng.root_stats()["root_N"].cpu().numpy().astype(np.int64)


def concat(batches):
    out = {}
    for f in EP_FIELDS:
        xs = [getattr(b, f) for b in batches]
        out[f] = np.concatenate(xs) if xs else np.zeros(0)
    return out


# ---- 1. the draw ---------------------------------------------------------------------------------------------------------------
def test_flags_are_the_host_draw():
    E, S, seed, p = 16384, 8, 0x1234_5678_9ABC_DEF0, 0.25
    eng = Engine(E, S)
    eng.reset_games()
    eng.set_playout_cap(3, p, seed)
    u = torch.zeros(E, dtype=torch.float64, device=eng.device)
    for step in range(5):
        b, f = budgets(eng)
        assert np.array_equal(f, cap_oracle.draw_full(seed, 0, E, step, p)), step
        assert np.array_equal(b, np.where(f == 1, S, 3)), step  # fresh roots: N_start = 0
        eng.sample_moves(u)  # no search ran: every slot keeps its root, the next step's flags are drawn
    eng.reset_games()  # back to step 0
    assert np.array_equal(budgets(eng)[1], cap_oracle.draw_full(seed, 0, E, 0, p))
    eng.close()


@pytest.mark.parametrize("p", [0.1, 0.25, 0.9])
def test_full_fraction_is_binomial(p):
    E = 16384
    eng = Engine(E, 4)
    eng.reset_games()
    eng.set_playout_cap(1, p, seed=7)
    k = int(budgets(eng)[1].sum())
    assert abs(k - E * p) < 6 * np.sqrt(E * p * (1 - p))
    eng.close()


def test_slot_offset_selects_rows():
    E, lo, hi, p = 4096, 1000, 3000, 0.4
    full = Engine(E, 4)
    part = Engine(hi - lo, 4)
    for eng, off in ((full, 0), (part, lo)):
        eng.reset_games()
        eng.set_playout_cap(2, p, seed=99, slot_offset=off)
    assert np.array_equal(budgets(full)[1][lo:hi], budgets(part)[1])
    full.close(); part.close()


def _selfplay_engine(E, S, steps, kind, cap, u, lanes=0, noise=None, greedy_from=None, V=0, slot_offset=0, final_search=False):
    """drive the engine's self-play loop; -> (episodes, flags [steps, E], eta [steps, E, 7] or None, engine stats).  final_search:
    one more search after the loop, its root statistics in stats["roots"]"""
    eng = Engine(E, S, lanes_per_tree=lanes)
    if V:
        eng.set_subtree_reuse(V)
    eng.set_greedy_from(greedy_from)
    if noise is not None:
        eng.set_root_noise(noise[0], noise[1], seed=noise[2], slot_offset=slot_offset)
    eng.reset_games()
    eng.set_playout_cap(cap["fast"], cap["p"], cap["seed"], slot_offset, cap.get("visit_budget", False))
    flags, etas, batches = [], [], []
    for k in range(steps):
        flags.append(budgets(eng)[1])
        ud = torch.from_numpy(u[k]).to(eng.device)
        if noise is not None:
            eng.run_simulations(1, kind)
            eng.apply_root_noise()
            etas.append(eng.root_noise_values().cpu().numpy())
            eng.run_move_step(S - 1, kind, ud)
        else:
            eng.run_move_step(S, kind, ud)
        batches.append(eng.drain_episodes())
    roots = None
    if final_search:
        eng.run_simulations(S, kind)
        roots = {k: v.cpu().numpy() for k, v in eng.root_stats().items()}
    st = dict(eng.stats(), **eng.cap_stats(), roots=roots)
    eng.close()
    return concat(batches), np.stack(flags), (np.stack(etas) if etas else None), st


def test_sharded_selfplay_is_unsharded():
    E, S, steps = 2048, 32, 40
    cap = dict(fast=6, p=0.3, seed=5)
    u = np.random.RandomState(1).random_sample((steps, E))
    whole, fw, _, _ = _selfplay_engine(E, S, steps, 2, cap, u)
    lo = 768
    a, fa, _, _ = _selfplay_engine(lo, S, steps, 2, cap, u[:, :lo])
    b, fb, _, _ = _selfplay_engine(E - lo, S, steps, 2, cap, u[:, lo:], slot_offset=lo)
    assert np.array_equal(fw, np.concatenate([fa, fb], 1))
    for part, off in ((a, 0), (b, lo)):
        sel = (whole["ep_slot"] >= off) & (whole["ep_slot"] < off + (lo if off == 0 else E - lo))
        assert np.array_equal(whole["ep_slot"][sel] - off, part["ep_slot"])
        assert np.array_equal(whole["ep_len"][sel], part["ep_len"])
        assert np.array_equal(whole["ep_outcome"][sel], part["ep_outcome"])


# ---- 2. budgets are exact ------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("lanes", [8, 32])
def test_budgets_exact_fused(lanes):
    E, S, F = 1024, 48, 9
    eng = Engine(E, S, lanes_per_tree=lanes)
    eng.set_subtree_reuse(4 * S)
    eng.reset_games()
    eng.set_playout_cap(F, 0.3, seed=3, visit_budget=True)
    rng = np.random.RandomState(2)
    for k in range(12):
        n0 = root_n(eng)
        b, f = budgets(eng)
        want = np.maximum(np.where(f == 1, S, F) - n0, 1)
        assert np.array_equal(b, n0 + want)
        s0 = eng.stats()["simulations"]
        eng.run_simulations(S, 2)
        assert np.array_equal(root_n(eng), n0 + want), k
        assert eng.stats()["simulations"] - s0 == int(want.sum())
        eng.sample_moves(torch.from_numpy(rng.random_sample(E)).to(eng.device))
    eng.close()


@pytest.mark.parametrize("compaction", [1, 2])
def test_budgets_exact_split_path_and_idle_leaves(compaction):
    E, S, F = 1024, 40, 7
    eng = Engine(E, S)
    eng.set_leaf_compaction(True, fused=compaction == 2)
    eng.reset_games()
    eng.set_playout_cap(F, 0.25, seed=11)
    rng = np.random.RandomState(4)
    logits = torch.from_numpy(rng.standard_normal((E, 7)).astype(np.float32)).to(eng.device)
    values = torch.zeros((E, 2), dtype=torch.float32, device=eng.device)
    for k in range(6):
        n0 = root_n(eng)
        b, f = budgets(eng)
        s0 = eng.stats()["simulations"]
        for s in range(S):
            before = root_n(eng)
            if s == 0:
                eng.select_leaves()
            else:
                eng.expand_backup_select(logits, values, POLICY_LOGITS)
            stopped = before >= b
            status = eng.leaf_info()["status"].cpu().numpy()
            assert (status[stopped] == LEAF_IDLE).all()
            lst, cnt = eng.leaf_compact()
            listed = lst[:int(cnt[0].item())].cpu().numpy()
            assert not stopped[listed].any()
        eng.expand_backup(logits, values, POLICY_LOGITS)
        want = np.where(f == 1, S, F)
        assert np.array_equal(root_n(eng), n0 + want), k
        assert eng.stats()["simulations"] - s0 == int(want.sum())
        eng.sample_moves(torch.from_numpy(rng.random_sample(E)).to(eng.device))
    eng.close()


# ---- 3. bit-exact self-play ----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kind,lanes,noise,greedy", [(1, 8, False, None), (2, 8, False, None), (2, 32, False, 6), (2, 8, True, None),
                                                     (1, 32, True, 10)])
def test_selfplay_matches_cap_oracle(kind, lanes, noise, greedy):
    E, S, steps = 4096, 48, 40
    cap = dict(fast=8, p=0.25, seed=21)
    u = np.random.RandomState(5).random_sample((steps, E))
    nz = (0.3, 0.25, 77) if noise else None
    got, flags, eta, st = _selfplay_engine(E, S, steps, kind, cap, u, lanes=lanes, noise=nz, greedy_from=greedy)
    ref, extra = cap_oracle.selfplay_cap(E, S, cap["fast"], flags, u, eps=0.25 if noise else 0.0, eta=eta,
                                         greedy_from=-1 if greedy is None else greedy, quota=E * steps, eval_kind=kind)
    assert len(ref.ep_slot) > E // 2
    for f in EP_FIELDS:
        assert np.array_equal(got[f], getattr(ref, f)), f
    assert st["simulations"] == ref.n_sims
    assert st["samples_recorded"] == int(ref.ep_len.sum()) and st["samples_dropped"] == extra["samples_dropped"]
    assert st["full_searches"] + st["fast_searches"] == E * steps
    assert (ref.ep_len == 0).any()  # games without a full search are still episodes


@pytest.mark.parametrize("visit_budget", [False, True])
def test_selfplay_with_reuse_matches_cap_oracle(visit_budget):
    E, S, V, steps = 4096, 40, 160, 40
    cap = dict(fast=8, p=0.25, seed=8, visit_budget=visit_budget)
    u = np.random.RandomState(6).random_sample((steps, E))
    got, flags, _, st = _selfplay_engine(E, S, steps, 2, cap, u, V=V)
    ref, extra = cap_oracle.selfplay_cap(E, S, cap["fast"], flags, u, V=V, visit_budget=visit_budget, quota=E * steps, eval_kind=2)
    for f in EP_FIELDS:
        assert np.array_equal(got[f], getattr(ref, f)), f
    assert st["simulations"] == ref.n_sims and extra["retained"] > 0


# ---- 4. network in the loop ----------------------------------------------------------------------------------------------------
def _net_selfplay(model, E, S, steps, cap, cache, graph, symmetric=False, dtype=torch.bfloat16):
    gen = az.EpisodeGenerator(model=model, num_simulations=S, num_episodes=E, game_initial_state=az.Config(6, 7, 4).sample_initial_state(),
                              uniform_source=lambda step, n: np.random.RandomState(1000 + step).random_sample(n), inference_dtype=dtype,
                              eval_cache=cache, use_cuda_graph=graph, symmetric=symmetric, playout_cap=cap)
    batches = [b for _, b, _ in gen.iter_steps(max_steps=steps) if b is not None]
    eng = gen.search._engine
    rs = {k: v.cpu().numpy() for k, v in eng.root_stats().items()}
    st = eng.cap_stats()
    gen.search.close()
    return concat(batches), rs, st


@pytest.mark.parametrize("symmetric", [False, True])
def test_resnet_cache_and_graph_change_nothing(symmetric):
    torch.manual_seed(0)
    model = az.ResNet(num_res_blocks=4, num_channels=64).cuda()
    cap = az.PlayoutCap(fast_simulations=160, full_probability=0.25, seed=4)
    E, S, steps = 2048, 800, 12
    runs = [_net_selfplay(model, E, S, steps, cap, cache, graph, symmetric) for cache, graph in ((True, True), (False, True), (True, False))]
    a = runs[0]
    assert a[2]["fast_searches"] > a[2]["full_searches"] > 0
    for b in runs[1:]:
        for f in EP_FIELDS:
            assert np.array_equal(a[0][f], b[0][f]), f
        for k in ("child_N", "child_W", "child_P", "root_N"):
            assert np.array_equal(a[1][k], b[1][k]), k
        assert a[2] == b[2]


def test_basicnn_graph_changes_nothing():
    torch.manual_seed(1)
    model = az.BasicNN().cuda()
    cap = az.PlayoutCap(fast_simulations=16, full_probability=0.3, seed=2)
    runs = [_net_selfplay(model, 1024, 64, 20, cap, False, graph, dtype=torch.bfloat16) for graph in (True, False)]
    for f in EP_FIELDS:
        assert np.array_equal(runs[0][0][f], runs[1][0][f]), f
    assert runs[0][2] == runs[1][2] and runs[0][2]["fast_searches"] > 0


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


@pytest.mark.parametrize("spec", ["resnet4x64", "basic"])
def test_network_trees_vs_cap_oracle(spec):
    """The production loop (k_resnet_wide with compaction and the cache, or k_mlp_fused without compaction; CUDA graph on) over
    2048 games x 800 simulations x 12 move steps, against the cap oracle fed the engine's flags and the kernels' outputs, on a
    sample of slots: the episodes they finished and the root visit counts of the last search."""
    E, S, steps, n_check = 2048, 800, 12, 12
    torch.manual_seed(0)
    model = az.ResNet(num_res_blocks=4, num_channels=64) if spec == "resnet4x64" else az.BasicNN()
    cap = az.PlayoutCap(fast_simulations=160, full_probability=0.25, seed=9)
    search = az.AlphaZeroSearch(model=model, num_simulations=S, inference_dtype=torch.bfloat16, playout_cap=cap)
    eng = search.engine_for(E, exact=True)
    eng.reset_games()
    eng.set_playout_cap(cap.fast_simulations, cap.full_probability, cap.seed)  # what simulate_and_move configures, before the first draw
    u = np.random.RandomState(21).random_sample((steps, E))
    flags, batches = [], []
    for k in range(steps):
        flags.append(budgets(eng)[1])
        if k + 1 < steps:
            search.simulate_and_move(eng, torch.from_numpy(u[k]).to(eng.device))
            batches.append(eng.drain_episodes())
        else:
            search.simulate(eng)
            last = eng.root_stats()["child_N"].cpu().numpy()
    flags = np.stack(flags)
    assert 0 < flags.mean() < 0.5
    got = concat(batches)
    idx = np.sort(np.random.RandomState(5).choice(E, n_check, replace=False))
    ref, extra = cap_oracle.selfplay_cap(n_check, S, cap.fast_simulations, flags[:, idx], u[:, idx], quota=n_check * steps,
                                         py_eval=KernelEvaluator(search._net))
    assert np.array_equal(last[idx], extra["last_counts"])
    assert (last[idx].sum(1) == np.where(flags[-1, idx] == 1, S, cap.fast_simulations) - 1).all()
    # the episodes of the sampled slots that ended before the last move step, with their samples
    start = np.cumsum(got["ep_len"]) - got["ep_len"]
    ref_start = np.cumsum(ref.ep_len) - ref.ep_len
    mine = [i for i in range(len(got["ep_slot"])) if got["ep_slot"][i] in idx]
    theirs = [i for i in range(len(ref.ep_slot)) if ref.ep_step[i] < steps - 1]
    assert len(mine) == len(theirs)
    for i, j in zip(mine, theirs):
        assert idx[ref.ep_slot[j]] == got["ep_slot"][i] and ref.ep_step[j] == got["ep_step"][i]
        assert ref.ep_len[j] == got["ep_len"][i] and np.array_equal(ref.ep_outcome[j], got["ep_outcome"][i])
        a, b, n = start[i], ref_start[j], got["ep_len"][i]
        for f in ("s_bb0", "s_bb1", "s_player", "s_counts"):
            assert np.array_equal(got[f][a:a + n], getattr(ref, f)[b:b + n]), f
    search.close()


# ---- 5. degenerate settings ----------------------------------------------------------------------------------------------------
def _plain_selfplay(E, S, steps, kind, u):
    eng = Engine(E, S)
    eng.reset_games()
    batches = []
    for k in range(steps):
        eng.run_move_step(S, kind, torch.from_numpy(u[k]).to(eng.device))
        batches.append(eng.drain_episodes())
    eng.run_simulations(S, kind)  # one more search: root statistics of searched trees
    rs = {k: v.cpu().numpy() for k, v in eng.root_stats().items()}
    st = eng.stats()
    eng.close()
    return concat(batches), rs, st


def test_p_full_one_is_off():
    E, S, steps = 2048, 40, 40
    u = np.random.RandomState(9).random_sample((steps, E))
    off, rs_off, st_off = _plain_selfplay(E, S, steps, 2, u)
    on, flags, _, st_on = _selfplay_engine(E, S, steps, 2, dict(fast=3, p=1.0, seed=1), u, final_search=True)
    assert flags.all()
    for f in EP_FIELDS:
        assert np.array_equal(off[f], on[f]), f
    for k in ("child_N", "child_W", "child_P", "root_W", "root_N", "legal", "err"):
        assert rs_off[k].tobytes() == st_on["roots"][k].tobytes(), k
    assert (rs_off["root_N"] == S).all()
    for k in ("simulations", "evaluations", "levels", "children_created", "moves", "episodes"):
        assert st_off[k] == st_on[k], k
    assert st_on["samples_dropped"] == 0 and st_on["samples_recorded"] == len(off["s_bb0"])


def test_all_fast_at_full_size_is_off_without_samples():
    E, S, steps = 2048, 40, 40
    u = np.random.RandomState(10).random_sample((steps, E))
    off, _, st_off = _plain_selfplay(E, S, steps, 1, u)
    on, flags, _, st_on = _selfplay_engine(E, S, steps, 1, dict(fast=S, p=0.0, seed=1), u, final_search=True)
    assert not flags.any()
    for f in ("ep_slot", "ep_step", "ep_outcome"):
        assert np.array_equal(off[f], on[f]), f
    assert (on["ep_len"] == 0).all() and len(on["s_bb0"]) == 0
    assert st_on["simulations"] == st_off["simulations"] and st_on["samples_dropped"] == len(off["s_bb0"])


# ---- 6. noise ------------------------------------------------------------------------------------------------------------------
def test_noise_only_on_full_searches():
    E, S = 4096, 16
    plain = Engine(E, S)
    capped = Engine(E, S)
    for eng in (plain, capped):
        eng.set_root_noise(0.3, 0.25, seed=3)
        eng.reset_games()
        eng.run_simulations(1, 2)
    capped.set_playout_cap(4, 0.5, seed=6)
    for eng in (plain, capped):
        eng.apply_root_noise()
    f = budgets(capped)[1].astype(bool)
    e_plain, e_cap = plain.root_noise_values().cpu().numpy(), capped.root_noise_values().cpu().numpy()
    assert (e_cap[~f] == 0).all() and np.array_equal(e_cap[f], e_plain[f]) and f.any() and (~f).any()
    p_plain, p_cap = plain.root_stats()["child_P"].cpu().numpy(), capped.root_stats()["child_P"].cpu().numpy()
    assert np.array_equal(p_cap[f].view(np.uint32), p_plain[f].view(np.uint32))
    assert not np.array_equal(p_cap[~f], p_plain[~f])
    plain.close(); capped.close()


# ---- 7. guards and integration -------------------------------------------------------------------------------------------------
def test_guards():
    eng = Engine(64, 20)
    with pytest.raises(RuntimeError):
        eng.search_budgets()  # nothing configured yet
    lib = eng.lib
    bad = [(0, 0.5, 0, 0, 0), (21, 0.5, 0, 0, 0), (5, -0.1, 0, 0, 0), (5, 1.5, 0, 0, 0), (5, float("nan"), 0, 0, 0), (5, 0.5, 0, -1, 0),
           (5, 0.5, 0, 2**62 + 1, 0), (5, 0.5, 0, 0, 2)]
    for args in bad:
        assert lib.az_set_playout_cap(eng.h, C.byref(az._lib.AzPlayoutCap(*args))) == AZ_E_INVALID, args
    assert eng.playout_cap is None
    eng.reset_games()
    eng.select_leaves()
    assert lib.az_set_playout_cap(eng.h, C.byref(az._lib.AzPlayoutCap(5, 0.5, 0, 0, 0))) == AZ_E_STATE
    assert lib.az_set_playout_cap(eng.h, None) == AZ_E_STATE
    eng.expand_backup(torch.zeros((64, 7), device=eng.device), torch.zeros((64, 2), device=eng.device))
    eng.set_playout_cap(5, 0.5)
    eng.set_playout_cap(None)
    eng.close()


def test_run_simulations_ignores_the_cap():
    nodes_a = [az.Node(az.Config(6, 7, 4).sample_initial_state()) for _ in range(32)]
    nodes_b = [az.Node(az.Config(6, 7, 4).sample_initial_state()) for _ in range(32)]
    torch.manual_seed(0)
    model = az.ResNet(num_res_blocks=1, num_channels=64).cuda()
    s = az.AlphaZeroSearch(model=model, num_simulations=40, inference_dtype=torch.bfloat16)
    s.run_simulations(nodes_a)
    eng = s.engine_for(32)
    eng.set_playout_cap(3, 0.0, seed=1)  # every self-play search would be fast
    s.run_simulations(nodes_b)
    for a, b in zip(nodes_a, nodes_b):
        assert a.visit_count == b.visit_count == 40
        assert [c.visit_count for c in a.children.values()] == [c.visit_count for c in b.children.values()]
    s.close()


@pytest.mark.parametrize("model_kind,reuse,noise", [("builtin", False, False), ("builtin", True, True), ("basic", False, True),
                                                    ("basic", True, False)])
def test_launches_per_move_step(model_kind, reuse, noise):
    E, S = 512, 48
    torch.manual_seed(0)
    if model_kind == "basic":
        model = az.BasicNN()
    else:
        from alphazero_implementation_b200.evaluators import HashEvaluator

        model = HashEvaluator()
    # un-graphed: a replayed CUDA graph launches its kernels without the host counting them
    s = az.AlphaZeroSearch(model=model, num_simulations=S, subtree_reuse=reuse, use_cuda_graph=False,
                           root_noise=az.RootNoise(0.3, 0.25) if noise else None, playout_cap=az.PlayoutCap(8, 0.25, seed=1))
    eng = s.engine_for(E, exact=True)
    eng.reset_games()
    u = torch.rand(E, dtype=torch.float64, device=eng.device)
    s.simulate_and_move(eng, u)  # first step: one-off allocations and the settings
    for _ in range(2):
        n0 = eng.launch_count
        s.simulate_and_move(eng, u)
        assert eng.launch_count - n0 == s.launches_per_move_step()
    s.close()


def test_generate_episodes_with_empty_episodes():
    torch.manual_seed(0)
    model = az.ResNet(num_res_blocks=1, num_channels=64).cuda()
    gen = az.EpisodeGenerator(model=model, num_simulations=32, num_episodes=256, game_initial_state=az.Config(6, 7, 4).sample_initial_state(),
                              inference_dtype=torch.bfloat16, playout_cap=az.PlayoutCap(4, 0.05, seed=2))
    eps = list(gen.generate_episodes())
    assert len(eps) == 256
    assert any(len(e.samples) == 0 for e in eps) and any(len(e.samples) > 0 for e in eps)
    from alphazero_implementation_b200.replay import ReplayBuffer

    buf = ReplayBuffer(100, 32, "cuda")
    for _, b, _ in gen.iter_steps(max_steps=60):
        if b is not None:
            buf.extend(b)
    assert len(buf) == 100  # empty episodes count
    assert buf.num_samples == int(buf.tensors()[0].shape[0])
    gen.search.close()


def _trainer_worker(rank, world, port, out):
    import torch.distributed as dist

    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", init_method=f"tcp://127.0.0.1:{port}", rank=rank, world_size=world)
    try:
        from alphazero_implementation_b200.trainer import Trainer

        torch.manual_seed(0)
        np.random.seed(0)
        tr = Trainer(az.BasicNN(), device=rank)
        hist = tr.train(num_iterations=2, episodes_per_iter=32, simulations_per_episode=32, epochs_per_iter=1,
                        initial_state=az.Config(6, 7, 4).sample_initial_state(), buffer_size=64,
                        playout_cap=az.PlayoutCap(fast_simulations=8, full_probability=0.5, seed=3))
        out.put((rank, [h["episodes"] for h in hist], [h["samples"] for h in hist]))
    finally:
        dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_trainer_with_playout_cap_on_two_gpus():
    import socket
    import torch.multiprocessing as mp

    with socket.socket() as sk:
        sk.bind(("127.0.0.1", 0))
        port = sk.getsockname()[1]
    ctx = mp.get_context("spawn")
    out = ctx.Queue()
    procs = [ctx.Process(target=_trainer_worker, args=(r, 2, port, out)) for r in range(2)]
    for p in procs:
        p.start()
    res = dict((r, (e, s)) for r, e, s in (out.get(timeout=600) for _ in procs))
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    assert res[0] == res[1]  # both ranks train on the all-gathered episodes
    assert res[0][0] == [32, 64] and 0 < res[0][1][0] < 32 * 42


def test_trainer_with_playout_cap():
    from alphazero_implementation_b200.trainer import Trainer

    torch.manual_seed(0)
    np.random.seed(0)
    tr = Trainer(az.BasicNN())
    hist = tr.train(num_iterations=2, episodes_per_iter=32, simulations_per_episode=32, epochs_per_iter=1,
                    initial_state=az.Config(6, 7, 4).sample_initial_state(), buffer_size=64,
                    playout_cap=az.PlayoutCap(fast_simulations=8, full_probability=0.5, seed=3))
    assert len(hist) == 2 and hist[0]["episodes"] == 32 and hist[1]["episodes"] == 64
    assert 0 < hist[0]["samples"] < 32 * 42 and hist[1]["loss"] is not None
