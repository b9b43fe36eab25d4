"""Forced playouts and policy target pruning (az_set_forced_playouts: the FORCED builds of k_select / k_expand_select / k_run_sims /
k_sample_moves, and k_policy_targets).  k = 0 is the mode off bit for bit; policy_targets() is the numpy restatement of the pruning;
self-play is bit-exact against tests/native/c4_forced_oracle.c fed the engine's eta and cap flags on the built-in evaluators, with
noise, the greedy cutoff, subtree reuse, the playout cap and its visit budget, and its counters are the oracle's; with ResNet 4x64 in
the loop the evaluation cache and the CUDA graph change no bit and the runs match the oracle fed the kernels' outputs; the guards
hold.  The SASS check of the FORCED level loop needs no GPU."""
import ctypes as C
import re

import numpy as np
import pytest
import torch

import alphazero_implementation_b200 as az
from alphazero_implementation_b200.engine import Engine
import forced_oracle
from test_abi import _sass_of
from test_gpu_playout_cap import EP_FIELDS, KernelEvaluator, budgets, concat

AZ_E_INVALID, AZ_E_STATE = -1, -4
ROOT_KEYS = ("child_N", "child_W", "child_P", "root_W", "root_N", "legal", "err")


def test_level_loop_of_a_forced_fused_tree_kernel_stays_straight_line():
    """The forced rule is a select on a predicate computed before the level loop: the loop of a FORCED k_run_sims build (4 trees
    per warp, uniform evaluator, latency variant, no fused move, tables in shared memory) has no reconvergence region."""
    from alphazero_implementation_b200 import _lib

    ins = _sass_of(_lib.build_library(), r"k_run_simsILi4ELi1ELb1ELb0ELb1ELb0ELb1E")
    assert len(ins) > 1000
    loops = []
    for addr, text in ins:
        m = re.search(r"\bBRA(?:\.U)?\s+(?:!?U?P\d,\s*)?0x([0-9a-f]+)", text)
        if m and int(m.group(1), 16) < addr:
            body = [t for a, t in ins if int(m.group(1), 16) <= a <= addr]
            if any("SHFL.BFLY" in t for t in body):
                loops.append(body)
    level = min(loops, key=len)
    assert 100 < len(level) <= 175, len(level)
    assert not any(t.startswith(("BSSY", "BSYNC")) or " BSSY" in t for t in level)


def _selfplay(E, S, steps, kind, u, k, lanes=0, noise=None, greedy=None, V=0, cap=None, final_search=False):
    """the engine's self-play loop with forced playouts of parameter k (None = off); -> (episodes, flags [steps, E] or None,
    eta [steps, E, 7] or None, stats, roots of one more search or None)"""
    eng = Engine(E, S, lanes_per_tree=lanes)
    if V:
        eng.set_subtree_reuse(V)
    eng.set_greedy_from(greedy)
    if noise is not None:
        eng.set_root_noise(noise[0], noise[1], seed=noise[2])
    eng.reset_games()
    if cap is not None:
        eng.set_playout_cap(cap["fast"], cap["p"], cap["seed"], 0, cap.get("visit_budget", False))
    eng.set_forced_playouts(k)
    flags, etas, batches = [], [], []
    for step in range(steps):
        if cap is not None:
            flags.append(budgets(eng)[1])
        ud = torch.from_numpy(u[step]).to(eng.device)
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
        roots = {k_: v.cpu().numpy() for k_, v in eng.root_stats().items()}
    st = dict(eng.stats(), **eng.forced_stats())
    eng.close()
    return concat(batches), (np.stack(flags) if flags else None), (np.stack(etas) if etas else None), st, roots


# ---- 1. k = 0 is the mode off --------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("kind,noise", [(1, False), (2, False), (2, True)])
def test_k0_is_off_builtin(kind, noise):
    E, S, steps = 2048, 40, 40
    u = np.random.RandomState(9).random_sample((steps, E))
    nz = (0.3, 0.25, 5) if noise else None
    off, _, eta_off, st_off, r_off = _selfplay(E, S, steps, kind, u, None, noise=nz, final_search=True)
    on, _, eta_on, st_on, r_on = _selfplay(E, S, steps, kind, u, 0.0, noise=nz, final_search=True)
    for f in EP_FIELDS:
        assert off[f].tobytes() == on[f].tobytes(), f
    for key in ROOT_KEYS:
        assert r_off[key].tobytes() == r_on[key].tobytes(), key
    if noise:
        assert eta_off.tobytes() == eta_on.tobytes()
    for key in ("simulations", "evaluations", "levels", "children_created", "moves", "episodes"):
        assert st_off[key] == st_on[key], key
    assert st_on["forced_selections"] == 0 and st_on["visits_pruned"] == 0 and st_on["forced_searches"] == E * steps


def _net_selfplay(model, E, S, steps, forced, cache=True, graph=True, noise=None):
    gen = az.EpisodeGenerator(model=model, num_simulations=S, num_episodes=E, game_initial_state=az.Config(6, 7, 4).sample_initial_state(),
                              uniform_source=lambda step, n: np.random.RandomState(1000 + step).random_sample(n),
                              inference_dtype=torch.bfloat16, eval_cache=cache, use_cuda_graph=graph, root_noise=noise,
                              forced_playouts=forced)
    batches = [b for _, b, _ in gen.iter_steps(max_steps=steps) if b is not None]
    eng = gen.search._engine
    rs = {k: v.cpu().numpy() for k, v in eng.root_stats().items()}
    st = eng.forced_stats()
    gen.search.close()
    return concat(batches), rs, st


@pytest.mark.gpu
def test_k0_is_off_with_resnet():
    torch.manual_seed(0)
    model = az.ResNet(num_res_blocks=4, num_channels=64).cuda()
    E, S, steps = 1024, 200, 12
    noise = az.RootNoise(alpha=1.0, fraction=0.25, seed=3)
    a = _net_selfplay(model, E, S, steps, None, noise=noise)
    b = _net_selfplay(model, E, S, steps, az.ForcedPlayouts(0.0), noise=noise)
    for f in EP_FIELDS:
        assert a[0][f].tobytes() == b[0][f].tobytes(), f
    for key in ROOT_KEYS:
        assert a[1][key].tobytes() == b[1][key].tobytes(), key


# ---- 2. policy targets ---------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("k", [2.0, 0.5])
def test_policy_targets_are_the_numpy_pruning(k):
    E, S = 16384, 200
    eng = Engine(E, S)
    eng.set_root_noise(0.3, 0.25, seed=11)
    eng.reset_games()
    eng.set_forced_playouts(k)
    eng.run_simulations(1, 2)
    eng.apply_root_noise()
    eng.run_simulations(S - 1, 2)
    rs = {key: v.cpu().numpy() for key, v in eng.root_stats().items()}
    got = eng.policy_targets().cpu().numpy()
    want = forced_oracle.prune_np(rs["child_N"], rs["child_W"], rs["child_P"], rs["legal"], rs["root_N"], 1.0, k)
    assert np.array_equal(got, want)
    assert (got != rs["child_N"]).any() and (rs["root_N"] == S).all()
    st = eng.forced_stats()
    assert st["forced_selections"] > 0 and st["forced_searches"] == 0 and st["visits_pruned"] == 0  # targets are a query
    eng.close()


# ---- 3. bit-exact self-play ----------------------------------------------------------------------------------------------------
CASES = [dict(kind=1, lanes=8), dict(kind=2, lanes=16, noise=True), dict(kind=2, lanes=32, noise=True, greedy=8),
         dict(kind=2, lanes=8, V=160), dict(kind=1, lanes=8, noise=True, cap=dict(fast=8, p=0.25, seed=21)),
         dict(kind=2, lanes=16, V=160, cap=dict(fast=8, p=0.3, seed=4, visit_budget=True)),
         dict(kind=2, lanes=32, V=160, noise=True, greedy=10, cap=dict(fast=6, p=0.5, seed=2))]


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES, ids=lambda c: "-".join(f"{k}{v if not isinstance(v, dict) else 'cap'}" for k, v in c.items()))
def test_selfplay_matches_forced_oracle(case):
    E, S, steps, k = 2048, 40, 40, 2.0
    kind, lanes, V, cap = case["kind"], case["lanes"], case.get("V", 0), case.get("cap")
    greedy = case.get("greedy")
    u = np.random.RandomState(5).random_sample((steps, E))
    nz = (0.3, 0.25, 77) if case.get("noise") else None
    got, flags, eta, st, _ = _selfplay(E, S, steps, kind, u, k, lanes=lanes, noise=nz, greedy=greedy, V=V, cap=cap)
    ref, extra = forced_oracle.selfplay_forced(E, S, k, u, full=flags, fast_sims=cap["fast"] if cap else None, V=V,
                                               visit_budget=bool(cap and cap.get("visit_budget")), eps=0.25 if nz else 0.0, eta=eta,
                                               greedy_from=-1 if greedy is None else greedy, quota=E * steps, eval_kind=kind)
    assert len(ref.ep_slot) > E // 2
    for f in EP_FIELDS:
        assert np.array_equal(got[f], getattr(ref, f)), f
    assert st["simulations"] == ref.n_sims
    for key in forced_oracle.FORCED_STATS:
        assert st[key] == extra[key], key
    assert extra["forced_selections"] > 0 and extra["visits_pruned"] > 0
    if V:
        assert extra["retained"] > 0


# ---- 4. network in the loop ----------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_resnet_cache_and_graph_change_nothing():
    torch.manual_seed(0)
    model = az.ResNet(num_res_blocks=4, num_channels=64).cuda()
    E, S, steps = 2048, 800, 12
    runs = [_net_selfplay(model, E, S, steps, az.ForcedPlayouts(2.0), cache, graph, az.RootNoise(1.0, 0.25, seed=4))
            for cache, graph in ((True, True), (False, True), (True, False))]
    a = runs[0]
    assert a[2]["forced_selections"] > 0 and a[2]["visits_pruned"] > 0
    for b in runs[1:]:
        for f in EP_FIELDS:
            assert np.array_equal(a[0][f], b[0][f]), f
        for key in ("child_N", "child_W", "child_P", "root_N"):
            assert np.array_equal(a[1][key], b[1][key]), key
        assert a[2] == b[2]


@pytest.mark.gpu
def test_resnet_trees_vs_forced_oracle():
    """The production loop (k_resnet_wide with compaction and the cache, CUDA graph on) over 2048 games x 800 simulations x 12 move
    steps with forced playouts, against the oracle fed the kernels' outputs on a sample of slots: the episodes they finished and
    the pruned counts of the last search."""
    E, S, steps, n_check, k = 2048, 800, 12, 12, 2.0
    torch.manual_seed(0)
    model = az.ResNet(num_res_blocks=4, num_channels=64)
    search = az.AlphaZeroSearch(model=model, num_simulations=S, inference_dtype=torch.bfloat16, forced_playouts=az.ForcedPlayouts(k))
    eng = search.engine_for(E, exact=True)
    eng.reset_games()
    u = np.random.RandomState(21).random_sample((steps, E))
    batches = []
    for step in range(steps):
        if step + 1 < steps:
            search.simulate_and_move(eng, torch.from_numpy(u[step]).to(eng.device))
            batches.append(eng.drain_episodes())
        else:
            search.simulate(eng)
            last = eng.policy_targets().cpu().numpy()
    got = concat(batches)
    idx = np.sort(np.random.RandomState(5).choice(E, n_check, replace=False))
    ref, extra = forced_oracle.selfplay_forced(n_check, S, k, u[:, idx], quota=n_check * steps, py_eval=KernelEvaluator(search._net))
    assert np.array_equal(last[idx], extra["last_counts"])
    assert (last[idx].sum(1) < S - 1).any()
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


# ---- 5. guards and integration -------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_guards():
    eng = Engine(64, 20)
    lib = eng.lib
    with pytest.raises(RuntimeError):
        eng.policy_targets()  # mode off
    for k in (-0.5, 1024.5, float("nan"), float("inf")):
        assert lib.az_set_forced_playouts(eng.h, C.byref(az._lib.AzForcedPlayouts(k))) == AZ_E_INVALID, k
    assert eng.forced_playouts is None
    eng.reset_games()
    eng.select_leaves()
    assert lib.az_set_forced_playouts(eng.h, C.byref(az._lib.AzForcedPlayouts(2.0))) == AZ_E_STATE
    assert lib.az_set_forced_playouts(eng.h, None) == AZ_E_STATE
    eng.expand_backup(torch.zeros((64, 7), device=eng.device), torch.zeros((64, 2), device=eng.device))
    eng.set_forced_playouts(1024.0)
    eng.set_forced_playouts(None)
    eng.close()
    with pytest.raises(ValueError):
        az.AlphaZeroPlayer(az.BasicNN(), forced_playouts=az.ForcedPlayouts())
    with pytest.raises(ValueError):
        az.elo_ladder({"a": az.BasicNN()}, az.Config(6, 7, 4).sample_initial_state(), forced_playouts=az.ForcedPlayouts())


@pytest.mark.gpu
@pytest.mark.parametrize("model_kind,cap", [("builtin", False), ("builtin", True), ("basic", False)])
def test_launches_per_move_step(model_kind, cap):
    E, S = 512, 48
    torch.manual_seed(0)
    if model_kind == "basic":
        model = az.BasicNN()
    else:
        from alphazero_implementation_b200.evaluators import HashEvaluator

        model = HashEvaluator()
    s = az.AlphaZeroSearch(model=model, num_simulations=S, use_cuda_graph=False, root_noise=az.RootNoise(0.3, 0.25),
                           playout_cap=az.PlayoutCap(8, 0.25, seed=1) if cap else None, forced_playouts=az.ForcedPlayouts(2.0))
    eng = s.engine_for(E, exact=True)
    eng.reset_games()
    u = torch.rand(E, dtype=torch.float64, device=eng.device)
    s.simulate_and_move(eng, u)
    for _ in range(2):
        n0 = eng.launch_count
        s.simulate_and_move(eng, u)
        assert eng.launch_count - n0 == s.launches_per_move_step()
    s.close()
