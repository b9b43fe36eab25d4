"""Opening positions (az_set_openings: k_openings and k_check_openings).  az_opening_positions is the C oracle bit for bit; after
reset_games every root is its step-0 opening; self-play with the mode on is bit-exact against tests/native/c4_openings_oracle.c on
the built-in evaluators, also with noise, subtree reuse, the playout cap or forced playouts; a game's first sample is its opening;
sharded engines draw what one engine draws; the mode off (or set and cleared) changes nothing; the guards hold; an arena of two
equal agents at temperature 0 over distinct openings scores exactly 0.5 with distinct games; ResNet 4x64 in the loop with the cache
and the CUDA graph changes no bit against the un-graphed run."""
import ctypes as C

import numpy as np
import pytest
import torch

import alphazero_implementation_b200 as az
from alphazero_implementation_b200.engine import Engine
import openings_oracle as oo
from test_gpu_playout_cap import EP_FIELDS, budgets, concat

AZ_E_INVALID, AZ_E_STATE = -1, -4
SET = (np.array([0, 1 << 21, 0, 0b11], np.uint64), np.array([0, 1 << 14, 1 << 21, 1 << 7], np.uint64), np.array([0, 0, 0, 1], np.uint8))
INIT = (1 << 21, 1 << 28, 0)


def _host(t3):
    o0, o1, pl = (t.cpu().numpy() for t in t3)
    return o0.view(np.uint64), o1.view(np.uint64), pl


# ---- 1. the query is the oracle ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("positions,lo,hi", [(None, 0, 8), (SET, 2, 6), (None, 30, 40), (SET, 0, 0)])
def test_opening_positions_are_the_oracle(positions, lo, hi):
    n, first = 16384, (1 << 33) + 12345
    eng = Engine(64, 4)
    eng.reset_games(*INIT)
    eng.set_openings(az.Openings(positions, lo, hi, seed=2**64 - 77))
    for step in (0, 1, 977, 2**32 - 1):
        got = _host(eng.opening_positions(first, n, step))
        want = oo.openings_c(first, n, step, positions=positions, min_plies=lo, max_plies=hi, seed=2**64 - 77, init=INIT)
        for a, b in zip(got, want):
            assert np.array_equal(a, b), step
    assert len(set(zip(got[0].tolist(), got[1].tolist()))) > (1 if hi == 0 else 1000)
    eng.close()


# ---- 2. reset_games --------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_reset_games_starts_every_game_from_its_step0_opening():
    E, off = 4096, 512
    eng = Engine(E, 8)
    eng.set_openings(az.Openings(SET, 1, 5, seed=9, slot_offset=off))
    eng.reset_games()
    eng.select_leaves()  # a fresh root is its own leaf
    info = {k: v.cpu().numpy() for k, v in eng.leaf_info().items()}
    eng.expand_backup(torch.zeros((E, 7), device=eng.device), torch.zeros((E, 2), device=eng.device))
    want = oo.openings_c(off, E, 0, positions=SET, min_plies=1, max_plies=5, seed=9)
    assert np.array_equal(info["bb0"].view(np.uint64), want[0]) and np.array_equal(info["bb1"].view(np.uint64), want[1])
    assert np.array_equal(info["player"], want[2])
    assert np.array_equal(_host(eng.opening_positions(off, E, 0))[0], want[0])
    eng.close()


# ---- 3. bit-exact self-play ----------------------------------------------------------------------------------------------------
def _selfplay(E, S, steps, kind, u, openings, lanes=0, noise=None, V=0, cap=None, k=None, greedy=None, slot_offset=0, fused=True):
    """the engine's self-play loop -> (episodes, cap flags [steps, E] or None, eta [steps, E, 7] or None, stats)"""
    eng = Engine(E, S, lanes_per_tree=lanes)
    if V:
        eng.set_subtree_reuse(V)
    eng.set_greedy_from(greedy)
    if noise is not None:
        eng.set_root_noise(noise[0], noise[1], seed=noise[2], slot_offset=slot_offset)
    eng.set_openings(openings)
    eng.reset_games()
    if cap is not None:
        eng.set_playout_cap(cap["fast"], cap["p"], cap["seed"], slot_offset)
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
        elif fused:
            eng.run_move_step(S, kind, ud)
        else:
            eng.run_simulations(S, kind)
            eng.sample_moves(ud)
        batches.append(eng.drain_episodes())
    st = eng.stats()
    eng.close()
    return concat(batches), (np.stack(flags) if flags else None), (np.stack(etas) if etas else None), st


CASES = [dict(kind=1, lanes=8), dict(kind=2, lanes=16), dict(kind=2, lanes=32, noise=True), dict(kind=2, lanes=8, V=160),
         dict(kind=1, lanes=8, cap=dict(fast=8, p=0.25, seed=21)), dict(kind=2, lanes=16, k=2.0), dict(kind=2, lanes=8, greedy=4)]
OPEN = dict(positions=SET, min_plies=0, max_plies=6, seed=31)


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES, ids=lambda c: "-".join(f"{k}{v if not isinstance(v, dict) else 'cap'}" for k, v in c.items()))
def test_selfplay_matches_openings_oracle(case):
    E, S, steps = 2048, 40, 40
    kind, cap = case["kind"], case.get("cap")
    u = np.random.RandomState(5).random_sample((steps, E))
    nz = (0.3, 0.25, 77) if case.get("noise") else None
    got, flags, eta, st = _selfplay(E, S, steps, kind, u, az.Openings(**OPEN), lanes=case["lanes"], noise=nz, V=case.get("V", 0),
                                    cap=cap, k=case.get("k"), greedy=case.get("greedy"))
    ref, extra = oo.selfplay_openings(E, S, u, **OPEN, k=case.get("k") or 0.0, full=flags, fast_sims=cap["fast"] if cap else None,
                                      V=case.get("V", 0), eps=0.25 if nz else 0.0, eta=eta, quota=E * steps, eval_kind=kind,
                                      greedy_from=-1 if case.get("greedy") is None else case["greedy"])
    assert len(ref.ep_slot) > E
    for f in EP_FIELDS:
        assert np.array_equal(got[f], getattr(ref, f)), f
    assert st["simulations"] == ref.n_sims


# ---- 4. the first sample is the opening ----------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_first_sample_is_the_opening():
    E, S, steps, off = 4096, 32, 40, 3 * 2**40
    u = np.random.RandomState(6).random_sample((steps, E))
    op = az.Openings(None, 0, 8, seed=12, slot_offset=off)
    got, _, _, _ = _selfplay(E, S, steps, 2, u, op, fused=False)
    eng = Engine(64, 4)
    eng.set_openings(op)
    start = np.cumsum(got["ep_len"]) - got["ep_len"]
    s0 = got["ep_step"] - got["ep_len"] + 1
    assert len(start) > E and (s0 > 0).any()
    for s in np.unique(s0):
        sel = np.nonzero(s0 == s)[0]
        o0, o1, pl = _host(eng.opening_positions(off, E, int(s)))
        slots = got["ep_slot"][sel]
        assert np.array_equal(got["s_bb0"][start[sel]], o0[slots]) and np.array_equal(got["s_bb1"][start[sel]], o1[slots])
        assert np.array_equal(got["s_player"][start[sel]], pl[slots])
    eng.close()


# ---- 5. sharding -----------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_sharded_engines_draw_the_unsharded_games():
    E, S, steps = 2048, 32, 30
    u = np.random.RandomState(1).random_sample((steps, E))
    whole, _, _, _ = _selfplay(E, S, steps, 2, u, az.Openings(SET, 1, 4, seed=5))
    h = E // 2
    parts = [_selfplay(h, S, steps, 2, u[:, o:o + h], az.Openings(SET, 1, 4, seed=5, slot_offset=o))[0] for o in (0, h)]
    for part, off in zip(parts, (0, h)):
        sel = (whole["ep_slot"] >= off) & (whole["ep_slot"] < off + h)
        assert np.array_equal(whole["ep_slot"][sel] - off, part["ep_slot"])
        for f in ("ep_step", "ep_len", "ep_outcome"):
            assert np.array_equal(whole[f][sel], part[f]), f
        st = np.cumsum(whole["ep_len"]) - whole["ep_len"]
        rows = np.concatenate([np.arange(a, a + n) for a, n in zip(st[sel], whole["ep_len"][sel])])
        for f in ("s_bb0", "s_bb1", "s_player", "s_counts"):
            assert np.array_equal(whole[f][rows], part[f]), f


# ---- 6. off is off ---------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("kind", [1, 2])
def test_off_and_cleared_are_never_set(kind):
    E, S, steps = 2048, 40, 40
    u = np.random.RandomState(2).random_sample((steps, E))
    ref, _, _, st_ref = _selfplay(E, S, steps, kind, u, None)

    eng = Engine(E, S)
    eng.set_openings(az.Openings(SET, 2, 6, seed=1))
    eng.set_openings(None)
    eng.reset_games()
    batches = []
    for step in range(steps):
        eng.run_move_step(S, kind, torch.from_numpy(u[step]).to(eng.device))
        batches.append(eng.drain_episodes())
    got = concat(batches)
    for f in EP_FIELDS:
        assert ref[f].tobytes() == got[f].tobytes(), f
    assert eng.stats() == st_ref
    eng.close()


# ---- 7. guards -------------------------------------------------------------------------------------------------------------------
def _cfg(eng, bb0, bb1, pl, lo=0, hi=2, off=0):
    keep = [eng._dev(np.array(bb0, np.uint64), torch.int64), eng._dev(np.array(bb1, np.uint64), torch.int64),
            eng._dev(np.array(pl, np.uint8), torch.uint8)]
    return az._lib.AzOpenings(*(t.data_ptr() for t in keep), len(bb0), lo, hi, 0, off), keep


@pytest.mark.gpu
def test_guards():
    eng = Engine(64, 20)
    lib = eng.lib
    with pytest.raises(RuntimeError):
        eng.opening_positions(0, 4, 0)  # mode off
    four = 0b1111  # four in column 0
    full0, full1 = 0xD1A0B1665334, 0x2C5B46898C8B  # a drawn full board
    bad = {"the boards overlap": (1, 1, 0), "off the board": (1 << 6, 0, 0), "above an empty cell": (0b10, 0, 0),
           "player is not 0 or 1": (0, 0, 2), "the game has ended": (four, 0, 0)}
    bad_full = (full0, full1, 0)
    for why, (b0, b1, p) in list(bad.items()) + [("the game has ended", bad_full)]:
        cfg, keep = _cfg(eng, [0, 1, b0], [0, 0, b1], [0, 1, p])
        assert lib.az_set_openings(eng.h, C.byref(cfg)) == AZ_E_INVALID, why
        msg = lib.az_last_error(eng.h).decode()
        assert "position 2" in msg and why in msg, msg
    for lo, hi, off in ((-1, 2, 0), (3, 2, 0), (0, 41, 0), (0, 2, -1), (0, 2, 2**62 + 1)):
        cfg, keep = _cfg(eng, [0], [0], [0], lo, hi, off)
        assert lib.az_set_openings(eng.h, C.byref(cfg)) == AZ_E_INVALID, (lo, hi, off)
    cfg = az._lib.AzOpenings(None, None, None, 3, 0, 2, 0, 0)
    assert lib.az_set_openings(eng.h, C.byref(cfg)) == AZ_E_INVALID
    cfg = az._lib.AzOpenings(None, None, None, -1, 0, 2, 0, 0)
    assert lib.az_set_openings(eng.h, C.byref(cfg)) == AZ_E_INVALID
    assert eng.openings is None
    with pytest.raises(RuntimeError):
        eng.opening_positions(0, 4, 0)  # still off after the failed calls
    eng.reset_games()
    eng.select_leaves()
    cfg, keep = _cfg(eng, [0], [0], [0])
    assert lib.az_set_openings(eng.h, C.byref(cfg)) == AZ_E_STATE
    assert lib.az_set_openings(eng.h, None) == AZ_E_STATE
    eng.expand_backup(torch.zeros((64, 7), device=eng.device), torch.zeros((64, 2), device=eng.device))
    eng.set_openings(az.Openings(min_plies=40, max_plies=40, slot_offset=2**62))
    eng.set_openings(az.Openings([az.Config(6, 7, 4).sample_initial_state()], 0, 3))
    assert len(eng.opening_positions(0, 5, 0)[0]) == 5
    eng.set_openings(None)
    eng.close()


# ---- 8. arena --------------------------------------------------------------------------------------------------------------------
def _recorded(agent, log):
    inner = agent.play_many

    def play_many(bb0, bb1, player):
        log.append((np.array(bb0), np.array(bb1)))
        return inner(bb0, bb1, player)

    agent.play_many = play_many
    return agent


def _games(log_a, log_b, n):
    """per game of the two colour groups: (group, the positions it went through)"""
    return [tuple((int(b0[i]), int(b1[i])) for b0, b1 in log) for log in (log_a, log_b) for i in range(n)]


@pytest.mark.gpu
def test_arena_of_equal_agents_over_distinct_openings():
    K = 24
    init = az.Config(6, 7, 4).sample_initial_state()
    ops = az.distinct_openings(K, 4, seed=3)
    assert len(set(zip(ops[0].tolist(), ops[1].tolist()))) == K

    def run(openings):
        a = az.AlphaZeroPlayer(az.HashEvaluator(), mcts_simulation=64, temperature=0)
        b = az.AlphaZeroPlayer(az.HashEvaluator(), mcts_simulation=64, temperature=0)
        logs = []
        arena = az.Arena(a, b, init, openings)
        group = arena._play_group

        def play_group(first, second, n, starts=None):  # one log per colour group, in the order play() runs them
            log = []
            _recorded(first, log)
            _recorded(second, log)
            try:
                return group(first, second, n, starts)
            finally:
                del first.play_many, second.play_many
                logs.append(log)

        arena._play_group = play_group
        res = arena.play(2 * K)
        return res, logs

    res, logs = run(ops)
    assert res["a_score"] == 0.5
    s = res["scores"]
    assert np.array_equal(s[0::2] + s[1::2], np.ones(K))  # each pair: the same game with the roles exchanged
    ga, gb = _games(logs[0], logs[1], K)[:K], _games(logs[0], logs[1], K)[K:]
    assert ga == gb
    assert len(set(ga)) == K  # 2K games: K distinct sequences, each once with A and once with B to move at the opening
    res0, logs0 = run(None)
    games0 = _games(logs0[0], logs0[1], K)
    assert len(set(games0[:K])) == 1 and len(set(games0[K:])) == 1


# ---- 9. network in the loop ------------------------------------------------------------------------------------------------------
def _net_selfplay(model, E, S, steps, openings, graph):
    gen = az.EpisodeGenerator(model=model, num_simulations=S, num_episodes=E, game_initial_state=az.Config(6, 7, 4).sample_initial_state(),
                              uniform_source=lambda step, n: np.random.RandomState(1000 + step).random_sample(n),
                              inference_dtype=torch.bfloat16, eval_cache=True, use_cuda_graph=graph, openings=openings)
    batches = [b for _, b, _ in gen.iter_steps(max_steps=steps) if b is not None]
    eng = gen.search._engine
    rs = {k: v.cpu().numpy() for k, v in eng.root_stats().items()}
    st = eng.eval_cache_stats()
    gen.search.close()
    return concat(batches), rs, st


@pytest.mark.gpu
def test_resnet_cache_and_graph_change_nothing():
    torch.manual_seed(0)
    model = az.ResNet(num_res_blocks=4, num_channels=64).cuda()
    E, S, steps = 1024, 200, 16
    op = az.Openings(None, 0, 4, seed=8)
    a = _net_selfplay(model, E, S, steps, op, True)
    b = _net_selfplay(model, E, S, steps, op, False)
    assert len(a[0]["ep_slot"]) > 0 and a[2]["hits"] > 0
    for f in EP_FIELDS:
        assert np.array_equal(a[0][f], b[0][f]), f
    for key in ("child_N", "child_W", "child_P", "root_N"):
        assert np.array_equal(a[1][key], b[1][key]), key


@pytest.mark.gpu
@pytest.mark.parametrize("model_kind", ["builtin", "basic"])
def test_launches_per_move_step(model_kind):
    E, S = 512, 48
    torch.manual_seed(0)
    model = az.BasicNN() if model_kind == "basic" else az.HashEvaluator()
    s = az.AlphaZeroSearch(model=model, num_simulations=S, use_cuda_graph=False)
    eng = s.engine_for(E, exact=True)
    eng.set_openings(az.Openings(None, 0, 4))
    eng.reset_games()
    u = torch.rand(E, dtype=torch.float64, device=eng.device)
    s.simulate_and_move(eng, u)
    for _ in range(2):
        n0 = eng.launch_count
        s.simulate_and_move(eng, u)
        assert eng.launch_count - n0 == s.launches_per_move_step()
    s.close()
