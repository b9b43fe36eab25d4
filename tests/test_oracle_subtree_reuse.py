"""CPU: the reuse oracle's entry points (tests/native/c4_reuse_oracle.c: c4o_advance_reuse, c4o_selfplay_reuse) - the yardstick the
GPU tests of the library's subtree reuse hold it against - and the policy targets of reused roots.  max_root_visits V = S never
retains a subtree, so it is c4o_selfplay_noise bit for bit; a retained tree is exactly the played child's subtree; trees stay within
1 + 7 V nodes; policy targets divide by each row's count sum, which is S - 1 for fresh roots."""
import numpy as np
import pytest
import torch

import noise_oracle
import reuse_oracle

FIELDS = ("ep_slot", "ep_len", "ep_step", "ep_outcome", "s_bb0", "s_bb1", "s_player", "s_counts")


def legal_cols(b0, b1):
    occ = int(b0) | int(b1)
    return [c for c in range(7) if not (occ >> (7 * c + 5)) & 1]


def play(b0, b1, pl, c):
    occ = int(b0) | int(b1)
    col = occ >> (7 * c) & 0x7F
    bit = ((col + 1) & ~col) << (7 * c)
    return (int(b0) | bit, int(b1), 1) if pl == 0 else (int(b0), int(b1) | bit, 0)


def walk(tree, k, b0, b1, pl, idx=0, path=()):
    """{column path: (N, W bits, P bits)} of the subtree of node idx of exported tree k; children found by the legal columns"""
    out = {path: (int(tree["N"][k, idx]), tree["W"][k, idx].tobytes(), tree["P"][k, idx].tobytes())}
    cb = int(tree["first_child"][k, idx])
    if cb:
        for j, c in enumerate(legal_cols(b0, b1)):
            out.update(walk(tree, k, *play(b0, b1, pl, c), cb + j, path + (c,)))
    return out


def random_positions(oracle, n, plies, seed):
    rng = np.random.RandomState(seed)
    b0 = np.zeros(n, np.uint64); b1 = np.zeros(n, np.uint64); pl = np.zeros(n, np.uint8)
    for _ in range(plies):
        info = oracle.state_info(b0, b1, pl)
        live = (info["ended"] == 0) & (info["legal"] != 0)
        col = np.array([rng.choice([c for c in range(7) if (m >> c) & 1]) if ok else 0 for m, ok in zip(info["legal"], live)], np.uint8)
        nxt = oracle.env_step(b0, b1, pl, col)
        ok = live & (nxt["ended"] == 0)
        b0 = np.where(ok, nxt["bb0"], b0); b1 = np.where(ok, nxt["bb1"], b1); pl = np.where(ok, nxt["player"], pl)
    return b0, b1, pl


@pytest.mark.parametrize("eval_kind", [1, 2])
@pytest.mark.parametrize("noise,greedy_from", [(False, -1), (True, -1), (True, 9)])
def test_v_equal_s_is_selfplay_noise(oracle, eval_kind, noise, greedy_from):
    E, S, steps = 48, 40, 70
    u = np.random.RandomState(3).random_sample((steps, E))
    eta = np.random.RandomState(4).dirichlet(np.ones(7), size=(steps, E)).astype(np.float32)
    eps = 0.25 if noise else 0.0
    ref = noise_oracle.selfplay_noise(E, S, u, eps, eta if noise else np.zeros((steps, E, 7), np.float32), greedy_from=greedy_from,
                                      eval_kind=eval_kind)
    got, st = reuse_oracle.selfplay_reuse(E, S, S, u, eps, eta if noise else None, greedy_from=greedy_from, eval_kind=eval_kind)
    for f in FIELDS:
        assert np.array_equal(getattr(ref, f), getattr(got, f)), f
    for f in ("n_steps", "n_uniforms_used", "n_sims", "n_evals"):
        assert getattr(ref, f) == getattr(got, f), f
    assert st["retained"] == 0 and st["fresh"] + st["dropped"] > 0


@pytest.mark.parametrize("eval_kind", [1, 2])
def test_reroot_keeps_the_played_subtree(oracle, eval_kind):
    E, S, V = 64, 60, 240
    b0, b1, pl = random_positions(oracle, E, 6, seed=11)
    rng = np.random.RandomState(5)
    # the trees before the move: every column illegal (7) leaves them untouched
    before = reuse_oracle.advance_reuse(b0, b1, pl, S, np.full(E, 7, np.uint8), S, V, eval_kind=eval_kind)
    assert (before["status"] == 1).all()
    cols = np.array([rng.choice(legal_cols(b0[i], b1[i])) for i in range(E)], np.uint8)
    after = reuse_oracle.advance_reuse(b0, b1, pl, S, cols, S, V, eval_kind=eval_kind)
    assert (after["status"] == 0).all()
    retained = 0
    for i in range(E):
        full = walk(before, i, b0[i], b1[i], int(pl[i]))
        c = int(cols[i])
        nb = play(b0[i], b1[i], int(pl[i]), c)
        sub = {p[1:]: v for p, v in full.items() if p[:1] == (c,)}
        got = walk(after, i, *nb)
        if after["used"][i] == 1 and after["first_child"][i, 0] == 0:  # fresh or dropped
            assert got == {(): (0, np.float64(0).tobytes(), np.float32(0).tobytes())}
            n_c = sub[()][0]
            assert len(sub) == 1 or n_c + S > V
            continue
        retained += 1
        assert sub[()][0] + S <= V
        root = sub.pop(())
        g_root = got.pop(())
        assert g_root == (root[0], root[1], np.float32(0).tobytes())  # N(c), W(c) kept, prior 0
        assert got == sub
        assert after["used"][i] == len(got) + 1  # every retained node is reachable, nothing else
        # children blocks are contiguous and lie above their parent
        cb = after["first_child"][i, :after["used"][i]]
        assert (cb[cb != 0] > np.nonzero(cb)[0]).all()
    assert retained > E // 2
    st = after["stats"]
    ended = int(oracle.env_step(b0, b1, pl, cols)["ended"].sum())  # recycled, not counted
    assert st["retained"] == retained and st["retained"] + st["fresh"] + st["dropped"] == E - ended


@pytest.mark.parametrize("V_mult", [1, 2, 4])
def test_trees_stay_within_the_bound(oracle, V_mult):
    E, S, steps = 32, 50, 60
    V = V_mult * S
    u = np.random.RandomState(7).random_sample((steps, E))
    got, st = reuse_oracle.selfplay_reuse(E, S, V, u, eval_kind=2, greedy_from=6)
    assert 1 < st["max_used"] <= 1 + 7 * V
    if V_mult > 1:
        assert st["retained"] > 0 and st["visits"] >= st["retained"]
    # a root that kept its subtree holds N(c) + S visits: the sample's counts sum to more than S - 1, never to more than V - 1
    sums = got.s_counts.sum(1)
    assert sums.min() == S - 1 and sums.max() <= V - 1
    assert (sums > S - 1).any() == (V_mult > 1)


class _Rules:
    def state_info(self, bb0, bb1):
        occ = np.asarray(bb0, np.uint64) | np.asarray(bb1, np.uint64)
        legal = sum(((((occ >> np.uint64(7 * c + 5)) & np.uint64(1)) == 0).astype(np.uint8) << c) for c in range(7))
        return {"legal": torch.from_numpy(legal.astype(np.uint8))}


def _batch(oracle, S, V):
    from alphazero_implementation_b200.engine import EpisodeBatch

    E, steps = 16, 60
    u = np.random.RandomState(1).random_sample((steps, E))
    r, _ = reuse_oracle.selfplay_reuse(E, S, V, u, eval_kind=2)
    off = (np.cumsum(r.ep_len) - r.ep_len).astype(np.int64)
    return EpisodeBatch(r.ep_slot, r.ep_step, r.ep_len, off, r.ep_outcome, r.s_bb0, r.s_bb1, r.s_player, r.s_counts)


def test_episode_targets(oracle, monkeypatch):
    from alphazero_implementation_b200 import game
    from alphazero_implementation_b200.episode import episodes_from_batch

    monkeypatch.setattr(game, "rules_engine", lambda: _Rules())
    S = 30
    fresh = _batch(oracle, S, S)
    for ep, o, n in zip(episodes_from_batch(fresh, S), fresh.ep_offset, fresh.ep_len):
        for k, smp in enumerate(ep.samples):
            counts = fresh.s_counts[o + k]
            assert {a.column: p for a, p in smp.policy.items()} == {c: int(counts[c]) / (S - 1) for c in range(7)
                                                                   if (smp.state.legal_mask >> c) & 1}
    reused = _batch(oracle, S, 4 * S)
    assert (reused.s_counts.sum(1) > S - 1).any()
    for ep in episodes_from_batch(reused, S):
        for smp in ep.samples:
            assert abs(sum(smp.policy.values()) - 1.0) < 1e-12


def test_replay_targets(oracle):
    from alphazero_implementation_b200.replay import ReplayBuffer

    S = 30
    for V in (S, 4 * S):
        b = _batch(oracle, S, V)
        counts = torch.from_numpy(b.s_counts).to(torch.float32)
        policy = {}
        for reuse in (False, True):
            rb = ReplayBuffer(10**6, S, "cpu", subtree_reuse=reuse)
            rb.extend(b)
            policy[reuse] = rb.tensors()[3]
        if V == S:
            for reuse in (False, True):  # the targets before subtree reuse existed
                assert torch.equal(policy[reuse], counts / float(S - 1))
        else:
            assert (counts.sum(1) > S - 1).any()
            assert torch.allclose(policy[True].sum(1), torch.ones(policy[True].shape[0]), atol=1e-6)
