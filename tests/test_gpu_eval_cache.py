"""The evaluation cache of the network-in-the-loop path (az_set_eval_cache) changes no result bit: self-play with the cache on
and off gives the same episodes, root statistics and counters - across a weights update (epoch bump) and with a table so small
that entries are evicted all the time - while the evaluator computes fewer rows."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

E, S, STEPS = 2048, 800, 12


def _model(seed):
    import alphazero_implementation_b200 as az

    torch.manual_seed(seed)
    m = az.ResNet(num_res_blocks=4, num_channels=64)
    with torch.no_grad():  # a non-trivial net: random BatchNorm statistics, so that priors and values differ between positions
        for mod in m.modules():
            if isinstance(mod, torch.nn.BatchNorm2d):
                mod.running_mean.uniform_(-0.5, 0.5)
                mod.running_var.uniform_(0.5, 2.0)
    return m.eval()


def _selfplay(cache, update_at=None):
    """STEPS move steps of E games; per step the root statistics after the search and the finished episodes."""
    import alphazero_implementation_b200 as az

    search = az.AlphaZeroSearch(model=_model(0), num_simulations=S, inference_dtype=torch.bfloat16, eval_cache=cache)
    eng = search.engine_for(E, exact=True)
    eng.reset_games()
    u = torch.from_numpy(np.random.RandomState(5).random_sample((STEPS, E))).cuda()
    roots, episodes = [], []
    for step in range(STEPS):
        if step == update_at:
            search.update_inference_model(_model(1))
        search.simulate(eng)
        roots.append({k: v.cpu().numpy() for k, v in eng.root_stats().items()})
        eng.sample_moves(u[step])
        b = eng.drain_episodes()
        episodes.append({f: np.asarray(getattr(b, f)).copy() for f in ("ep_slot", "ep_step", "ep_len", "ep_outcome", "s_bb0", "s_bb1", "s_player", "s_counts")})
    out = dict(roots=roots, episodes=episodes, stats=eng.stats(), cache=eng.eval_cache_stats(), log2=eng.eval_cache_log2,
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


@pytest.fixture(scope="module")
def uncached():
    return _selfplay(False)


def test_cache_changes_no_result_and_saves_rows(uncached):
    on = _selfplay(True)
    assert on["kernel"] == "k_resnet_wide" and on["log2"] > 0 and uncached["log2"] == 0
    _assert_same(uncached, on)
    c = on["cache"]
    assert c["hits"] > 0 and c["followers"] > 0
    assert c["rows"] + c["hits"] + c["followers"] == on["stats"]["evaluations"]
    assert c["rows"] < on["stats"]["evaluations"] // 2
    off = uncached["cache"]
    assert off["hits"] == off["followers"] == 0 and off["rows"] == uncached["stats"]["evaluations"]


def test_weights_update_bumps_the_epoch():
    off, on = _selfplay(False, update_at=STEPS // 2), _selfplay(True, update_at=STEPS // 2)
    _assert_same(off, on)
    assert on["cache"]["hits"] > 0


def test_tiny_table_with_constant_eviction(uncached):
    on = _selfplay(10)
    assert on["log2"] == 10
    _assert_same(uncached, on)
    assert on["cache"]["evictions"] > 0 and on["cache"]["failed_claims"] > 0
