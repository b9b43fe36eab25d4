"""Consumers of the search outside training (SURVEY §8 f4): the interactive player, an arena between two agents and the Elo
ladder over checkpoints.

  AlphaZeroPlayer.play(state) -> Action        ui/cli/player.py:42-76  (temperature 0 / t / inf move selection)
  play_game / Arena                            src/elo.ipynb#cell3, ui/cli/arena.py:39-57 (agent vs agent until `has_ended`)
  calculate_expected_score / update_elo / elo_ladder   src/elo.ipynb#cell1,#cell4

The single-position path is `AlphaZeroSearch.run(Node(state))` on the GPU engine with E = 1.  `Arena` is the batched form the
reference does not have: G games at once, both agents searching all positions that are theirs to move in ONE engine call per ply
(every game of a colour group is at the same ply, so one side moves in all of them), moves picked on the host from the root
visit counts with the reference's temperature rule.
"""
from __future__ import annotations

import random
from abc import ABC, abstractmethod
from collections import defaultdict
from itertools import combinations

import numpy as np

from .game import Action, State
from .openings import Openings, position_arrays
from .search import AlphaZeroSearch, Node


class Player(ABC):
    """Abstract base class of AI player (ui/cli/player.py:10-15)."""

    @abstractmethod
    def play(self, state: State) -> Action:
        pass


def _pick(counts: np.ndarray, legal: int, temperature: float, rng: random.Random) -> int:
    """The reference's move rule on root child visit counts (ui/cli/player.py:66-74): the policy is N_c / (N - 1); temperature 0
    takes the first maximum (`max` over the dict in action order), otherwise p ** (1 / t) renormalised and sampled."""
    cols = [c for c in range(7) if (legal >> c) & 1]
    if temperature == float("inf"):
        return rng.choice(cols)
    total = float(counts.sum())
    pol = [float(counts[c]) / total for c in cols]
    if temperature == 0:
        return cols[max(range(len(cols)), key=lambda i: pol[i])]
    probs = [p ** (1 / temperature) for p in pol]
    s = sum(probs)
    return rng.choices(cols, weights=[p / s for p in probs])[0]


class AlphaZeroPlayer(Player):
    """MCTS agent with the reference's constructor and temperature semantics (ui/cli/player.py:18-76).  The reference builds a new
    `AlphaZeroSearch` (a deep copy of the model) for every move; here the search - and its engine, packed weights and CUDA graph -
    is built once and kept.  (`agent.run` returns `(policy, value)`; the reference's `play` indexes that tuple as if it were the
    policy, ui/cli/player.py:64 - the intended behaviour is implemented.)  `search_kwargs` go to `AlphaZeroSearch` (for example
    `symmetric=True`), and an `Arena` plays through its agents' searches."""

    def __init__(self, model, *, mcts_simulation: int = 100, temperature: float = 1.0, **search_kwargs) -> None:
        if search_kwargs.get("forced_playouts") is not None:
            raise ValueError("forced_playouts is a self-play option: the player picks its move from the raw root visit counts, and "
                             "those of a forced search are not a move policy")
        self.model = model
        self.mcts_simulation = mcts_simulation
        self.temperature = temperature
        self._search_kwargs = search_kwargs
        self._search: AlphaZeroSearch | None = None
        self._rng = random.Random()

    @property
    def search(self) -> AlphaZeroSearch:
        if self._search is None:
            self._search = AlphaZeroSearch(model=self.model, num_simulations=self.mcts_simulation, **self._search_kwargs)
        return self._search

    def seed(self, s: int):
        self._rng.seed(s)

    def play(self, state: State) -> Action:
        if self.temperature == float("inf"):
            return self._rng.choice(state.actions)
        policy, _ = self.search.run(Node(state))
        if self.temperature == 0:
            return max(policy.items(), key=lambda x: x[1])[0]
        probs = [p ** (1 / self.temperature) for p in policy.values()]
        total = sum(probs)
        return self._rng.choices(list(policy.keys()), weights=[p / total for p in probs])[0]

    # batched: one engine call for all positions
    def play_many(self, bb0: np.ndarray, bb1: np.ndarray, player: np.ndarray) -> np.ndarray:
        """Columns for a batch of positions that are all this agent's to move."""
        n = len(bb0)
        eng = self.search.engine_for(n)
        eng.set_roots(bb0, bb1, player)
        if self.temperature == float("inf"):
            legal = eng.state_info(bb0, bb1)["legal"].cpu().numpy()
            return np.array([_pick(np.zeros(7), int(legal[i]), self.temperature, self._rng) for i in range(n)], np.uint8)
        self.search.simulate(eng)
        st = eng.root_stats()
        counts, legal = st["child_N"][:n].cpu().numpy(), st["legal"][:n].cpu().numpy()
        return np.array([_pick(counts[i], int(legal[i]), self.temperature, self._rng) for i in range(n)], np.uint8)


def play_game(agent1: Player, agent2: Player, initial_state: State) -> float:
    """One game, agent1 moving first (src/elo.ipynb#cell3).  Returns agent1's score: 1 win, 0.5 draw, 0 loss."""
    state = initial_state
    while not state.has_ended:
        state = (agent1 if state.player == 0 else agent2).play(state).sample_next_state()
    r = state.reward.tolist()
    return 0.5 if r[0] == r[1] else (1.0 if r[0] > r[1] else 0.0)


class Arena:
    """G games between two agents, all at once; half of them with agent A moving first, half with agent B.

    `openings` (optional): the games start from opening positions instead of `initial_state`, each opening played twice, once with
    A and once with B as the side to move at the opening - the standard remedy for deterministic agents (temperature 0), which
    otherwise play the same two games over and over.  A list of `State`s or a (bb0, bb1, player) array triple (for example from
    `distinct_openings`): games 2i and 2i + 1 of `play` start from opening i mod K; or an `Openings`: opening i is then the one
    `Engine.opening_positions` draws for slot i at move step 0 from `initial_state`."""

    def __init__(self, agent_a: AlphaZeroPlayer, agent_b: AlphaZeroPlayer, initial_state: State, openings=None):
        self.a, self.b, self.initial_state, self.openings = agent_a, agent_b, initial_state, openings

    def _starts(self, n: int) -> tuple[np.ndarray, np.ndarray, np.ndarray]:
        """the start positions of n colour-swapped pairs"""
        op = self.openings
        if isinstance(op, Openings):
            eng = self.a.search.engine_for(1)
            saved = eng.openings
            s0 = self.initial_state
            eng.set_openings(Openings(op.positions if op.positions is not None else [s0], op.min_plies, op.max_plies, op.seed, 0))
            o0, o1, pl = (t.cpu().numpy() for t in eng.opening_positions(op.slot_offset, n, 0))
            eng.set_openings(saved)
            return o0.view(np.uint64), o1.view(np.uint64), pl
        bb0, bb1, pl = position_arrays(op)
        if len(bb0) == 0:
            raise ValueError("Arena: empty opening set")
        idx = np.arange(n) % len(bb0)
        return bb0[idx], bb1[idx], pl[idx]

    def _play_group(self, first: AlphaZeroPlayer, second: AlphaZeroPlayer, n: int, starts=None) -> np.ndarray:
        """n games with `first` as player 0 from `initial_state` -> score of `first` per game.  `starts` = (bb0, bb1, player) of the
        n games: each starts there, with `first` as its side to move."""
        if starts is None:
            s0 = self.initial_state
            bb0, bb1, pl = np.full(n, s0.bb0, np.uint64), np.full(n, s0.bb1, np.uint64), np.full(n, s0.player, np.uint8)
            first_pl = np.zeros(n, np.uint8)
        else:
            bb0, bb1, pl = (np.array(x) for x in starts)
            first_pl = pl.copy()
        fill = bb0.copy(), bb1.copy(), pl.copy()
        score = np.full(n, np.nan)
        live = np.ones(n, bool)
        rules = first.search.engine_for(n)
        while live.any():
            i0 = int(np.argmax(live))
            mover = first if pl[i0] == first_pl[i0] else second  # every live game is at the same ply of its own start
            # the batch keeps its size (one engine, one captured graph per agent): finished games sit at their start position
            cols = mover.play_many(np.where(live, bb0, fill[0]), np.where(live, bb1, fill[1]), np.where(live, pl, fill[2]).astype(np.uint8))
            idx = np.nonzero(live)[0]
            nxt = {k: v.cpu().numpy() for k, v in rules.env_step(bb0[idx], bb1[idx], pl[idx], cols[idx]).items()}
            assert (nxt["status"] == 0).all()
            bb0[idx], bb1[idx], pl[idx] = nxt["bb0"].view(np.uint64), nxt["bb1"].view(np.uint64), nxt["player"]
            ended = nxt["ended"].astype(bool)
            r = nxt["reward"][ended]
            mine = r[np.arange(len(r)), first_pl[idx[ended]]]  # the reward of the side `first` played
            score[idx[ended]] = np.where(mine > 0, 1.0, np.where(mine < 0, 0.0, 0.5))
            live[idx[ended]] = False
        return score

    def play(self, num_games: int) -> dict:
        """-> wins / draws / losses of agent A and its mean score.  With openings, games 2i (A to move at the opening) and 2i + 1 (B)
        start from opening i and `scores` lists them in that order."""
        if self.openings is not None:
            k = (num_games + 1) // 2
            starts = self._starts(k)
            sa = self._play_group(self.a, self.b, k, starts)
            nb = num_games - k
            sb = 1.0 - self._play_group(self.b, self.a, nb, tuple(x[:nb] for x in starts)) if nb else np.zeros(0)
            s = np.empty(num_games)
            s[0::2], s[1::2] = sa, sb
        else:
            n1 = (num_games + 1) // 2
            sa = self._play_group(self.a, self.b, n1)
            sb = 1.0 - self._play_group(self.b, self.a, num_games - n1) if num_games > n1 else np.zeros(0)
            s = np.concatenate([sa, sb])
        return dict(games=num_games, a_wins=int((s == 1).sum()), draws=int((s == 0.5).sum()), b_wins=int((s == 0).sum()),
                    a_score=float(s.mean()), scores=s)


# ---- Elo (src/elo.ipynb#cell1) -------------------------------------------------------------------------------------------
def calculate_expected_score(rating1: float, rating2: float) -> float:
    """Expected score of player 1 against player 2."""
    return 1 / (1 + 10 ** ((rating2 - rating1) / 400))


def update_elo(rating1: int, rating2: int, score: float, K: int = 32) -> tuple[int, int]:
    """Ratings after one game; score: 1 win, 0.5 draw, 0 loss from rating1's side.  Truncated to int like the notebook."""
    expected = calculate_expected_score(rating1, rating2)
    new1 = rating1 + K * (score - expected)
    new2 = rating2 + K * ((1 - score) - (1 - expected))
    return int(new1), int(new2)


def elo_ladder(models: dict, initial_state: State, games_per_pair: int = 2, mcts_simulation: int = 100, temperature: float = 0,
               K: int = 32, openings=None, **search_kwargs) -> dict:
    """Round robin over named models / checkpoints (src/elo.ipynb#cell4), every pairing played as a batched `Arena`, ratings
    updated game by game from 1500.  `openings`: every pairing plays from these opening positions, each twice with the colours
    swapped (`Arena(openings=)`): at temperature 0 the games are otherwise the same two games repeated."""
    ratings: dict = defaultdict(lambda: 1500)
    if search_kwargs.get("forced_playouts") is not None:
        raise ValueError("forced_playouts is a self-play option: the ladder's players pick their moves from raw root visit counts")
    players = {name: AlphaZeroPlayer(m, mcts_simulation=mcts_simulation, temperature=temperature, **search_kwargs) for name, m in models.items()}
    for n1, n2 in combinations(list(models), 2):
        res = Arena(players[n1], players[n2], initial_state, openings).play(games_per_pair)
        for s in res["scores"]:
            ratings[n1], ratings[n2] = update_elo(ratings[n1], ratings[n2], float(s), K)
    return {name: ratings[name] for name in models}
