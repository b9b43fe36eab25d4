"""`Sample` / `Episode` containers with the reference's fields and JSON shape
(core/training/episode.py:9-71; file format of `episodes_iter{N}.json`, datamodule.py:71-80).
"""
from __future__ import annotations

import ast
from dataclasses import dataclass, field
from typing import Any

from .game import Action, State

ActionPolicy = dict  # dict[Action, float]   (models/base/prediction_types.py)
Value = list  # list[float], one entry per player


@dataclass
class Sample:
    state: State
    policy: ActionPolicy  # action -> MCTS visit probability
    value: Value  # game outcome [r_player0, r_player1]

    def to_dict(self) -> dict[str, Any]:
        return {
            "state": self.state.to_json(),
            "policy": {str(action.to_json()): prob for action, prob in self.policy.items()},
            "value": self.value,
        }

    @classmethod
    def from_dict(cls, data: dict[str, Any]) -> "Sample":
        state = State.from_json(data["state"])
        # the reference eval()s the key (episode.py:33); keys are `str({"column": c})`, a literal
        policy = {Action.from_json(ast.literal_eval(k), state): p for k, p in data["policy"].items()}
        return cls(state=state, policy=policy, value=data["value"])


@dataclass
class Episode:
    samples: list[Sample] = field(default_factory=list)

    def __len__(self) -> int:
        return len(self.samples)

    def add_sample(self, sample: Sample) -> None:
        self.samples.append(sample)

    def backpropagate_outcome(self, value: Value) -> None:
        for sample in self.samples:
            sample.value = value

    @property
    def current_state(self) -> State:
        return self.samples[-1].state

    def to_dict(self) -> dict[str, Any]:
        return {"samples": [s.to_dict() for s in self.samples]}

    @classmethod
    def from_dict(cls, data: dict[str, Any]) -> "Episode":
        ep = cls()
        ep.samples = [Sample.from_dict(d) for d in data["samples"]]
        return ep


def episodes_from_batch(batch, num_simulations: int) -> list[Episode]:
    """Materialise an `EpisodeBatch` (flat arrays from the device ring) as reference-style objects.

    policy[a] = child visits / (root visits - 1) as a Python float (int / int true division, node.py:27), where root visits - 1
    is the sample's count sum: S - 1 for a search on a fresh root (the first simulation expands the root, every later one passes
    through a child), N(c) + S - 1 on a root that kept its subtree (`AlphaZeroSearch(subtree_reuse=...)`).  `num_simulations` is
    kept for the signature; the row sum gives the same denominator for fresh roots.
    value = outcome list shared by every sample of the episode (episode.py:52-54).
    """
    from .game import DEFAULT_CONFIG, rules_engine

    out = []
    if len(batch) == 0:
        return out
    # State.actions of every sample position from the rules kernel, one call for the whole batch (an episode of a game whose
    # searches were all fast under `AlphaZeroSearch(playout_cap=)` has no samples: it is still an episode)
    legal_all = rules_engine().state_info(batch.s_bb0, batch.s_bb1)["legal"].cpu().numpy() if batch.num_samples else None
    for e in range(len(batch)):
        o, n = int(batch.ep_offset[e]), int(batch.ep_len[e])
        value = [float(batch.ep_outcome[e, 0]), float(batch.ep_outcome[e, 1])]
        ep = Episode()
        for i in range(o, o + n):
            counts = batch.s_counts[i]
            denom = int(counts.sum())
            bb0, bb1 = int(batch.s_bb0[i]), int(batch.s_bb1[i])
            legal = int(legal_all[i])
            st = State(DEFAULT_CONFIG, bb0, bb1, int(batch.s_player[i]), legal=legal, ended=False, reward=(0, 0))
            policy = {Action(st, c): int(counts[c]) / denom for c in range(7) if (legal >> c) & 1}
            ep.add_sample(Sample(state=st, policy=policy, value=value))
        out.append(ep)
    return out


def save_episodes(episodes: list[Episode], path: str) -> None:
    """`episodes_iter{N}.json` writer (DataModule.save_episodes, datamodule.py:71-80): a JSON list of `Episode.to_dict()`."""
    import json

    with open(path, "w") as f:
        json.dump([ep.to_dict() for ep in episodes], f)


def load_episodes(path: str) -> list[Episode]:
    """Reader for the same file (DataModule.load_episodes, datamodule.py:82-87)."""
    import json

    with open(path) as f:
        return [Episode.from_dict(d) for d in json.load(f)]
