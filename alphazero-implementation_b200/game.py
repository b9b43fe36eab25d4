"""Game-state interface of the reference (`simulator.game.connect` Config / State / Action, as used at the
call sites listed in SURVEY.md Appendix B) backed by the CUDA rules kernels.

Every rule (legal moves, play, has_ended, reward) is evaluated by `az_env_step` / `az_state_info`;
this module only formats results.  A `State` is immutable: two bitboards + side to move, plus the
rule results cached from the kernel that produced it.
"""
from __future__ import annotations

import numpy as np

HEIGHT, WIDTH, COUNT = 6, 7, 4

_rules_engine = None


def rules_engine():
    """Small shared engine used for stand-alone rule queries at the API edge."""
    global _rules_engine
    if _rules_engine is None:
        from .engine import Engine

        _rules_engine = Engine(num_games=1, num_simulations=1)
    return _rules_engine


def grid_to_bitboards(grid) -> tuple[int, int]:
    """grid[row][col] in {-1, 0, 1}, row 0 = bottom -> (bb0, bb1), bit = col*7 + row."""
    g = np.asarray(grid)
    bb = [0, 0]
    for r in range(g.shape[0]):
        for c in range(g.shape[1]):
            v = int(g[r, c])
            if v >= 0:
                bb[v] |= 1 << (c * 7 + r)
    return bb[0], bb[1]


def bitboards_to_grid(bb0: int, bb1: int) -> np.ndarray:
    g = np.full((HEIGHT, WIDTH), -1, dtype=np.int8)
    for c in range(WIDTH):
        for r in range(HEIGHT):
            b = 1 << (c * 7 + r)
            if bb0 & b:
                g[r, c] = 0
            elif bb1 & b:
                g[r, c] = 1
    return g


_COL = np.uint64(0x7F)


def _mirror(b: np.ndarray) -> np.ndarray:
    out = b & (_COL << np.uint64(21))
    for c in range(3):  # columns c and 6 - c trade places; column 3 stays
        s, lo = np.uint64(7 * (6 - 2 * c)), _COL << np.uint64(7 * c)
        out |= ((b & lo) << s) | ((b >> s) & lo)
    return out


def mirror_bitboards(bb0, bb1) -> tuple[np.ndarray, np.ndarray]:
    """Left-right mirror of positions (what `az_mirror_states` computes on the device): column c's 7 bits (bit 7c + r) move to
    column 6 - c, in both bitboards; the side to move does not change."""
    return _mirror(np.asarray(bb0, np.uint64)), _mirror(np.asarray(bb1, np.uint64))


def canonical_bitboards(bb0, bb1) -> tuple[np.ndarray, np.ndarray, np.ndarray]:
    """Canonical form of positions under the mirror: the smaller of (bb0, bb1) and its mirror as unsigned 64-bit values, bb0
    first -> (bb0, bb1, mirrored).  A palindrome (its own mirror) is its own canonical form and is not marked mirrored."""
    b0, b1 = np.asarray(bb0, np.uint64), np.asarray(bb1, np.uint64)
    m0, m1 = mirror_bitboards(b0, b1)
    mirrored = (m0 < b0) | ((m0 == b0) & (m1 < b1))
    return np.where(mirrored, m0, b0), np.where(mirrored, m1, b1), mirrored


class Config:
    """`Config(6, 7, 4)` (scripts/train.py:12).  Only that configuration has kernels."""

    def __init__(self, height: int = HEIGHT, width: int = WIDTH, count: int = COUNT):
        if (height, width, count) != (HEIGHT, WIDTH, COUNT):
            raise ValueError("only Config(6, 7, 4) is supported by the CUDA rules kernels")
        self.height, self.width, self.count = int(height), int(width), int(count)
        self.num_players = 2

    def sample_initial_state(self) -> "State":
        return State(self, 0, 0, 0, legal=0x7F, ended=False, reward=(0, 0))

    def to_json(self):
        return {"count": self.count, "height": self.height, "width": self.width}

    def __eq__(self, other):
        return isinstance(other, Config) and self.to_json() == other.to_json()

    def __hash__(self):
        return hash((self.height, self.width, self.count))


DEFAULT_CONFIG = Config()


class State:
    __slots__ = ("config", "bb0", "bb1", "player", "_legal", "_ended", "_reward")

    def __init__(self, config: Config, bb0: int, bb1: int, player: int, legal=None, ended=None, reward=None):
        self.config = config
        self.bb0, self.bb1, self.player = int(bb0), int(bb1), int(player)
        self._legal, self._ended, self._reward = legal, ended, reward

    def _fill(self):
        if self._legal is None:
            info = rules_engine().state_info(np.array([self.bb0], np.uint64), np.array([self.bb1], np.uint64))
            self._legal = int(info["legal"].cpu()[0])
            self._ended = bool(info["ended"].cpu()[0])
            r = info["reward"].cpu().numpy()[0]
            self._reward = (int(r[0]), int(r[1]))

    @property
    def grid(self) -> np.ndarray:
        return bitboards_to_grid(self.bb0, self.bb1)

    @property
    def legal_mask(self) -> int:
        self._fill()
        return self._legal

    @property
    def has_ended(self) -> bool:
        self._fill()
        return self._ended

    @property
    def reward(self) -> np.ndarray:
        self._fill()
        return np.array(self._reward, dtype=np.float32)

    @property
    def actions(self) -> list["Action"]:
        m = self.legal_mask
        return [Action(self, c) for c in range(WIDTH) if (m >> c) & 1]

    def to_json(self):
        return {"config": self.config.to_json(), "grid": [[int(v) for v in row] for row in self.grid], "player": self.player}

    @classmethod
    def from_json(cls, data) -> "State":
        cfg = data["config"]
        config = Config(cfg["height"], cfg["width"], cfg["count"])
        bb0, bb1 = grid_to_bitboards(np.array(data["grid"]).reshape(config.height, config.width))
        return cls(config, bb0, bb1, data["player"])

    def _key(self):
        return (self.player, self.bb0, self.bb1)

    def __eq__(self, other):
        return isinstance(other, State) and self._key() == other._key()

    def __hash__(self):
        return hash(self._key())

    def __repr__(self):
        return f"State(player={self.player}, grid=\n{self.grid[::-1]})"


class Action:
    __slots__ = ("state", "column")

    def __init__(self, state: State | None, column: int):
        self.state = state
        self.column = int(column)

    def sample_next_state(self) -> State:
        s = self.state
        out = rules_engine().env_step(np.array([s.bb0], np.uint64), np.array([s.bb1], np.uint64),
                                      np.array([s.player], np.uint8), np.array([self.column], np.uint8))
        host = {k: v.cpu().numpy() for k, v in out.items()}
        if host["status"][0] != 0:
            raise ValueError(f"column {self.column} is not playable in this state")
        r = host["reward"][0]
        return State(s.config, int(host["bb0"][0]), int(host["bb1"][0]), int(host["player"][0]), legal=int(host["legal"][0]),
                     ended=bool(host["ended"][0]), reward=(int(r[0]), int(r[1])))

    def to_json(self):
        return {"column": self.column}

    @classmethod
    def from_json(cls, data, state: State | None = None) -> "Action":
        return cls(state, data["column"])

    def __eq__(self, other):
        return (isinstance(other, Action) and self.column == other.column
                and (self.state is other.state or self.state == other.state))

    def __hash__(self):
        return hash(("A", self.column, None if self.state is None else self.state._key()))

    def __repr__(self):
        return f"Action(column={self.column})"


def states_from_arrays(bb0, bb1, player, legal=None, ended=None, reward=None, config: Config = DEFAULT_CONFIG) -> list[State]:
    """Bulk constructor used when engine results are materialised at the API edge."""
    n = len(bb0)
    out = []
    for i in range(n):
        out.append(State(config, int(bb0[i]), int(bb1[i]), int(player[i]),
                         legal=None if legal is None else int(legal[i]),
                         ended=None if ended is None else bool(ended[i]),
                         reward=None if reward is None else (int(reward[i][0]), int(reward[i][1]))))
    return out
