"""Importable alias of the product package.

The package directory is `alphazero-implementation_b200/` (the name the build contract fixes);
a hyphen cannot appear in a Python import, so this module points its `__path__` there and
re-exports the public surface.  All code lives in that directory.
"""
import os as _os

_PKG_DIR = _os.path.join(_os.path.dirname(_os.path.dirname(_os.path.abspath(__file__))), "alphazero-implementation_b200")
__path__.insert(0, _PKG_DIR)  # type: ignore[name-defined]
__version__ = "0.1.0"

from ._lib import LIB_PATH, build_library, library_available  # noqa: E402,F401
from .engine import Engine, EpisodeBatch  # noqa: E402,F401
from .evaluators import HashEvaluator, UniformEvaluator  # noqa: E402,F401
from .game import Action, Config, State, canonical_bitboards, mirror_bitboards  # noqa: E402,F401
from .episode import Episode, Sample  # noqa: E402,F401
from .search import AlphaZeroSearch, ForcedPlayouts, Node, PlayoutCap, RootNoise  # noqa: E402,F401
from .openings import Openings, distinct_openings  # noqa: E402,F401
from .episode_generator import EpisodeGenerator  # noqa: E402,F401
from .models import BasicNN, CNNModel, Connect4Model, Model, ResNet  # noqa: E402,F401
from .player import AlphaZeroPlayer, Arena, Player, calculate_expected_score, elo_ladder, play_game, update_elo  # noqa: E402,F401
