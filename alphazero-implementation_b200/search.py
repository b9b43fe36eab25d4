"""`AlphaZeroSearch` / `Node` with the reference's call surface (core/search/mcts/search.py:10-91,
core/search/mcts/node.py:7-73), executed by the CUDA tree arena.

`run_simulations(nodes)` uploads the roots' positions, runs `num_simulations` simulations per tree on
the GPU (fused kernel for the built-in deterministic evaluators; select -> gather -> net -> expand/backup
for a network; select -> `predict(states)` -> expand/backup for any other object with a `predict`), and
writes the result back into the caller's `Node`s in place: visit_count, value_sum and one level of
children with their statistics (what `improved_policy`, `value` and `select_next_node` read).
`materialize="full"` rebuilds the entire tree as `Node`s.
"""
from __future__ import annotations

import os
from dataclasses import dataclass

import numpy as np
import torch

from .engine import (EVAL_HASH, EVAL_UNIFORM, LEAF_EVAL, POLICY_LOGITS, POLICY_PRIORS, TREE_ROOT_ENDED, Engine)
from .game import Action, State, states_from_arrays


class Node:
    """Host-side view of a tree node; same attributes and properties as the reference (node.py:7-73)."""

    __slots__ = ("state", "parent", "children", "visit_count", "value_sum", "prior")

    def __init__(self, state: State, parent: "Node | None" = None, prior: float = 0.0):
        self.state = state
        self.parent = parent
        self.children: dict[Action, Node] = {}
        self.visit_count = 0
        self.value_sum = 0.0
        self.prior = prior

    @property
    def raw_policy(self) -> dict[Action, float]:
        return {a: ch.prior for a, ch in self.children.items()}

    @property
    def improved_policy(self) -> dict[Action, float]:
        return {a: ch.visit_count / (self.visit_count - 1) for a, ch in self.children.items()}

    def select_next_node(self) -> "Node":
        """Sample the move from the visit distribution with the global NumPy stream (node.py:31-42)."""
        pol = self.improved_policy
        index = np.random.choice(len(pol), p=list(pol.values()))
        action = list(pol.keys())[index]
        child = self.children[action]
        return Node(state=child.state if child.state is not None else action.sample_next_state(), parent=self,
                    prior=pol[action])

    def add_child(self, action: Action, child_state: State, prior: float) -> "Node":
        child = Node(state=child_state, parent=self, prior=prior)
        self.children[action] = child
        return child

    @property
    def value(self) -> float:
        if self.visit_count == 0:
            return 0
        return self.value_sum / self.visit_count

    @property
    def is_expanded(self) -> bool:
        return len(self.children) > 0

    @property
    def is_terminal(self) -> bool:
        return self.state.has_ended

    @property
    def utility_values(self) -> list[float]:
        return self.state.reward.tolist()

    @property
    def is_root(self) -> bool:
        return self.parent is None


@dataclass(frozen=True)
class RootNoise:
    """Dirichlet noise on the root priors of every search (`add_exploration_noise` of DeepMind's AlphaZero pseudocode):
    after the first simulation has expanded the root, each root child's prior becomes (1 - fraction) * P + fraction * eta,
    eta ~ Dirichlet(alpha) over the legal columns (`Engine.set_root_noise`).  Draws are a function of (seed, slot_offset + slot,
    search number, column) only: `slot_offset` is the global index of the engine's first game, so sharded self-play draws what
    the unsharded run draws.  Off (None) by default: then the search is the reference's, bit for bit."""

    alpha: float = 1.0
    fraction: float = 0.25
    seed: int = 0
    slot_offset: int = 0


@dataclass(frozen=True)
class PlayoutCap:
    """Playout cap randomization of the self-play searches (KataGo; `Engine.set_playout_cap`): each search of a move step is full
    with probability `full_probability` (num_simulations new simulations) or fast (`fast_simulations`).  Every move is played, but
    only the full searches become training samples, so a game costs fewer simulations while the policy targets keep the full
    search's depth.  Fast searches get no root noise.  `visit_budget` (with subtree reuse): a search tops the root up to that many
    visits instead of adding them, at least one new simulation.  The draws are a function of (seed, slot_offset + slot, move step)
    only.  Off (None) by default."""

    fast_simulations: int
    full_probability: float = 0.25
    seed: int = 0
    slot_offset: int = 0
    visit_budget: bool = False


class _GraphedStep:
    """The simulation loop of the network-in-the-loop path, optionally replayed as a CUDA graph.

    n simulations = select, then (evaluate, expand + backup + next select) n - 1 times, then evaluate, expand + backup:
    between two evaluator calls only `az_expand_backup_select` runs.  The repeated part has fixed shapes (row i of the packed
    batch = slot i), so one capture serves every simulation of every move.  Capture only records; the warm-up steps that
    precede it are real simulations.
    """

    UNROLL = int(os.environ.get("AZ_GRAPH_UNROLL", "32"))  # simulations per replayed graph (a second capture; 1 = none): 16384 x 800, ResNet 4x64: 381.8 -> 372.7 ms per move step

    def __init__(self, engine: Engine, net, layout: int, cache: bool | int = True):
        self.engine, self.net, self.layout = engine, net, layout
        # before the first selection (and any capture).  AZ_COMPACT_FUSED=0: the list of the leaves to evaluate comes from one more
        # launch per simulation (k_compact_leaves) instead of from k_expand_select itself
        engine.set_leaf_compaction(getattr(net, "wants_leaf_compaction", False), fused=os.environ.get("AZ_COMPACT_FUSED", "1") != "0")
        # the evaluation cache changes no result bit when a leaf's outputs depend on its position alone
        exact = engine.leaf_compaction and getattr(net, "position_only_outputs", False)
        engine.set_eval_cache((None if cache is True else int(cache)) if cache and exact else 0)
        self.graph = None
        self.graph_unrolled = None
        self.n = -1
        self.x = None

    def evaluate(self):
        e = self.engine
        if getattr(self.net, "evaluates_leaves_directly", False):  # tcgen05 kernels with the leaf gather fused in
            return self.net.forward_leaves(e)
        e.gather_leaves(self.layout, self.x)
        return self.net(self.x)

    def middle(self):
        """evaluate the selected leaves, expand + back up, select the next leaves"""
        logits, values = self.evaluate()
        self.engine.expand_backup_select(logits, values, POLICY_LOGITS)

    def run(self, num_steps: int, use_graph: bool, evaluator_events: list | None = None):
        """`evaluator_events`: run un-graphed and append a (start, end) CUDA-event pair around every evaluator call."""
        e = self.engine
        if num_steps <= 0:
            return
        if evaluator_events is not None:
            if self.n != e.n_active:
                self.n = e.n_active
                self.x = e.gather_leaves(self.layout)
                self.graph = self.graph_unrolled = None
            e.select_leaves()
            for i in range(num_steps):
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                logits, values = self.evaluate()
                b.record()
                evaluator_events.append((a, b))
                if i + 1 < num_steps:
                    e.expand_backup_select(logits, values, POLICY_LOGITS)
                else:
                    e.expand_backup(logits, values, POLICY_LOGITS)
            return
        if self.n != e.n_active:
            self.n = e.n_active
            self.x = e.gather_leaves(self.layout)  # allocates the packed batch once per batch size
            self.graph = self.graph_unrolled = None
        e.select_leaves()
        middles = num_steps - 1
        done = 0
        if use_graph and self.graph is None and middles > 2:
            for _ in range(2):  # cuDNN / cuBLAS pick algorithms and allocate workspaces outside capture
                self.middle()
            done = 2
            torch.cuda.current_stream().synchronize()
            g = torch.cuda.CUDAGraph()
            side = torch.cuda.Stream(device=e.device)
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                # thread_local: a training thread may allocate while the self-play thread captures (trainer.py overlap)
                with torch.cuda.graph(g, stream=side, capture_error_mode="thread_local"):
                    self.middle()
                # ... and UNROLL of them in a second graph: fewer graph launches (and gaps between them) per move step
                # (only for long searches: the engine's host-side guard counts every call, recorded ones included, against the
                # arena's num_simulations)
                if self.UNROLL > 1 and middles >= 4 * self.UNROLL:
                    gu = torch.cuda.CUDAGraph()
                    with torch.cuda.graph(gu, stream=side, capture_error_mode="thread_local"):
                        for _ in range(self.UNROLL):
                            self.middle()
                    self.graph_unrolled = gu
            torch.cuda.current_stream().wait_stream(side)
            self.graph = g
        todo = middles - done
        if use_graph and self.graph is not None:
            if self.graph_unrolled is not None:
                for _ in range(todo // self.UNROLL):
                    self.graph_unrolled.replay()
                todo %= self.UNROLL
            for _ in range(todo):
                self.graph.replay()
        else:
            for _ in range(todo):
                self.middle()
        logits, values = self.evaluate()
        e.expand_backup(logits, values, POLICY_LOGITS)


class AlphaZeroSearch:
    def __init__(self, *, model, num_simulations: int, exploration_weight: float = 1.0, device: int | None = None,
                 lanes_per_tree: int = 0, inference_dtype: torch.dtype | None = None, use_cuda_graph: bool = True,
                 use_tensor_core_kernels: bool = True, trunk_variant: int | None = None, eval_cache: bool | int = True,
                 root_noise: RootNoise | None = None, symmetric: bool = False, subtree_reuse: bool | int = False,
                 playout_cap: PlayoutCap | None = None):
        """`eval_cache`: serve repeated leaf positions from the engine's evaluation cache (`Engine.set_eval_cache`) when the
        evaluator's outputs depend on the position alone (`InferenceNet.position_only_outputs`); same results, fewer evaluator rows.
        True = a table sized for the engine, False = off, an int = log2 of its entry count.
        `root_noise`: every search runs one simulation, mixes Dirichlet noise into the root priors (`RootNoise`), then runs the
        other num_simulations - 1; None (default) = no noise.
        `symmetric`: evaluate every leaf in its canonical orientation under Connect4's left-right mirror (`Engine.set_symmetric_eval`):
        a position and its mirror get the same value and mirrored priors, and share one evaluator row and one cache entry.  Network
        and `predict` evaluators only (ValueError for the built-in ones); off (default) = the reference's search, bit for bit.
        `subtree_reuse`: in the self-play move step (`simulate_and_move`) the played child becomes the next root and keeps its subtree
        with all its statistics (AlphaGo Zero), as long as N(child) + num_simulations <= max_root_visits (`Engine.set_subtree_reuse`);
        each search still runs num_simulations new simulations, so a root then holds more visits.  True = max_root_visits of
        4 num_simulations, an int = max_root_visits, False (default) = every move step starts from a fresh root, as the reference
        does.  `run_simulations(nodes)` always starts from the given fresh roots.
        `playout_cap`: the self-play move steps run full or fast searches (`PlayoutCap`) and record only the full ones as samples;
        None (default) = every search is full.  `run_simulations(nodes)` always runs full searches."""
        self.symmetric = bool(symmetric)
        self.playout_cap = playout_cap
        self.subtree_reuse = subtree_reuse
        self.inference_model = model.get_inference_clone()
        self.eval_cache = eval_cache
        self.root_noise = root_noise
        self.num_simulations = int(num_simulations)
        self.exploration_weight = exploration_weight
        self.device_index = device
        self.lanes_per_tree = lanes_per_tree
        self.inference_dtype = inference_dtype
        self.use_cuda_graph = use_cuda_graph
        self.use_tensor_core_kernels = use_tensor_core_kernels
        self.trunk_variant = trunk_variant
        self._engine: Engine | None = None
        self._net = None
        self._mode = None
        self._graphed: _GraphedStep | None = None
        self._refresh_net()

    # -- weights ---------------------------------------------------------------------------------
    def update_inference_model(self, model):
        """Copy the training model's weights into the inference clone (search.py:22-25)."""
        self.inference_model.load_state_dict(model.state_dict())
        self.inference_model.eval()
        self._refresh_net()

    def _refresh_net(self):
        """(Re)build the search-time form of the inference model.  With unchanged architecture the packed weights are rewritten
        in place (same device addresses), so the captured CUDA graph of the simulation step stays valid.  The weights are
        produced on the caller's current stream and consumed on whichever stream the search runs on (trainer.py plays on its own
        stream from another thread): the stream is synchronised before returning, so no search can read half-written weights."""
        from .models import BasicNN, InferenceNet, Model

        m = self.inference_model
        if getattr(m, "az_builtin_eval_kind", 0) in (EVAL_UNIFORM, EVAL_HASH):
            self._mode, self._net, self._graphed = "builtin", None, None
        elif isinstance(m, Model):
            # Defaults: BasicNN in fp32 (the reference's arithmetic: BASELINE config 1 reproduces the reference's episodes); the conv
            # nets on the hand-written tensor-core kernels with fp16 operands, which stay within 1e-3 of the fp32 `predict`
            # (tests/test_gpu_config3.py) at the speed of bf16.  bf16 (BASELINE config 3's format) and fp32 are one argument away.
            dtype = self.inference_dtype or (torch.float32 if isinstance(m, BasicNN) else torch.float16)
            dev = torch.device("cuda", torch.cuda.current_device() if self.device_index is None else self.device_index)
            if self._net is not None and self._mode == "net" and self._net.refresh(m):
                pass  # in place: graph kept
            else:
                self._graphed = None
                self._mode, self._net = "net", InferenceNet(m, dtype=dtype, device=dev, use_tensor_core_kernels=self.use_tensor_core_kernels,
                                                              trunk_variant=self.trunk_variant)
            torch.cuda.current_stream(dev).synchronize()
        else:
            self._mode, self._net, self._graphed = "predict", None, None
        if self.symmetric and self._mode == "builtin":
            raise ValueError("symmetric=True needs a network or predict() evaluator: the built-in evaluators run in the fused "
                             "k_run_sims path, which has no symmetric variant (and the uniform one is symmetric already)")
        if self._engine is not None:
            self._engine.bump_eval_epoch()  # other weights or another evaluator: what the cache holds no longer applies
            torch.cuda.current_stream(self._engine.device).synchronize()

    @property
    def evaluator_name(self) -> str:
        """The kernel that evaluates the leaves (bench.py's roofline names it)."""
        if self._mode == "builtin":
            return "k_run_sims (built-in evaluator)"
        if self._mode == "net":
            return self._net.kernel_name
        return "user predict()"

    def _search_runs(self, S: int) -> list[int]:
        """A search of S simulations as runs of consecutive simulations: with root noise, one simulation, the noise, the rest."""
        return [1, S - 1] if self.root_noise is not None and S > 0 else [S]

    @property
    def max_root_visits(self) -> int:
        """max_root_visits of the self-play engine's subtree reuse: 0 = off"""
        r = self.subtree_reuse
        if r is True:
            return 4 * self.num_simulations
        return 0 if r is False or r is None else int(r)

    def launches_per_move_step(self) -> int:
        """Kernels of libaz_engine.so per self-play move step (`simulate_and_move`)."""
        S = self.num_simulations
        runs = [n for n in self._search_runs(S) if n > 0]
        noise = 1 if self.root_noise is not None else 0
        greedy = self._engine is not None and self._engine.greedy_from >= 0
        reuse = 1 if self.max_root_visits else 0  # k_reroot after k_sample_moves
        cap = self.playout_cap is not None
        redraw = 1 if cap and reuse else 0  # k_cap_draw after k_reroot (without reuse k_sample_moves draws the next budgets itself)
        if self._mode == "builtin":
            # one k_run_sims per run, the last one with the move fused in - unless the greedy cutoff, subtree reuse, the playout cap (or
            # a search of one simulation with noise) leaves the move to k_sample_moves
            return len(runs) + noise + (1 if greedy or reuse or cap or noise and S == 1 else 0) + reuse + redraw
        # per run of n: k_select; n - 1 x (evaluator or gather, k_expand_select); evaluator, k_expand_backup.  Then k_root_noise
        # between the runs and k_sample_moves.  When the evaluator walks the compacted leaf list: one k_compact_leaves after
        # every k_select (the later lists come out of k_expand_select) or, AZ_COMPACT_FUSED=0, one per selection
        n = sum(2 * r + 1 for r in runs) + noise + 1 + reuse + redraw
        if not getattr(self._net, "wants_leaf_compaction", False):
            return n
        return n + (len(runs) if os.environ.get("AZ_COMPACT_FUSED", "1") != "0" else S)

    def _configure_noise(self, engine: Engine):
        rn = self.root_noise
        if rn is None:
            if engine.root_noise is not None:
                engine.set_root_noise(None)
        elif engine.root_noise != (float(rn.alpha), float(rn.fraction), int(rn.seed), int(rn.slot_offset)):
            engine.set_root_noise(rn.alpha, rn.fraction, rn.seed, rn.slot_offset)

    def _configure_symmetry(self, engine: Engine):
        """before any selection of this search and any capture of its CUDA graph (launches bake the kernel choice in)"""
        if engine.symmetric_eval != self.symmetric:
            engine.set_symmetric_eval(self.symmetric)
            if self._graphed is not None and self._graphed.engine is engine:
                self._graphed = None

    def _configure_reuse(self, engine: Engine):
        """before the move step's search and any capture of its CUDA graph (launches bake the tree arena in); a change resets every
        tree to a fresh root"""
        v = self.max_root_visits
        if engine.subtree_reuse != v:
            engine.set_subtree_reuse(v)
            if self._graphed is not None and self._graphed.engine is engine:
                self._graphed = None

    def _configure_cap(self, engine: Engine):
        """before the move step's search and any capture of its CUDA graph (switching the cap on or off changes the kernels)"""
        pc = self.playout_cap
        want = None if pc is None else (int(pc.fast_simulations), float(pc.full_probability), int(pc.seed), int(pc.slot_offset),
                                        bool(pc.visit_budget))
        if engine.playout_cap == want:
            return
        switched = (engine.playout_cap is None) != (want is None)
        if want is None:
            engine.set_playout_cap(None)
        else:
            engine.set_playout_cap(*want)
        if switched and self._graphed is not None and self._graphed.engine is engine:
            self._graphed = None

    def close(self):
        if self._engine is not None:
            self._engine.close()
            self._engine = None
        self._graphed = None

    # -- engine ----------------------------------------------------------------------------------
    def engine_for(self, n: int, exact: bool = False) -> Engine:
        """The engine for n trees: grown when too small; `exact` (the self-play loop, whose slots ARE the games) also replaces a
        larger one left behind by an earlier `run_simulations` call."""
        if self._engine is None or self._engine.num_games < n or (exact and self._engine.num_games != n):
            if self._engine is not None:
                self._engine.close()
            self._engine = Engine(num_games=n, num_simulations=self.num_simulations, c_puct=float(self.exploration_weight),
                                  device=self.device_index, lanes_per_tree=self.lanes_per_tree)
            self._graphed = None
        self._configure_symmetry(self._engine)
        return self._engine

    def simulate(self, engine: Engine, num_simulations: int | None = None, evaluator_events: list | None = None):
        """`num_simulations` simulations on every active tree of `engine` (fresh roots already set); with `root_noise`, the noise
        is mixed into the root priors after the first.  `evaluator_events` (network evaluators only): run the steps un-graphed and
        collect a CUDA-event pair around every evaluator call."""
        S = self.num_simulations if num_simulations is None else num_simulations
        self._configure_symmetry(engine)
        self._configure_noise(engine)
        runs = self._search_runs(S)
        for i, n in enumerate(runs):
            if i:
                engine.apply_root_noise()
            self._simulate_run(engine, n, evaluator_events)

    def _simulate_run(self, engine: Engine, S: int, evaluator_events: list | None):
        if S <= 0:
            return
        if self._mode == "builtin":
            engine.run_simulations(S, self.inference_model.az_builtin_eval_kind)
        elif self._mode == "net":
            if self._graphed is None or self._graphed.engine is not engine:
                self._graphed = _GraphedStep(engine, self._net, self._net.input_layout, self.eval_cache)
            self._graphed.run(S, self.use_cuda_graph, evaluator_events)
        else:
            self._simulate_predict(engine, S)

    def simulate_and_move(self, engine: Engine, uniforms: torch.Tensor, finished: torch.Tensor | None = None):
        """One self-play move step: `simulate` then `Engine.sample_moves(uniforms)`.  With a built-in evaluator both run in
        one launch (`az_run_move_step`), with identical results.  With `subtree_reuse`, the move keeps the played child's subtree
        (`k_reroot`) for the next step's search."""
        self._configure_reuse(engine)
        self._configure_cap(engine)
        if self._mode == "builtin":
            kind = self.inference_model.az_builtin_eval_kind
            self._configure_noise(engine)
            *head, last = self._search_runs(self.num_simulations)
            for n in head:
                engine.run_simulations(n, kind)
                engine.apply_root_noise()
            if last > 0:
                engine.run_move_step(last, kind, uniforms, finished)
            else:
                engine.sample_moves(uniforms, finished)
        else:
            self.simulate(engine)
            engine.sample_moves(uniforms, finished)

    def _simulate_predict(self, engine: Engine, S: int):
        """Generic evaluator: any object with the reference's `predict(states)`."""
        n = engine.n_active
        for _ in range(S):
            engine.select_leaves()
            info = {k: v.cpu().numpy() for k, v in engine.leaf_info().items()}
            rows = np.nonzero(info["status"] == LEAF_EVAL)[0]
            pri = np.zeros((n, 7), np.float32)
            val = np.zeros((n, 2), np.float32)
            if len(rows):
                states = states_from_arrays(info["bb0"][rows], info["bb1"][rows], info["player"][rows], legal=info["legal"][rows],
                                            ended=np.zeros(len(rows), bool), reward=np.zeros((len(rows), 2), np.int8))
                policies, values = self.inference_model.predict(states)
                for r, pol, v in zip(rows, policies, values):
                    for a, p in pol.items():
                        pri[r, a.column] = p
                    val[r] = v
            engine.expand_backup(torch.from_numpy(pri).to(engine.device), torch.from_numpy(val).to(engine.device), POLICY_PRIORS)

    # -- reference surface -----------------------------------------------------------------------
    def run(self, root: Node) -> tuple[dict[Action, float], float]:
        self.run_simulations([root])
        return root.improved_policy, root.value

    def run_simulations(self, current_nodes: list[Node], materialize: str = "root") -> None:
        if not current_nodes:
            return
        # A terminal node WITH a parent is a leaf the reference visits num_simulations times (search.py:75-77): the reward of the
        # player who moved into it is backed up along the parent chain (no sign flip at the terminal node itself, :55-56).
        # Host arithmetic, exact (rewards are -1 / 0 / +1).  A terminal node without a parent raises below, as in the reference.
        done = [nd for nd in current_nodes if nd.parent is not None and nd.state.has_ended]
        for nd in done:
            for _ in range(self.num_simulations):
                v = float(nd.state.reward[nd.parent.state.player])
                walk = nd
                while walk is not None:
                    walk.value_sum += v
                    walk.visit_count += 1
                    if not walk.is_terminal:
                        v = -v
                    walk = walk.parent
        if done:
            current_nodes = [nd for nd in current_nodes if not (nd.parent is not None and nd.state.has_ended)]
            if not current_nodes:
                return
        for nd in current_nodes:
            if nd.children or nd.visit_count:
                raise ValueError("run_simulations expects fresh roots (the reference always passes Node(state)); "
                                 "continuing a search on an already expanded Node is not supported")
        n = len(current_nodes)
        eng = self.engine_for(n)
        bb0 = np.array([nd.state.bb0 for nd in current_nodes], np.uint64)
        bb1 = np.array([nd.state.bb1 for nd in current_nodes], np.uint64)
        pl = np.array([nd.state.player for nd in current_nodes], np.uint8)
        eng.set_roots(bb0, bb1, pl)
        self.simulate(eng)
        st = {k: v.cpu().numpy() for k, v in eng.root_stats().items()}
        if (st["err"] == TREE_ROOT_ENDED).any():
            # the reference dereferences node.parent (None) for a terminal root (search.py:76)
            raise AttributeError("'NoneType' object has no attribute 'state'")
        # successor states of every legal root move, one rules-kernel call
        cols = np.tile(np.arange(7, dtype=np.uint8), n)
        nxt = {k: v.cpu().numpy() for k, v in eng.env_step(np.repeat(bb0, 7), np.repeat(bb1, 7), np.repeat(pl, 7), cols).items()}
        for i, nd in enumerate(current_nodes):
            nd.visit_count = int(st["root_N"][i])
            nd.value_sum = float(st["root_W"][i])
            nd.state._legal, nd.state._ended, nd.state._reward = int(st["legal"][i]), False, (0, 0)
            for c in range(7):
                if not (st["legal"][i] >> c) & 1:
                    continue
                k = 7 * i + c
                child_state = State(nd.state.config, int(nxt["bb0"][k]), int(nxt["bb1"][k]), int(nxt["player"][k]),
                                    legal=int(nxt["legal"][k]), ended=bool(nxt["ended"][k]),
                                    reward=(int(nxt["reward"][k][0]), int(nxt["reward"][k][1])))
                ch = nd.add_child(Action(nd.state, c), child_state, float(st["child_P"][i, c]))
                ch.visit_count = int(st["child_N"][i, c])
                ch.value_sum = float(st["child_W"][i, c])
        if materialize == "full":
            for i, nd in enumerate(current_nodes):
                _materialize_subtree(eng, i, nd)


def _materialize_subtree(eng: Engine, slot: int, root: Node):
    """Rebuild every expanded node of tree `slot` below `root` as `Node`s (children in column order)."""
    t = eng.export_tree(slot)
    W, N, P, CB = t["W"], t["N"], t["P"], t["first_child"]
    rules = eng

    def expand(node: Node, idx: int):
        cb = int(CB[idx])
        if cb == 0:
            return
        s = node.state
        legal = [c for c in range(7) if (s.legal_mask >> c) & 1]
        n = len(legal)
        nxt = {k: v.cpu().numpy() for k, v in rules.env_step(np.full(n, s.bb0, np.uint64), np.full(n, s.bb1, np.uint64),
                                                             np.full(n, s.player, np.uint8), np.array(legal, np.uint8)).items()}
        node.children = {}
        for j, c in enumerate(legal):
            cs = State(s.config, int(nxt["bb0"][j]), int(nxt["bb1"][j]), int(nxt["player"][j]), legal=int(nxt["legal"][j]),
                       ended=bool(nxt["ended"][j]), reward=(int(nxt["reward"][j][0]), int(nxt["reward"][j][1])))
            ch = node.add_child(Action(s, c), cs, float(P[cb + j]))
            ch.visit_count, ch.value_sum = int(N[cb + j]), float(W[cb + j])
            expand(ch, cb + j)

    expand(root, 0)
