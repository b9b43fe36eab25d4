"""`EpisodeGenerator` with the reference's surface (core/training/episode_generator.py:12-81): E concurrent
self-play games on the GPU engine, episodes yielded in the reference's order.

Per move step: S simulations for every slot (`AlphaZeroSearch.simulate`), then one `az_sample_moves`
launch that records the samples, draws the moves from the uniforms this process takes from NumPy's global
stream (one per slot in slot order — exactly what `np.random.choice` consumes in node.py:33), advances or
recycles the slots and moves finished games to the device episode ring.
"""
from __future__ import annotations

from typing import Callable, Generator

import numpy as np
import torch

from .engine import EpisodeBatch
from .episode import Episode, episodes_from_batch
from .game import State
from .search import AlphaZeroSearch


class EpisodeGenerator:
    def __init__(self, *, model, num_simulations: int, num_episodes: int, game_initial_state: State,
                 exploration_weight: float = 1.0, uniform_source: Callable[[int, int], np.ndarray] | None = None,
                 sampling_moves: int | None = None, **search_kwargs):
        """`sampling_moves` = n: the first n plies of every game are sampled from the visit counts as in the reference, later
        ones play the most visited move (lowest column on ties; `num_sampling_moves` of DeepMind's AlphaZero pseudocode).  The
        uniform of every (step, slot) is still drawn, so NumPy's global stream advances exactly as without it.  None = off.
        Root noise, symmetric leaf evaluation, subtree reuse and playout cap randomization come through `search_kwargs`
        (`root_noise=RootNoise(...)`, `symmetric=True`, `subtree_reuse=True`, `playout_cap=PlayoutCap(...)`: see `AlphaZeroSearch`).
        With the playout cap an episode holds the samples of its full searches only, possibly none; it still counts as an episode."""
        self.sampling_moves = sampling_moves
        self.search = AlphaZeroSearch(model=model, num_simulations=num_simulations, exploration_weight=exploration_weight,
                                      **search_kwargs)
        self.num_episodes = int(num_episodes)
        self.game_initial_state = game_initial_state
        self.num_players = game_initial_state.config.num_players
        self.uniform_source = uniform_source  # (step, E) -> float64[E]; default: np.random.random_sample
        self.last_run: dict = {}

    def update_inference_model(self, model):
        self.search.update_inference_model(model)

    # ------------------------------------------------------------------------------------------
    def iter_steps(self, initial_state: State | None = None, max_steps: int | None = None, reset: bool = True):
        """Run the self-play loop; for every move step yield (step, EpisodeBatch-or-None, rng_state_before_draw).

        Host buffers in, host buffers out: each step's uniforms are copied from pinned host memory, its finished
        episodes are copied to pinned host memory.  The loop is software-pipelined one step deep: step k+1 is
        enqueued on the compute stream before step k's episodes are read back on a copy stream from the other
        half of the device's double-buffered episode ring, so the readback overlaps the next step's kernels.
        Consequently a step's tuple is yielded one step late (and the last one after the loop) - and step k+1's uniforms are taken
        from NumPy's global stream before step k's episodes are yielded: a consumer that draws from `np.random` between yields
        shifts the stream relative to the reference (`generate_episodes` repairs the final position of the stream; pass a
        `uniform_source` for full control).  `reset=False` continues the games already in the engine's slots."""
        from .engine import PinnedEpisodeBuffers

        if initial_state is None:
            initial_state = self.game_initial_state
        E = self.num_episodes
        eng = self.search.engine_for(E, exact=True)  # the slots are the games: an engine grown by a larger run_simulations call is replaced
        eng.set_greedy_from(self.sampling_moves)
        if reset:
            eng.reset_games(initial_state.bb0, initial_state.bb1, initial_state.player)
        elif eng.n_active != E:
            raise RuntimeError("reset=False needs an engine whose slots hold this generator's games")
        u_host = [torch.empty(E, dtype=torch.float64).pin_memory() for _ in range(2)]
        u_dev = [torch.empty(E, dtype=torch.float64, device=eng.device) for _ in range(2)]
        host_buf = PinnedEpisodeBuffers()
        copy_stream = torch.cuda.Stream(device=eng.device)
        compute = torch.cuda.current_stream(eng.device)
        pending = None  # (step, ring, event, rng_state)
        step = 0
        self.h2d_bytes = self.d2h_bytes = 0
        while max_steps is None or step < max_steps:
            # the step's uniforms are drawn before its search is enqueued (the search consumes no NumPy randomness, so the
            # global stream sees the same draws in the same order as the reference's search-then-sample loop)
            rng_state = np.random.get_state() if self.uniform_source is None else None
            u = np.random.random_sample(E) if self.uniform_source is None else np.asarray(self.uniform_source(step, E), np.float64)
            uh, ud = u_host[step & 1], u_dev[step & 1]
            uh.numpy()[:] = u
            ud.copy_(uh, non_blocking=True)
            self.search.simulate_and_move(eng, ud)  # finished games of this step go to the active ring
            ev = torch.cuda.Event()
            ev.record(compute)
            self.h2d_bytes += E * 8
            if pending is not None:  # read the previous step's ring (the inactive one) while this step runs
                yield self._finish_step(eng, pending, host_buf, copy_stream)
            # only now may the other ring be recycled: zero it and make it the target of the next step
            ring = eng.swap_episode_ring()
            pending = (step, ring, ev, rng_state)
            step += 1
        if pending is not None:
            yield self._finish_step(eng, pending, host_buf, copy_stream)

    def _finish_step(self, eng, pending, host_buf, copy_stream):
        step, ring, ev, rng_state = pending
        copy_stream.wait_event(ev)
        batch = eng.read_ring_to_host(ring, host_buf, copy_stream)
        self.d2h_bytes += 32 + (0 if batch is None else sum(getattr(batch, f).nbytes for f in (
            "ep_slot", "ep_step", "ep_len", "ep_offset", "ep_outcome", "s_bb0", "s_bb1", "s_player", "s_counts")))
        return step, batch, rng_state

    def generate_episodes(self, initial_state: State | None = None) -> Generator[Episode, None, None]:
        """Reference semantics: yield episodes in (move step, slot) order, stop after `num_episodes`,
        abandoning games in flight (episode_generator.py:48-81)."""
        count = 0
        S = self.search.num_simulations
        for step, batch, rng_state in self.iter_steps(initial_state):
            if batch is None:
                continue
            episodes = episodes_from_batch(batch, S)
            for i, ep in enumerate(episodes):
                count += 1
                if count >= self.num_episodes:
                    if rng_state is not None:
                        # the reference stops drawing after this slot: leave NumPy's global stream where it would be
                        np.random.set_state(rng_state)
                        np.random.random_sample(int(batch.ep_slot[i]) + 1)
                    self.last_run = dict(steps=step + 1, episodes=count)
                    yield ep
                    return
                yield ep

    def generate_batches(self, initial_state: State | None = None, max_steps: int | None = None,
                         quota: int | None = None) -> Generator[EpisodeBatch, None, None]:
        """Array-level variant for large E: yields `EpisodeBatch`es (flat host arrays) as games finish.
        With `quota`, truncates at the reference's stopping point."""
        count = 0
        for step, batch, _ in self.iter_steps(initial_state, max_steps):
            if batch is None:
                continue
            if quota is not None and count + len(batch) >= quota:
                keep = quota - count
                yield _truncate(batch, keep)
                return
            count += len(batch)
            yield batch


def _truncate(b: EpisodeBatch, keep: int) -> EpisodeBatch:
    ns = int(b.ep_len[:keep].sum())
    return EpisodeBatch(b.ep_slot[:keep], b.ep_step[:keep], b.ep_len[:keep], b.ep_offset[:keep], b.ep_outcome[:keep],
                        b.s_bb0[:ns], b.s_bb1[:ns], b.s_player[:ns], b.s_counts[:ns])
