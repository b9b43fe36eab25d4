"""AlphaZero iteration loop with the reference `Trainer.train(...)` signature (core/training/trainer.py:28-38),
without Lightning: self-play on the GPU engine -> replay buffer -> `Model.training_step` epochs -> weight sync.

Multi-GPU (one process per GPU): every rank plays its shard of the games; finished episodes are all-gathered
over NCCL into every rank's replay buffer; rank 0 runs the optimiser and broadcasts the new weights
(`update_inference_model`, search.py:22-25 / datamodule.py:100).  Like the reference (datamodule.py:89-101), self-play of
iteration k+1 runs on a background thread — here with its own CUDA stream — while iteration k trains.
"""
from __future__ import annotations

import dataclasses
import time

import torch
import torch.distributed as dist

from .distributed import all_gather_episodes, broadcast_weights, shard_range
from .episode_generator import EpisodeGenerator
from .replay import ReplayBuffer


class _GraphedTraining:
    """The optimiser steps of one iteration (models/base/model.py:27-48 per minibatch: CE(soft visit targets) + MSE, Adam) with
    every full-size minibatch after the first three replayed from ONE CUDA graph.

    The eager loop is launch-bound once the layouts are right (ResNet 4x64, batch 2048, one B200, scripts/bench_training.py:
    7.6 ms per step eager NCHW, 3.9 ms eager NHWC, 3.0 ms replayed; BasicNN 1.29 -> 0.47 ms), and while it holds the GIL it
    also starves the self-play thread.  Everything a step needs is therefore
    a device-side function of a device-side step counter: rows `perm[ctr*B : (ctr+1)*B]` of the replay set are gathered,
    expanded to planes by `az_encode_states`, run through forward / backward / Adam(capturable), the loss is added to a
    device accumulator and the counter is incremented - so a replay takes no host arguments.  The first three steps run
    eagerly on the training stream (they ARE training steps; cuDNN / cuBLAS pick algorithms and the optimiser state is
    created there), the capture only records.  The replay set is copied into static buffers every iteration, so one capture
    serves the whole training run (a buffer that has to grow drops the graph; the next iteration captures again).
    `mirror_augment`: every epoch draws one Bernoulli(1/2) flag per sample (next to the permutation, from the same generator);
    a flagged sample is trained in its left-right mirror image - bitboards mirrored by `az_mirror_states` before the encoding,
    policy target columns reversed.  The flags are device data read by the step, so the graph still takes no host arguments.
    """

    MIN_REPLAYS = 4  # fewer full-size steps than 3 eager + this: not worth a capture

    def __init__(self, model, opt, batch_size: int, precision: str, device: torch.device, channels_last: bool = True,
                 mirror_augment: bool = False):
        from .game import rules_engine

        self.model, self.opt, self.B, self.precision, self.device = model, opt, int(batch_size), precision, device
        # conv nets train in NHWC: cuDNN's NCHW batch-norm kernels take 3.3 of the 6.4 ms of GPU time of a ResNet 4x64 step at
        # 6x7 boards and every conv is wrapped in layout transposes (scripts/profile_train_step.py); same arithmetic
        self.channels_last = channels_last and any(p.dim() == 4 for p in model.parameters())
        if self.channels_last:
            model.to(memory_format=torch.channels_last)
        self.eng = rules_engine()
        self.stream = torch.cuda.Stream(device=device)
        self.base = torch.arange(self.B, device=device)
        self.ctr = torch.zeros(1, dtype=torch.int64, device=device)
        self.loss_sum = torch.zeros((), dtype=torch.float32, device=device)
        self.replays = 0  # graph replays so far (reported by Trainer.history)
        self.mirror_augment = bool(mirror_augment)
        self.cap, self.data, self.perm, self.flip, self.graph = 0, None, None, None, None

    def _step_on(self, j):
        bb0, bb1, pl, policy, value = self.data
        if self.mirror_augment:
            f = self.flip.index_select(0, j)
            b0, b1 = self.eng.mirror_states(bb0.index_select(0, j), bb1.index_select(0, j), f)
            x = self.eng.encode_states(b0, b1, pl.index_select(0, j), self.model.input_layout)
            pol = policy.index_select(0, j)
            pol = torch.where(f.bool().unsqueeze(1), pol.flip(1), pol)
        else:
            x = self.eng.encode_states(bb0.index_select(0, j), bb1.index_select(0, j), pl.index_select(0, j), self.model.input_layout)
            pol = policy.index_select(0, j)
        if self.channels_last and x.dim() == 4:
            x = x.contiguous(memory_format=torch.channels_last)
        self.opt.zero_grad(set_to_none=True)
        with torch.autocast("cuda", dtype=torch.bfloat16, enabled=self.precision == "bf16-mixed"):
            loss = self.model.training_step((x, pol, value.index_select(0, j)), 0)
        loss.backward()
        self.opt.step()
        self.loss_sum += loss.detach().float()

    def _body(self):
        self._step_on(self.perm.index_select(0, self.base + self.ctr * self.B))
        self.ctr += 1

    def _load(self, replay: ReplayBuffer) -> int:
        """This iteration's replay set -> the static buffers the graph reads (grown by doubling; growing drops the graph)."""
        fresh = replay.tensors()
        n = int(fresh[0].numel())
        if n > self.cap:
            self.cap = max(2 * n, 1 << 16)
            self.data = tuple(torch.empty((self.cap,) + tuple(t.shape[1:]), dtype=t.dtype, device=self.device) for t in fresh)
            self.perm = torch.zeros(self.cap, dtype=torch.int64, device=self.device)
            self.flip = torch.zeros(self.cap, dtype=torch.uint8, device=self.device) if self.mirror_augment else None
            self.graph = None
        for dst, src in zip(self.data, fresh):
            dst[:n].copy_(src)
        return n

    def run(self, replay: ReplayBuffer, epochs: int, generator: torch.Generator, use_graph: bool = True):
        """-> (sum of the minibatch losses as a device scalar, number of optimiser steps)"""
        cur = torch.cuda.current_stream(self.device)
        self.stream.wait_stream(cur)
        with torch.cuda.stream(self.stream):
            n = self._load(replay)
            full, tail = divmod(n, self.B)
            self.loss_sum.zero_()
            for _ in range(epochs):
                self.perm[:n].copy_(torch.randperm(n, generator=generator))
                if self.mirror_augment:
                    self.flip[:n].copy_(torch.randint(0, 2, (n,), generator=generator, dtype=torch.uint8))
                self.ctr.zero_()
                done = 0
                if use_graph and self.graph is None and full >= 3 + self.MIN_REPLAYS:
                    for _ in range(3):
                        self._body()
                    done = 3
                    # capture_begin / capture_end rather than `with torch.cuda.graph(...)`: that context manager starts with a
                    # device-wide synchronize, i.e. it would wait for everything the self-play thread has queued.
                    # thread_local: the self-play thread allocates and launches while this thread captures.
                    self.stream.synchronize()
                    graph = torch.cuda.CUDAGraph()
                    graph.capture_begin(capture_error_mode="thread_local")
                    try:
                        self._body()
                    finally:
                        graph.capture_end()
                    self.graph = graph
                for _ in range(full - done):
                    if use_graph and self.graph is not None:
                        self.graph.replay()
                        self.replays += 1
                    else:
                        self._body()
                if tail:  # DataLoader(drop_last=False): the short last minibatch, eager
                    self._step_on(self.perm[full * self.B:n])
            self.stream.synchronize()
        cur.wait_stream(self.stream)
        return self.loss_sum.clone(), epochs * (full + (1 if tail else 0))


class Trainer:
    def __init__(self, model, device: int | None = None):
        self.model = model
        self.device_index = torch.cuda.current_device() if device is None else device
        self.device = torch.device("cuda", self.device_index)
        self.history: list[dict] = []

    def train(self, *, num_iterations: int, episodes_per_iter: int, simulations_per_episode: int, epochs_per_iter: int,
              initial_state, buffer_size: int, save_every_n_iterations: int = 0, batch_size: int = 32, seed: int = 0,
              overlap: bool = True, inference_dtype: torch.dtype | None = None, precision: str = "32-true",
              cuda_graph: bool = True, trainer_share: float | None = None, save_dir: str | None = None, root_noise=None,
              sampling_moves: int | None = None, symmetric: bool = False, mirror_augment: bool = False,
              subtree_reuse: bool | int = False, playout_cap=None, forced_playouts=None, openings=None):
        """`overlap=True` reproduces the reference's pipeline (datamodule.py:89-101): the self-play of iteration k+1 runs on a
        background thread (own CUDA stream, weights as of the end of iteration k-1's training) while iteration k trains.
        `precision`: "32-true" (the reference's Lightning default) or "bf16-mixed" (forward / backward under bf16 autocast,
        fp32 master weights and optimiser state).  `cuda_graph`: replay the optimiser steps from a CUDA graph (`_GraphedTraining`);
        False runs the same steps eagerly (same minibatches, same arithmetic).  `trainer_share`: fraction of the games rank 0 plays
        (`distributed.shard_range`); None = equal shards.  `save_every_n_iterations` > 0: after every n-th round of games rank 0
        writes the replay deque as `<save_dir>/episodes_iter{N}.json` (`DataModule._save_episodes`, datamodule.py:71-80,109-112;
        default directory "episodes", datamodule.py:63) and, after that iteration's training, a Lightning-shaped checkpoint
        `<save_dir>/model_iter{N}.ckpt` (`{"state_dict", "hyper_parameters", "epoch", "global_step"}`, the reference's
        `ModelCheckpoint(every_n_epochs=...)`, trainer.py:66-70; read back with `Model.load_from_checkpoint`, scripts/play.py:19).
        `root_noise` (`search.RootNoise`) and `sampling_moves` (`EpisodeGenerator`): AlphaZero's self-play exploration, off by
        default.  Each rank's noise is keyed by the global index of its games (`slot_offset` = the first slot of its shard), so
        the draws do not depend on how the games are sharded.
        `symmetric`: self-play evaluates every leaf in its canonical orientation under the left-right mirror
        (`AlphaZeroSearch(symmetric=True)`).  `mirror_augment`: each epoch trains a random half of the samples in their mirror
        image (`_GraphedTraining`).  Both off by default.
        `subtree_reuse`: each self-play move keeps the played child's subtree for the next search (`AlphaZeroSearch(subtree_reuse=)`:
        True = max_root_visits of 4 simulations_per_episode, an int = max_root_visits); off by default.  The replay buffer then divides
        each sample's visit counts by their sum (`ReplayBuffer(subtree_reuse=True)`).
        `playout_cap` (`search.PlayoutCap`): most self-play moves get a fast search and only the full searches become samples
        (`AlphaZeroSearch(playout_cap=)`); off by default.  Like `root_noise`, its `slot_offset` is set to the rank's first game.
        `forced_playouts` (`search.ForcedPlayouts`): self-play forces root visits and records the pruned counts
        (`AlphaZeroSearch(forced_playouts=)`); off by default.  Pruned counts no longer sum to N - 1, so the replay buffer then divides
        each sample's counts by their sum, as for subtree reuse.
        `openings` (`openings.Openings`): self-play games start from opening positions (`EpisodeGenerator(openings=)`); off by
        default.  Like `root_noise`, its `slot_offset` is set to the rank's first game, so a sharded run starts the same games."""
        import threading

        world = dist.get_world_size() if dist.is_initialized() else 1
        rank = dist.get_rank() if dist.is_initialized() else 0
        # the whole shard table is checked identically on every rank BEFORE any collective: a rank that raised alone would leave
        # the others waiting in the all-gather
        shards = [shard_range(episodes_per_iter, r, world, trainer_share) for r in range(world)]
        if any(h == l for l, h in shards):
            raise ValueError(f"every rank needs at least one game: shards {shards} (episodes_per_iter={episodes_per_iter}, "
                             f"world={world}, trainer_share={trainer_share})")
        lo, hi = shards[rank]
        model = self.model.to(self.device)
        kw = {} if inference_dtype is None else dict(inference_dtype=inference_dtype)
        if root_noise is not None:
            kw["root_noise"] = dataclasses.replace(root_noise, slot_offset=lo)
        if symmetric:
            kw["symmetric"] = True
        if subtree_reuse:
            kw["subtree_reuse"] = subtree_reuse
        if playout_cap is not None:
            kw["playout_cap"] = dataclasses.replace(playout_cap, slot_offset=lo)
        if forced_playouts is not None:
            kw["forced_playouts"] = forced_playouts
        gen = EpisodeGenerator(model=model, num_simulations=simulations_per_episode, num_episodes=hi - lo,
                               game_initial_state=initial_state, device=self.device_index, sampling_moves=sampling_moves,
                               openings=None if openings is None else dataclasses.replace(openings, slot_offset=lo), **kw)
        replay = ReplayBuffer(buffer_size, simulations_per_episode, self.device, subtree_reuse="subtree_reuse" in kw or "forced_playouts" in kw)
        opt = model.configure_optimizers()
        for group in opt.param_groups:  # Adam's step counter on the device, so that optimiser steps can be captured
            group["capturable"] = True
        g = torch.Generator().manual_seed(seed)
        steps = _GraphedTraining(model, opt, batch_size, precision, self.device, mirror_augment=mirror_augment)
        play_stream = torch.cuda.Stream(device=self.device)
        box: dict = {}

        def play():  # the generator thread (EpisodeGeneratorThread.run, datamodule.py:24-30)
            try:
                torch.cuda.set_device(self.device)
                t = time.perf_counter()
                local = None
                with torch.cuda.stream(play_stream):
                    for batch in gen.generate_batches(quota=hi - lo):
                        local = batch if local is None else _concat(local, batch)
                    play_stream.synchronize()
                box["episodes"], box["selfplay_s"], box["error"] = local, time.perf_counter() - t, None
            except BaseException as exc:  # surfaced on the main thread
                box["error"] = exc

        def start():
            # the inference weights were (re)built on this thread's current stream; the games run on play_stream
            play_stream.wait_stream(torch.cuda.current_stream(self.device))
            th = threading.Thread(target=play, daemon=True)
            th.start()
            return th

        thread = start() if overlap else None
        for it in range(num_iterations):
            t0 = time.perf_counter()
            if overlap:
                thread.join()
            else:
                play()
            if box.get("error") is not None:
                raise box["error"]
            local, selfplay_s = box["episodes"], box["selfplay_s"]
            t1 = time.perf_counter()
            if world > 1:
                # one collective: every rank contributes exactly its shard's quota of episodes, of at most 42 samples each
                cap_e = max(h - l for l, h in shards)
                merged = all_gather_episodes(_to_device(local, self.device), slot_offset=lo, capacity=(cap_e, 42 * cap_e))
                replay.extend({k: merged[k] for k in ("ep_len", "ep_offset", "ep_outcome", "s_bb0", "s_bb1", "s_player", "s_counts")})
            else:
                replay.extend(local)
            t2 = time.perf_counter()
            saving = save_every_n_iterations > 0 and rank == 0 and (it + 1) % save_every_n_iterations == 0
            if saving:
                import os

                from .episode import episodes_from_batch, save_episodes

                os.makedirs(save_dir or "episodes", exist_ok=True)
                save_episodes(episodes_from_batch(replay.to_episode_batch(), simulations_per_episode),
                              os.path.join(save_dir or "episodes", f"episodes_iter{it + 1}.json"))
            # weight sync, then the next iteration's games start and overlap the training below
            nbytes = broadcast_weights(model, src=0) if world > 1 else 0
            gen.update_inference_model(model)
            if overlap and it + 1 < num_iterations:
                thread = start()
            loss_sum, n_steps = None, 0
            if rank == 0:
                model.train()
                loss_sum, n_steps = steps.run(replay, epochs_per_iter, g, use_graph=cuda_graph)
                model.eval()
            torch.cuda.current_stream(self.device).synchronize()
            if saving:  # the reference's ModelCheckpoint file shape (trainer.py:66-70), readable by Model.load_from_checkpoint
                gstep = sum(h["optimizer_steps"] for h in self.history) + n_steps
                model.save_checkpoint(os.path.join(save_dir or "episodes", f"model_iter{it + 1}.ckpt"),
                                      epoch=(it + 1) * epochs_per_iter, global_step=gstep)
            t3 = time.perf_counter()
            self.history.append(dict(iteration=it, episodes=len(replay), samples=replay.num_samples, selfplay_s=selfplay_s,
                                     wait_for_selfplay_s=t1 - t0, gather_s=t2 - t1, train_s=t3 - t2, weight_bytes=nbytes,
                                     optimizer_steps=n_steps, graph_replays=steps.replays,
                                     loss=float(loss_sum) / n_steps if n_steps else None))
        if world > 1:  # everyone ends with the trainer rank's final weights
            broadcast_weights(model, src=0)
        gen.update_inference_model(model)
        return self.history


def _concat(a, b):
    import numpy as np

    from .engine import EpisodeBatch

    off = np.concatenate([a.ep_offset, b.ep_offset + len(a.s_bb0)])
    return EpisodeBatch(np.concatenate([a.ep_slot, b.ep_slot]), np.concatenate([a.ep_step, b.ep_step]), np.concatenate([a.ep_len, b.ep_len]),
                        off, np.concatenate([a.ep_outcome, b.ep_outcome]), np.concatenate([a.s_bb0, b.s_bb0]),
                        np.concatenate([a.s_bb1, b.s_bb1]), np.concatenate([a.s_player, b.s_player]), np.concatenate([a.s_counts, b.s_counts]))


def _to_device(b, device):
    import numpy as np

    d = dict(ep_slot=b.ep_slot, ep_step=b.ep_step, ep_len=b.ep_len, ep_offset=b.ep_offset, ep_outcome=b.ep_outcome,
             s_bb0=b.s_bb0.view(np.int64), s_bb1=b.s_bb1.view(np.int64), s_player=b.s_player, s_counts=b.s_counts)
    return {k: torch.from_numpy(np.ascontiguousarray(v)).to(device) for k, v in d.items()}
