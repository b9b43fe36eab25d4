"""Device-resident replay buffer fed straight from the episode ring / all-gather.

Reference semantics (core/training/datamodule.py:57,114-130; models/base/model.py:76-82;
models/games/connect4/model.py:45-51): the buffer holds the last `buffer_size` EPISODES (a deque), the
training set is every sample of those episodes, inputs are `Model._states_to_tensor(states)`, policy
targets are dense [B,7] visit distributions (0 on illegal columns), value targets are [B,2] outcomes,
batches of 32, shuffled.  Here the samples stay on the GPU as bitboards + visit counts and are
expanded to planes by the `az_encode_states` kernel per minibatch.

Storage is flat: every `extend` call adds one chunk (the episode batch as it came off the ring or the
all-gather, samples contiguous per episode); the deque's eviction drops whole episodes from the front of the
oldest chunk by moving a pointer.  No per-episode Python objects: a 65536-game round is one chunk.
"""
from __future__ import annotations

from collections import deque

import numpy as np
import torch

from .engine import EpisodeBatch
from .game import rules_engine


class _Chunk:
    """One batch of finished episodes in arrival order; episodes [first, n) are still in the buffer."""

    def __init__(self, ep_len, ep_outcome, s_bb0, s_bb1, s_player, s_counts):
        self.ep_len, self.ep_outcome = ep_len, ep_outcome
        self.s_bb0, self.s_bb1, self.s_player, self.s_counts = s_bb0, s_bb1, s_player, s_counts
        self.lens = ep_len.tolist()  # host copy: eviction arithmetic without device syncs
        self.first = 0               # episodes evicted from the front
        self.first_sample = 0

    @property
    def num_episodes(self) -> int:
        return len(self.lens) - self.first

    @property
    def num_samples(self) -> int:
        return int(self.s_bb0.numel()) - self.first_sample

    def drop_front(self, k: int):
        self.first_sample += sum(self.lens[self.first:self.first + k])
        self.first += k


class ReplayBuffer:
    def __init__(self, buffer_size: int, num_simulations: int, device: torch.device | str = "cuda", *, subtree_reuse: bool = False):
        """`subtree_reuse`: the samples come from searches whose roots may have kept their subtree (`AlphaZeroSearch(subtree_reuse=)`),
        so a root holds N(c) + S visits: policy targets are the counts over each row's own sum (root visits - 1) instead of over
        S - 1.  Rows of fresh roots sum to S - 1 and get the same bits either way."""
        self.buffer_size = int(buffer_size)
        self.num_simulations = int(num_simulations)
        self.subtree_reuse = bool(subtree_reuse)
        self.device = torch.device(device)
        self.chunks: deque[_Chunk] = deque()

    def __len__(self) -> int:
        return sum(c.num_episodes for c in self.chunks)

    @property
    def num_samples(self) -> int:
        return sum(c.num_samples for c in self.chunks)

    def extend(self, batch: EpisodeBatch | dict):
        """Append finished episodes in order (`buffer.append(episode)`, datamodule.py:29-30); the deque keeps the last
        `buffer_size` of them.  Episodes must be stored with their samples back to back in episode order.  `buffer_size` counts
        episodes, empty ones included (an episode of `AlphaZeroSearch(playout_cap=)` self-play may have no samples)."""
        if isinstance(batch, EpisodeBatch):
            d = dict(ep_len=batch.ep_len, ep_offset=batch.ep_offset, ep_outcome=batch.ep_outcome, s_bb0=batch.s_bb0.view(np.int64),
                     s_bb1=batch.s_bb1.view(np.int64), s_player=batch.s_player, s_counts=batch.s_counts)
            d = {k: torch.from_numpy(np.ascontiguousarray(v)).to(self.device) for k, v in d.items()}
        else:
            d = {k: v.to(self.device) for k, v in batch.items()}
        if d["ep_len"].numel() == 0:
            return
        ep_len = d["ep_len"].to(torch.int64)
        expect = torch.cumsum(ep_len, 0) - ep_len
        if not torch.equal(d["ep_offset"].to(torch.int64), expect):  # e.g. a batch sorted by (step, slot): regroup the samples
            idx = torch.repeat_interleave(d["ep_offset"].to(torch.int64) - expect, ep_len) + torch.arange(int(ep_len.sum()), device=self.device)
            d = dict(d, s_bb0=d["s_bb0"][idx], s_bb1=d["s_bb1"][idx], s_player=d["s_player"][idx], s_counts=d["s_counts"][idx])
        self.chunks.append(_Chunk(ep_len, d["ep_outcome"], d["s_bb0"], d["s_bb1"], d["s_player"], d["s_counts"]))
        excess = len(self) - self.buffer_size
        while excess > 0:
            head = self.chunks[0]
            k = min(excess, head.num_episodes)
            head.drop_front(k)
            if head.num_episodes == 0:
                self.chunks.popleft()
            excess -= k

    def tensors(self):
        """Flatten the deque (datamodule.py:114-122) -> (bb0, bb1, player, policy_target[B,7], value_target[B,2])."""
        cs = list(self.chunks)
        bb0 = torch.cat([c.s_bb0[c.first_sample:] for c in cs])
        bb1 = torch.cat([c.s_bb1[c.first_sample:] for c in cs])
        pl = torch.cat([c.s_player[c.first_sample:] for c in cs])
        counts = torch.cat([c.s_counts[c.first_sample:] for c in cs]).to(torch.float32)
        policy = counts / float(self.num_simulations - 1)  # Node.improved_policy (node.py:27), fp32 like torch.zeros(...)[i, col] = prob
        if self.subtree_reuse:
            # counts / (root visits - 1) = over the row's sum, more than S - 1 for a root that kept its subtree.  Rows that sum to
            # S - 1 keep the scalar division above (on CUDA a multiply by the fp32 reciprocal): the same bits as without reuse
            rows = counts.sum(1, keepdim=True)
            policy = torch.where(rows == float(self.num_simulations - 1), policy, counts / rows)
        value = torch.cat([torch.repeat_interleave(c.ep_outcome[c.first:].to(torch.float32), c.ep_len[c.first:], dim=0) for c in cs])
        return bb0, bb1, pl, policy, value

    def to_episode_batch(self) -> EpisodeBatch:
        """The deque's content, oldest episode first, as flat host arrays (what `DataModule._save_episodes` iterates over,
        datamodule.py:71-80).  Slots and steps of the episodes are not kept by the buffer: -1 / 0."""
        cs = list(self.chunks)
        if not cs:
            z = np.zeros(0, np.int64)
            return EpisodeBatch(z.astype(np.int32), z.astype(np.int32), z.astype(np.int32), z, np.zeros((0, 2), np.int8),
                                z.astype(np.uint64), z.astype(np.uint64), z.astype(np.uint8), np.zeros((0, 7), np.int32))
        ep_len = torch.cat([c.ep_len[c.first:] for c in cs]).cpu().numpy().astype(np.int32)
        outcome = torch.cat([c.ep_outcome[c.first:] for c in cs]).cpu().numpy().astype(np.int8)
        bb0 = torch.cat([c.s_bb0[c.first_sample:] for c in cs]).cpu().numpy().view(np.uint64)
        bb1 = torch.cat([c.s_bb1[c.first_sample:] for c in cs]).cpu().numpy().view(np.uint64)
        pl = torch.cat([c.s_player[c.first_sample:] for c in cs]).cpu().numpy().astype(np.uint8)
        counts = torch.cat([c.s_counts[c.first_sample:] for c in cs]).cpu().numpy().astype(np.int32)
        off = np.cumsum(ep_len, dtype=np.int64) - ep_len
        n = ep_len.shape[0]
        return EpisodeBatch(np.full(n, -1, np.int32), np.zeros(n, np.int32), ep_len, off, outcome, bb0, bb1, pl, counts)

    def batches(self, layout: int, batch_size: int = 32, shuffle: bool = True, generator: torch.Generator | None = None,
                mirror: bool = False):
        """Yield (x, policy_target, value_target) minibatches on the device (DataLoader(batch 32, shuffle), datamodule.py:124-130).
        `mirror`: one Bernoulli(1/2) flag per sample, drawn after the permutation from `generator`; flagged samples come as their
        left-right mirror image (bitboards through `az_mirror_states`, policy target columns reversed)."""
        bb0, bb1, pl, policy, value = self.tensors()
        n = bb0.numel()
        perm = torch.randperm(n, generator=generator).to(self.device) if shuffle else torch.arange(n, device=self.device)
        # one gather per epoch instead of five per minibatch: the shuffled set is materialised once, minibatches are views
        bb0, bb1, pl, policy, value = bb0[perm], bb1[perm], pl[perm], policy[perm], value[perm]
        eng = rules_engine()
        if mirror:
            flip = torch.randint(0, 2, (n,), generator=generator, dtype=torch.uint8).to(self.device)
            bb0, bb1 = eng.mirror_states(bb0, bb1, flip, out=(bb0, bb1))
            policy = torch.where(flip.bool().unsqueeze(1), policy.flip(1), policy)
        for i in range(0, n, batch_size):
            x = eng.encode_states(bb0[i:i + batch_size], bb1[i:i + batch_size], pl[i:i + batch_size], layout)
            yield x, policy[i:i + batch_size], value[i:i + batch_size]
