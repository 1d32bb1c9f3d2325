"""Device-resident replay ring buffer: the zero-copy hand-off of step outputs to the learner side.

Replaces the reference's host-side buffers — `ReplayMemory` (pytorch_sac_temp/replay_memory.py:7-24: python list
of tuples, `random.sample` + `np.stack` per batch) and `buffer_tensor.ReplayBuffer` (pytorch_ddpg/buffer_tensor.py:
19-92: deque of per-item CUDA tensors, recency-weighted sampling) — with five preallocated CUDA tensors.  A step's
`B*N` transitions are appended by ONE kernel (`uavca_replay_push`) straight from the env's output tensors, with
`mask = float(not done)` as the training loops store it (test_sac_multi.py:101-103).
"""
from __future__ import annotations

from typing import Optional

import torch

from . import ops


class DeviceReplay:
    def __init__(self, capacity: int, obs_dim: int, act_dim: int = 2, device="cuda", seed: Optional[int] = None):
        self.capacity, self.obs_dim, self.act_dim = int(capacity), int(obs_dim), int(act_dim)
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise ValueError("DeviceReplay lives on a CUDA device")
        kw = dict(dtype=torch.float32, device=self.device)
        self.state = torch.zeros((capacity, obs_dim), **kw)
        self.action = torch.zeros((capacity, act_dim), **kw)
        self.reward = torch.zeros(capacity, **kw)
        self.next_state = torch.zeros((capacity, obs_dim), **kw)
        self.mask = torch.zeros(capacity, **kw)
        # ring head and fill level live ON THE DEVICE (int64: head, scratch, size, spare): the append kernel reads and
        # advances them itself, so an acting step captured in a CUDA graph appends where the previous replay stopped
        self.meta = torch.zeros(4, dtype=torch.int64, device=self.device)
        self.gen = torch.Generator(device=self.device)
        if seed is not None:
            self.gen.manual_seed(seed)
        self._sample_seed, self._draws = int(seed if seed is not None else 0x5A3B1E) & (2 ** 63 - 1), 0  # sample_fused

    @property
    def position(self) -> int:
        """Next slot to write (ReplayMemory.position); reading it synchronises with the device."""
        return int(self.meta[0].item())

    @property
    def size(self) -> int:
        return int(self.meta[2].item())

    def __len__(self) -> int:
        return self.size

    def push(self, state: torch.Tensor, action: torch.Tensor, reward: torch.Tensor, next_state: torch.Tensor,
             done: torch.Tensor) -> None:
        """Append every transition of a step: tensors of shape [..., obs_dim] / [..., act_dim] / [...] (e.g. the env's
        [B, N, 10] obs, [B, N, 2] policy action, [B, N] reward and uint8 done).  One kernel launch, no host sync."""
        M = reward.numel()
        if M > self.capacity:
            raise ValueError(f"{M} transitions do not fit a ring of {self.capacity}")
        if state.numel() != M * self.obs_dim or next_state.numel() != M * self.obs_dim or action.numel() != M * self.act_dim:
            raise ValueError("transition tensors disagree on the number of transitions")
        if done.dtype == torch.bool:
            done = done.view(torch.uint8)
        ops.replay_push_dev(state.contiguous(), action.contiguous(), reward.contiguous(), next_state.contiguous(),
                            done.contiguous(), self.state, self.action, self.reward, self.next_state, self.mask, self.meta)

    def sample_fused(self, batch_size: int, recency_weighted: bool = False, out=None, want_index: bool = False):
        """`memory.sample(batch_size)` in ONE launch with no host synchronisation (`uavca_replay_sample`): the slots are
        drawn on the device from Philox4x32-10 keyed by (seed, sample, draws so far + appends so far) against the head and
        fill level in `self.meta`, so a learner step captured in a CUDA graph keeps sampling fresh transitions as the ring
        grows.  Returns (state, action, reward, next_state, mask[, index]); `out` reuses a previous result's tensors.
        Uniform slot: (x * size) >> 32 of a 32-bit draw x; recency-weighted: age = floor(sqrt((x + 0.5) / 2^32) * size),
        at most size - 1, counted from the oldest slot (`head` once the ring is full).  An empty ring cannot raise here
        without a host synchronisation: every slot is 0 and the batch holds ring row 0 (zeros until the first append)."""
        if out is None:
            kw = dict(dtype=torch.float32, device=self.device)
            out = (torch.empty((batch_size, self.obs_dim), **kw), torch.empty((batch_size, self.act_dim), **kw),
                   torch.empty(batch_size, **kw), torch.empty((batch_size, self.obs_dim), **kw), torch.empty(batch_size, **kw))
            if want_index:
                out = out + (torch.empty(batch_size, dtype=torch.int64, device=self.device),)
        idx = out[5] if len(out) > 5 else None
        ops.replay_sample(self.state, self.action, self.reward, self.next_state, self.mask, self.meta, self._sample_seed,
                          self._draws, bool(recency_weighted), out[0], out[1], out[2], out[3], out[4], idx)
        self._draws += 1
        return out

    def sample(self, batch_size: int, recency_weighted: bool = False):
        """-> (state [b,obs], action [b,act], reward [b], next_state [b,obs], mask [b]) as `memory.sample` returns them
        (pytorch_sac_temp/sac.py:48).  Uniform with replacement, or with probability rising linearly with recency
        (the `unbalance_p` scheme of pytorch_ddpg/buffer_tensor.py:78-87: p_i ~ i + 1/2 over insertion order)."""
        head, size = (int(v) for v in self.meta[[0, 2]].tolist())
        if size == 0:
            raise ValueError("empty replay buffer")
        if recency_weighted:
            u = torch.rand(batch_size, generator=self.gen, device=self.device)
            age = (u.sqrt() * size).long().clamp_(max=size - 1)  # inverse CDF of p_i ~ i + 1/2
            oldest = head if size == self.capacity else 0
            idx = (age + oldest) % self.capacity
        else:
            idx = torch.randint(0, size, (batch_size,), generator=self.gen, device=self.device)
        return self.state[idx], self.action[idx], self.reward[idx], self.next_state[idx], self.mask[idx]
