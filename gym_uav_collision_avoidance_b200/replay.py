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

    def sample_nstep(self, batch_size: int, n: int, gamma: float, stride: int, recency_weighted: bool = False, out=None,
                     want_index: bool = False):
        """`sample_fused` with n-step returns, in ONE launch with no host synchronisation (`uavca_replay_sample_nstep`):
        the same slots as `sample_fused` at the same draw count, then up to n - 1 successors `stride` slots apart
        (stride = envs * agents of the multi world, envs of the single world) are folded while they continue the
        episode.  Returns (state, action, reward_n, next_state_n, discount[, index]); the learner's target is
        reward_n + discount * V(next_state_n), which for n = 1 is r + gamma * mask * V.  The episode rule (include/uavca.h):
        a successor chains when the ring's mask is 1 and its observation equals the previous next observation bit for bit,
        so auto-resets, terminal transitions and the newest slots all end the return early with the matching gamma^k.
        Checked before the launch: 1 <= n <= 16, 1 <= stride <= capacity, 0 <= gamma <= 1.  Advances the draw count
        of `sample_fused`."""
        if out is None:
            kw = dict(dtype=torch.float32, device=self.device)
            out = (torch.empty((batch_size, self.obs_dim), **kw), torch.empty((batch_size, self.act_dim), **kw),
                   torch.empty(batch_size, **kw), torch.empty((batch_size, self.obs_dim), **kw), torch.empty(batch_size, **kw))
            if want_index:
                out = out + (torch.empty(batch_size, dtype=torch.int64, device=self.device),)
        idx = out[5] if len(out) > 5 else None
        ops.replay_sample_nstep(self.state, self.action, self.reward, self.next_state, self.mask, self.meta,
                                self._sample_seed, self._draws, bool(recency_weighted), int(stride), int(n), float(gamma),
                                out[0], out[1], out[2], out[3], out[4], idx)
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


PER_MAX_CAPACITY = 1 << 26  # UAVCA_PER_MAX_CAPACITY (include/uavca.h)


class PrioritizedDeviceReplay(DeviceReplay):
    """`DeviceReplay` with proportional prioritized sampling (Schaul et al. 2016, as the Ape-X learner uses it, Horgan et
    al. 2018): a float64 sum-tree over the ring's slots lives on the device next to the ring (`tree`, `per_meta`; layout in
    include/uavca.h).  New transitions enter with the largest priority set so far (1.0 at first); the learner draws
    stratified batches with importance weights and writes back (|td| + eps)^alpha.  Every call is one launch with no host
    synchronisation, so both the acting step and the learner step can be captured in CUDA graphs.  The inherited `sample` /
    `sample_fused` keep drawing uniformly or by recency.

    Keep the tree in step with the ring: `push` syncs after its append, and `BatchedMultiUAVWorld2D.step_replay` syncs after
    its fused append.  An append that reaches the ring another way must be followed by `sync()` before the next append;
    otherwise the sync cannot tell which slots are new, gives every filled slot the largest priority and counts the miss
    in `missed_syncs`."""

    def __init__(self, capacity: int, obs_dim: int, act_dim: int = 2, device="cuda", seed: Optional[int] = None,
                 alpha: float = 0.6, eps: float = 1e-6):
        if not 1 <= int(capacity) <= PER_MAX_CAPACITY:
            raise ValueError(f"a prioritized ring holds 1 to 2^26 slots, not {capacity}")
        super().__init__(capacity, obs_dim, act_dim, device, seed)
        self.alpha, self.eps = float(alpha), float(eps)
        self.leaves = 1 << (self.capacity - 1).bit_length()
        self.tree = torch.zeros(2 * self.leaves, dtype=torch.float64, device=self.device)
        # [0] appends and [1] head at the last sync, [2] largest priority so far (float64 bits), [3] missed syncs,
        # [4] refused updates
        self.per_meta = torch.zeros(5, dtype=torch.int64, device=self.device)
        self.per_meta[2:3].view(torch.float64).fill_(1.0)
        self._per_draws = 0

    def push(self, state: torch.Tensor, action: torch.Tensor, reward: torch.Tensor, next_state: torch.Tensor,
             done: torch.Tensor) -> None:
        """`DeviceReplay.push`, then `sync()`: the new transitions take the largest priority so far.  Two launches."""
        super().push(state, action, reward, next_state, done)
        self.sync()

    def sync(self) -> None:
        """Give every slot appended since the last sync the largest priority so far (one launch, no host sync)."""
        ops.per_sync(self.tree, self.per_meta, self.meta, self.capacity)

    def sample_prioritized(self, batch_size: int, beta: float, out=None):
        """Draw `batch_size` transitions with probability leaf / total, stratified over `batch_size` equal strata of the
        total, in ONE launch: -> (state, action, reward, next_state, mask, index int64, weight float32).  weight =
        (size * P)^-beta divided by the batch's largest.  `out` reuses a previous result's tensors.  `beta` is frozen into
        a captured CUDA graph; the draws of a captured learner step change as appends advance the ring (as `sample_fused`).
        An empty ring yields slot 0 with weight 0."""
        if out is None:
            kw = dict(dtype=torch.float32, device=self.device)
            out = (torch.empty((batch_size, self.obs_dim), **kw), torch.empty((batch_size, self.act_dim), **kw),
                   torch.empty(batch_size, **kw), torch.empty((batch_size, self.obs_dim), **kw), torch.empty(batch_size, **kw),
                   torch.empty(batch_size, dtype=torch.int64, device=self.device), torch.empty(batch_size, **kw))
        ops.per_sample(self.state, self.action, self.reward, self.next_state, self.mask, self.meta, self.tree, batch_size,
                       float(beta), self._sample_seed, self._per_draws, *out)
        self._per_draws += 1
        return out

    def sample_prioritized_nstep(self, batch_size: int, beta: float, n: int, gamma: float, stride: int, out=None):
        """`sample_prioritized` with the n-step returns of `DeviceReplay.sample_nstep`, in ONE launch: -> (state, action,
        reward_n, next_state_n, discount, index int64, weight float32).  The same slots and weights as
        `sample_prioritized` at the same draw count; write the n-step TD error of `index` back with `update_priorities`
        (the Ape-X learner).  Advances the draw count of `sample_prioritized`."""
        if out is None:
            kw = dict(dtype=torch.float32, device=self.device)
            out = (torch.empty((batch_size, self.obs_dim), **kw), torch.empty((batch_size, self.act_dim), **kw),
                   torch.empty(batch_size, **kw), torch.empty((batch_size, self.obs_dim), **kw), torch.empty(batch_size, **kw),
                   torch.empty(batch_size, dtype=torch.int64, device=self.device), torch.empty(batch_size, **kw))
        ops.per_sample_nstep(self.state, self.action, self.reward, self.next_state, self.mask, self.meta, self.tree,
                             batch_size, float(beta), int(stride), int(n), float(gamma), self._sample_seed, self._per_draws,
                             *out)
        self._per_draws += 1
        return out

    def update_priorities(self, index: torch.Tensor, td_error: torch.Tensor) -> None:
        """Set the priorities of slots `index` to (|td_error| + eps)^alpha, formed in float64 by torch; the last occurrence
        of a repeated slot wins.  An out-of-range index or a NaN / infinite error drops the whole update on the device
        (counted in `refused_updates`).  One launch beside torch's element-wise ops, no host sync."""
        index = index.reshape(-1)
        td = td_error.reshape(-1)
        if index.numel() != td.numel():
            raise ValueError(f"{index.numel()} slots but {td.numel()} TD errors")
        p = (td.detach().to(torch.float64).abs() + self.eps).pow(self.alpha)
        ops.per_update(self.tree, self.per_meta, index.to(torch.int64).contiguous(), p.contiguous(), self.capacity)

    @property
    def max_priority(self) -> float:
        """The largest priority set so far (synchronises with the device)."""
        return float(self.per_meta[2:3].view(torch.float64).item())

    @property
    def missed_syncs(self) -> int:
        """Syncs that found more than one append since the previous one (synchronises with the device)."""
        return int(self.per_meta[3].item())

    @property
    def refused_updates(self) -> int:
        """Priority updates dropped for an out-of-range slot or a negative / non-finite priority (synchronises)."""
        return int(self.per_meta[4].item())
