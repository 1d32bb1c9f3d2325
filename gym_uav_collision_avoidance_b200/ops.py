"""PyTorch custom ops over the C-ABI (include/uavca.h).

Each op hands `tensor.data_ptr()` of CUDA tensors and torch's current CUDA stream to the shim; nothing is
copied and nothing runs on the CPU.  Outputs are written into caller-provided tensors (``mutates_args``) so the
observation / reward / done buffers are handed zero-copy to the policy and the replay buffer, and so the ops
can be captured in CUDA graphs.  The handle travels as an integer (the `uavca_handle*`).
"""
from __future__ import annotations

from typing import Optional

import torch

from . import _capi


def _stream(t: torch.Tensor) -> int:
    return torch.cuda.current_stream(t.device).cuda_stream


def _ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


def _need_cuda(*tensors: Optional[torch.Tensor]) -> None:
    for t in tensors:
        if t is not None and not t.is_cuda:
            raise _capi.UavcaError("uavca ops take CUDA tensors only (there is no CPU fallback)")
        if t is not None and not t.is_contiguous():
            raise _capi.UavcaError("uavca ops take contiguous tensors")


@torch.library.custom_op("uavca::step_multi", mutates_args=("state", "obs", "reward", "done", "final_obs", "reset_mask"))
def step_multi(handle: int, state: torch.Tensor, action: torch.Tensor, action_mode: int, evaluate: bool,
               obs: torch.Tensor, reward: torch.Tensor, done: torch.Tensor, final_obs: Optional[torch.Tensor],
               reset_mask: Optional[torch.Tensor]) -> None:
    """MultiUAVWorld2D.step for B envs x N UAVs (multi_uav_world_2d.py:177-241)."""
    _need_cuda(state, action, obs, reward, done, final_obs, reset_mask)
    _capi.check(_capi.load().uavca_step_multi(handle, state.data_ptr(), action.data_ptr(), action_mode, int(evaluate),
                                              obs.data_ptr(), reward.data_ptr(), done.data_ptr(), _ptr(final_obs),
                                              _ptr(reset_mask), _stream(state)), "uavca_step_multi")


@torch.library.custom_op("uavca::step_single",
                         mutates_args=("state", "obs", "reward", "done", "distance", "final_obs", "reset_mask"))
def step_single(handle: int, state: torch.Tensor, action: torch.Tensor, action_mode: int, obs: torch.Tensor,
                reward: torch.Tensor, done: torch.Tensor, distance: Optional[torch.Tensor],
                final_obs: Optional[torch.Tensor], reset_mask: Optional[torch.Tensor]) -> None:
    """UAVWorld2D.step for B envs (uav_world_2d.py:137-173)."""
    _need_cuda(state, action, obs, reward, done, distance, final_obs, reset_mask)
    _capi.check(_capi.load().uavca_step_single(handle, state.data_ptr(), action.data_ptr(), action_mode, obs.data_ptr(),
                                               reward.data_ptr(), done.data_ptr(), _ptr(distance), _ptr(final_obs),
                                               _ptr(reset_mask), _stream(state)), "uavca_step_single")


@torch.library.custom_op("uavca::rollout", mutates_args=("state", "obs", "reward", "done", "action_out", "final_obs",
                                                        "reset_mask", "distance"))
def rollout(handle: int, state: torch.Tensor, steps: int, action_block: Optional[torch.Tensor], action_mode: int,
            evaluate: bool, action_seed: int, step0: int, obs: torch.Tensor, reward: torch.Tensor, done: torch.Tensor,
            action_out: Optional[torch.Tensor], final_obs: Optional[torch.Tensor], reset_mask: Optional[torch.Tensor],
            distance: Optional[torch.Tensor]) -> None:
    """K = `steps` consecutive env steps in one launch (run.py:10-16 / run_multi.py:10-16); outputs are [K, ...] blocks."""
    _need_cuda(state, action_block, obs, reward, done, action_out, final_obs, reset_mask, distance)
    _capi.check(_capi.load().uavca_rollout(handle, state.data_ptr(), steps, _ptr(action_block), action_mode, int(evaluate),
                                           action_seed, step0, obs.data_ptr(), reward.data_ptr(), done.data_ptr(),
                                           _ptr(action_out), _ptr(final_obs), _ptr(reset_mask), _ptr(distance),
                                           _stream(state)), "uavca_rollout")


@torch.library.custom_op("uavca::sample_actions", mutates_args=("out",))
def sample_actions(handle: int, action_seed: int, step: int, out: torch.Tensor) -> None:
    """The policy-space actions uavca::rollout draws at global step `step` (env.action_space.sample() for every UAV)."""
    _need_cuda(out)
    _capi.check(_capi.load().uavca_sample_actions(handle, action_seed, step, out.data_ptr(), _stream(out)),
                "uavca_sample_actions")


@torch.library.custom_op("uavca::reset", mutates_args=("state", "obs"))
def reset(handle: int, state: torch.Tensor, mask: Optional[torch.Tensor], obs: torch.Tensor) -> None:
    """reset() of all (mask=None) or the masked envs (multi_uav_world_2d.py:116-175, uav_world_2d.py:119-135)."""
    _need_cuda(state, mask, obs)
    _capi.check(_capi.load().uavca_reset(handle, state.data_ptr(), _ptr(mask), obs.data_ptr(), _stream(state)),
                "uavca_reset")


@torch.library.custom_op("uavca::observe", mutates_args=("obs",))
def observe(handle: int, state: torch.Tensor, obs: torch.Tensor) -> None:
    """_get_obs() of the current state (multi_uav_world_2d.py:60-109, uav_world_2d.py:77-112)."""
    _need_cuda(state, obs)
    _capi.check(_capi.load().uavca_observe(handle, state.data_ptr(), obs.data_ptr(), _stream(state)), "uavca_observe")


@torch.library.custom_op("uavca::map_action", mutates_args=("out",))
def map_action(handle: int, action: torch.Tensor, action_mode: int, out: torch.Tensor) -> None:
    """Caller-side action mapping (test_sac_multi.py:77-80, test_pytorch_multi.py:80)."""
    _need_cuda(action, out)
    _capi.check(_capi.load().uavca_map_action(handle, action.data_ptr(), action_mode, out.data_ptr(), _stream(action)),
                "uavca_map_action")


@torch.library.custom_op("uavca::stats", mutates_args=("out8",))
def stats(handle: int, state: torch.Tensor, out8: torch.Tensor) -> None:
    """Episode statistics (env.steps / target_reach_count / collision_count, multi_uav_world_2d.py:166-168)."""
    _need_cuda(state, out8)
    _capi.check(_capi.load().uavca_stats(handle, state.data_ptr(), out8.data_ptr(), _stream(state)), "uavca_stats")


@torch.library.custom_op("uavca::replay_push",
                         mutates_args=("ring_obs", "ring_action", "ring_reward", "ring_next_obs", "ring_mask"))
def replay_push(obs: torch.Tensor, action: torch.Tensor, reward: torch.Tensor, next_obs: torch.Tensor, done: torch.Tensor,
                ring_obs: torch.Tensor, ring_action: torch.Tensor, ring_reward: torch.Tensor, ring_next_obs: torch.Tensor,
                ring_mask: torch.Tensor, head: int) -> None:
    """Append M transitions to a device replay ring at slot `head` (ReplayMemory.push,
    pytorch_sac_temp/replay_memory.py:15-19, for all B*N transitions of a step at once)."""
    _need_cuda(obs, action, reward, next_obs, done, ring_obs, ring_action, ring_reward, ring_next_obs, ring_mask)
    M = reward.numel()
    _capi.check(_capi.load().uavca_replay_push(obs.data_ptr(), action.data_ptr(), reward.data_ptr(), next_obs.data_ptr(),
                                               done.data_ptr(), M, obs.numel() // max(M, 1), action.numel() // max(M, 1),
                                               ring_obs.data_ptr(), ring_action.data_ptr(), ring_reward.data_ptr(),
                                               ring_next_obs.data_ptr(), ring_mask.data_ptr(), ring_reward.numel(), head,
                                               _stream(obs)), "uavca_replay_push")


@torch.library.custom_op("uavca::replay_push_dev",
                         mutates_args=("ring_obs", "ring_action", "ring_reward", "ring_next_obs", "ring_mask", "ring_meta"))
def replay_push_dev(obs: torch.Tensor, action: torch.Tensor, reward: torch.Tensor, next_obs: torch.Tensor, done: torch.Tensor,
                    ring_obs: torch.Tensor, ring_action: torch.Tensor, ring_reward: torch.Tensor, ring_next_obs: torch.Tensor,
                    ring_mask: torch.Tensor, ring_meta: torch.Tensor) -> None:
    """The same append with the ring head on the device (`ring_meta` int64[4]: head, scratch, size): safe to replay from
    a CUDA graph, every replay appends where the previous one stopped."""
    _need_cuda(obs, action, reward, next_obs, done, ring_obs, ring_action, ring_reward, ring_next_obs, ring_mask, ring_meta)
    M = reward.numel()
    _capi.check(_capi.load().uavca_replay_push_dev(obs.data_ptr(), action.data_ptr(), reward.data_ptr(), next_obs.data_ptr(),
                                                   done.data_ptr(), M, obs.numel() // max(M, 1), action.numel() // max(M, 1),
                                                   ring_obs.data_ptr(), ring_action.data_ptr(), ring_reward.data_ptr(),
                                                   ring_next_obs.data_ptr(), ring_mask.data_ptr(), ring_reward.numel(),
                                                   ring_meta.data_ptr(), _stream(obs)), "uavca_replay_push_dev")


@torch.library.custom_op("uavca::replay_sample",
                         mutates_args=("out_obs", "out_action", "out_reward", "out_next_obs", "out_mask", "out_index"))
def replay_sample(ring_obs: torch.Tensor, ring_action: torch.Tensor, ring_reward: torch.Tensor, ring_next_obs: torch.Tensor,
                  ring_mask: torch.Tensor, ring_meta: torch.Tensor, seed: int, draw: int, recency_weighted: bool,
                  out_obs: torch.Tensor, out_action: torch.Tensor, out_reward: torch.Tensor, out_next_obs: torch.Tensor,
                  out_mask: torch.Tensor, out_index: Optional[torch.Tensor]) -> None:
    """`memory.sample(batch)` (pytorch_sac_temp/replay_memory.py:21-24) in one launch, slots drawn on the device."""
    _need_cuda(ring_obs, ring_action, ring_reward, ring_next_obs, ring_mask, ring_meta, out_obs, out_action, out_reward,
               out_next_obs, out_mask, out_index)
    cap, batch = ring_reward.numel(), out_reward.numel()
    _capi.check(_capi.load().uavca_replay_sample(ring_obs.data_ptr(), ring_action.data_ptr(), ring_reward.data_ptr(),
                                                 ring_next_obs.data_ptr(), ring_mask.data_ptr(), cap, ring_obs.numel() // cap,
                                                 ring_action.numel() // cap, ring_meta.data_ptr(), batch, seed, draw,
                                                 int(recency_weighted), out_obs.data_ptr(), out_action.data_ptr(),
                                                 out_reward.data_ptr(), out_next_obs.data_ptr(), out_mask.data_ptr(),
                                                 _ptr(out_index), _stream(ring_obs)), "uavca_replay_sample")


@torch.library.custom_op("uavca::replay_sample_nstep",
                         mutates_args=("out_obs", "out_action", "out_reward", "out_next_obs", "out_discount", "out_index"))
def replay_sample_nstep(ring_obs: torch.Tensor, ring_action: torch.Tensor, ring_reward: torch.Tensor,
                        ring_next_obs: torch.Tensor, ring_mask: torch.Tensor, ring_meta: torch.Tensor, seed: int, draw: int,
                        recency_weighted: bool, stride: int, n: int, gamma: float, out_obs: torch.Tensor,
                        out_action: torch.Tensor, out_reward: torch.Tensor, out_next_obs: torch.Tensor,
                        out_discount: torch.Tensor, out_index: Optional[torch.Tensor]) -> None:
    """The slots of `replay_sample` with n-step returns folded over up to `n` successors `stride` slots apart, in one
    launch (rule in include/uavca.h, uavca_replay_sample_nstep)."""
    _need_cuda(ring_obs, ring_action, ring_reward, ring_next_obs, ring_mask, ring_meta, out_obs, out_action, out_reward,
               out_next_obs, out_discount, out_index)
    cap, batch = ring_reward.numel(), out_reward.numel()
    _capi.check(_capi.load().uavca_replay_sample_nstep(ring_obs.data_ptr(), ring_action.data_ptr(), ring_reward.data_ptr(),
                                                       ring_next_obs.data_ptr(), ring_mask.data_ptr(), cap,
                                                       ring_obs.numel() // cap, ring_action.numel() // cap,
                                                       ring_meta.data_ptr(), batch, seed, draw, int(recency_weighted),
                                                       stride, n, float(gamma), out_obs.data_ptr(), out_action.data_ptr(),
                                                       out_reward.data_ptr(), out_next_obs.data_ptr(), out_discount.data_ptr(),
                                                       _ptr(out_index), _stream(ring_obs)), "uavca_replay_sample_nstep")


def _per_tree(tree: torch.Tensor, per_meta: Optional[torch.Tensor]) -> int:
    """Checks the sum-tree and per_meta tensors of prioritized replay; returns L."""
    if tree.dtype != torch.float64 or tree.dim() != 1 or tree.numel() < 2 or tree.numel() % 2:
        raise _capi.UavcaError("the priority tree is a 1-D float64 tensor of 2L elements")
    if per_meta is not None and (per_meta.dtype != torch.int64 or per_meta.numel() != 5):
        raise _capi.UavcaError("per_meta is an int64 tensor of 5 elements")
    return tree.numel() // 2


@torch.library.custom_op("uavca::per_sync", mutates_args=("tree", "per_meta"))
def per_sync(tree: torch.Tensor, per_meta: torch.Tensor, ring_meta: torch.Tensor, capacity: int) -> None:
    """Give the slots appended since the last sync the largest priority so far (one launch, no host sync)."""
    _need_cuda(tree, per_meta, ring_meta)
    L = _per_tree(tree, per_meta)
    _capi.check(_capi.load().uavca_per_sync(tree.data_ptr(), L, per_meta.data_ptr(), ring_meta.data_ptr(), capacity,
                                            _stream(tree)), "uavca_per_sync")


@torch.library.custom_op("uavca::per_update", mutates_args=("tree", "per_meta"))
def per_update(tree: torch.Tensor, per_meta: torch.Tensor, index: torch.Tensor, priority: torch.Tensor, capacity: int) -> None:
    """Set leaf index[j] to priority[j] (last occurrence wins) and form the ancestors again; an update with a bad index or
    priority is dropped whole on the device and counted in per_meta[4]."""
    _need_cuda(tree, per_meta, index, priority)
    L = _per_tree(tree, per_meta)
    if index.dtype != torch.int64 or priority.dtype != torch.float64 or index.numel() != priority.numel():
        raise _capi.UavcaError("per_update takes int64 indices and as many float64 priorities")
    _capi.check(_capi.load().uavca_per_update(tree.data_ptr(), L, capacity, per_meta.data_ptr(), index.data_ptr(),
                                              priority.data_ptr(), index.numel(), _stream(tree)), "uavca_per_update")


@torch.library.custom_op("uavca::per_sample", mutates_args=("tree", "out_obs", "out_action", "out_reward", "out_next_obs",
                                                           "out_mask", "out_index", "out_weight"))
def per_sample(ring_obs: torch.Tensor, ring_action: torch.Tensor, ring_reward: torch.Tensor, ring_next_obs: torch.Tensor,
               ring_mask: torch.Tensor, ring_meta: torch.Tensor, tree: torch.Tensor, batch: int, beta: float, seed: int,
               draw: int, out_obs: torch.Tensor, out_action: torch.Tensor, out_reward: torch.Tensor, out_next_obs: torch.Tensor,
               out_mask: torch.Tensor, out_index: torch.Tensor, out_weight: torch.Tensor) -> None:
    """Stratified proportional draw of `batch` slots from the sum-tree, gathered with importance weights, in one launch.
    (`tree` is listed as mutated: its element 0 is the launch's CTA ticket.)"""
    _need_cuda(ring_obs, ring_action, ring_reward, ring_next_obs, ring_mask, ring_meta, tree, out_obs, out_action,
               out_reward, out_next_obs, out_mask, out_index, out_weight)
    L = _per_tree(tree, None)
    if out_index.dtype != torch.int64 or out_weight.dtype != torch.float32 or out_index.numel() != batch or \
            out_weight.numel() != batch or out_reward.numel() != batch:
        raise _capi.UavcaError("per_sample: out_index int64 [batch], out_weight float32 [batch]")
    cap = ring_reward.numel()
    _capi.check(_capi.load().uavca_per_sample(ring_obs.data_ptr(), ring_action.data_ptr(), ring_reward.data_ptr(),
                                              ring_next_obs.data_ptr(), ring_mask.data_ptr(), cap, ring_obs.numel() // cap,
                                              ring_action.numel() // cap, ring_meta.data_ptr(), tree.data_ptr(), L, batch,
                                              float(beta), seed, draw, out_obs.data_ptr(), out_action.data_ptr(),
                                              out_reward.data_ptr(), out_next_obs.data_ptr(), out_mask.data_ptr(),
                                              out_index.data_ptr(), out_weight.data_ptr(), _stream(tree)), "uavca_per_sample")


@torch.library.custom_op("uavca::per_sample_nstep", mutates_args=("tree", "out_obs", "out_action", "out_reward",
                                                                 "out_next_obs", "out_discount", "out_index", "out_weight"))
def per_sample_nstep(ring_obs: torch.Tensor, ring_action: torch.Tensor, ring_reward: torch.Tensor,
                     ring_next_obs: torch.Tensor, ring_mask: torch.Tensor, ring_meta: torch.Tensor, tree: torch.Tensor,
                     batch: int, beta: float, stride: int, n: int, gamma: float, seed: int, draw: int,
                     out_obs: torch.Tensor, out_action: torch.Tensor, out_reward: torch.Tensor, out_next_obs: torch.Tensor,
                     out_discount: torch.Tensor, out_index: torch.Tensor, out_weight: torch.Tensor) -> None:
    """The slots and weights of `per_sample` with n-step returns (include/uavca.h, uavca_per_sample_nstep), one launch.
    (`tree` is listed as mutated: its element 0 is the launch's CTA ticket.)"""
    _need_cuda(ring_obs, ring_action, ring_reward, ring_next_obs, ring_mask, ring_meta, tree, out_obs, out_action,
               out_reward, out_next_obs, out_discount, out_index, out_weight)
    L = _per_tree(tree, None)
    if out_index.dtype != torch.int64 or out_weight.dtype != torch.float32 or out_index.numel() != batch or \
            out_weight.numel() != batch or out_reward.numel() != batch:
        raise _capi.UavcaError("per_sample_nstep: out_index int64 [batch], out_weight float32 [batch]")
    cap = ring_reward.numel()
    _capi.check(_capi.load().uavca_per_sample_nstep(ring_obs.data_ptr(), ring_action.data_ptr(), ring_reward.data_ptr(),
                                                    ring_next_obs.data_ptr(), ring_mask.data_ptr(), cap,
                                                    ring_obs.numel() // cap, ring_action.numel() // cap,
                                                    ring_meta.data_ptr(), tree.data_ptr(), L, batch, float(beta), stride, n,
                                                    float(gamma), seed, draw, out_obs.data_ptr(), out_action.data_ptr(),
                                                    out_reward.data_ptr(), out_next_obs.data_ptr(), out_discount.data_ptr(),
                                                    out_index.data_ptr(), out_weight.data_ptr(), _stream(tree)),
                "uavca_per_sample_nstep")


@torch.library.custom_op("uavca::step_multi_replay",
                         mutates_args=("state", "obs", "reward", "done", "final_obs", "reset_mask", "ring_obs", "ring_action",
                                       "ring_reward", "ring_next_obs", "ring_mask", "ring_meta"))
def step_multi_replay(handle: int, state: torch.Tensor, action: torch.Tensor, action_mode: int, evaluate: bool,
                      prev_obs: torch.Tensor, obs: torch.Tensor, reward: torch.Tensor, done: torch.Tensor,
                      final_obs: Optional[torch.Tensor], reset_mask: Optional[torch.Tensor], ring_obs: torch.Tensor,
                      ring_action: torch.Tensor, ring_reward: torch.Tensor, ring_next_obs: torch.Tensor,
                      ring_mask: torch.Tensor, ring_meta: torch.Tensor) -> None:
    """MultiUAVWorld2D.step and the N `memory.push` calls that follow it in a training step (test_sac_multi.py:99-103) as
    ONE launch: the step kernel appends every UAV's transition to the device replay ring itself."""
    _need_cuda(state, action, prev_obs, obs, reward, done, final_obs, reset_mask, ring_obs, ring_action, ring_reward,
               ring_next_obs, ring_mask, ring_meta)
    _capi.check(_capi.load().uavca_step_multi_replay(handle, state.data_ptr(), action.data_ptr(), action_mode, int(evaluate),
                                                     prev_obs.data_ptr(), obs.data_ptr(), reward.data_ptr(), done.data_ptr(),
                                                     _ptr(final_obs), _ptr(reset_mask), ring_obs.data_ptr(),
                                                     ring_action.data_ptr(), ring_reward.data_ptr(), ring_next_obs.data_ptr(),
                                                     ring_mask.data_ptr(), ring_reward.numel(), ring_meta.data_ptr(),
                                                     _stream(state)), "uavca_step_multi_replay")


@torch.library.custom_op("uavca::policy_act", mutates_args=("action", "head"))
def policy_act(obs: torch.Tensor, w1: torch.Tensor, w2: torch.Tensor, w2b: torch.Tensor, w3: torch.Tensor, w3b: torch.Tensor,
               noise: Optional[torch.Tensor], seed: int, counter: int, counter_dev: Optional[torch.Tensor],
               action: torch.Tensor, head: Optional[torch.Tensor]) -> None:
    """GaussianPolicy acting path (pytorch_sac_temp/model.py:74-101) for all rows of `obs` in one tcgen05 kernel.
    Weight operands are the fp16 packings described in include/uavca.h."""
    _need_cuda(obs, w1, w2, w2b, w3, w3b, noise, counter_dev, action, head)
    _capi.check(_capi.load().uavca_policy_act(obs.data_ptr(), obs.numel() // 10, w1.data_ptr(), w2.data_ptr(), w2b.data_ptr(),
                                              w3.data_ptr(), w3b.data_ptr(), _ptr(noise), seed, counter, _ptr(counter_dev),
                                              action.data_ptr(), _ptr(head), _stream(obs)), "uavca_policy_act")
