"""GPU: the 32-bit step offsets of the plain `uavca_rollout` launch at their bound.

The plain instance addresses every per-step output by one 32-bit element offset k * M + m, so the launcher runs it only
where the observation block's K * M * 10 floats stay below 2^31; a longer launch runs the general instance.  Both sides
of the bound are pinned bit for bit, outputs and final state:
  - just above it (K * M * 10 = 2.1495e9), the general instance against the same steps as two plain launches;
  - just below it (2.1443e9), the plain instance at its largest offsets against the general instance.
B = 65,536 envs of N = 8 UAVs (M = 2^19); each launch writes about 9 GB of outputs."""
import pytest
import torch

from oracle import oracle as O

pytestmark = pytest.mark.gpu

B, N = 65536, 8
M = B * N


def _env(seed):
    import gym_uav_collision_avoidance_b200 as G

    e = G.BatchedMultiUAVWorld2D(B, num_agents=N, reset_mode=O.RESET_ON_DONE0, max_episode_steps=60, x_size=20.0,
                                 y_size=20.0, seed=seed)
    e.reset()
    return e


def _actions(K, seed):
    gen = torch.Generator(device="cuda").manual_seed(seed)
    return torch.rand((K, B, N, 2), generator=gen, device="cuda") * 20 - 10


def _check(whole, parts, k0):
    for key in ("obs", "reward", "done"):
        assert torch.equal(whole[key][k0:k0 + parts[key].shape[0]], parts[key]), f"{key} differs in steps from {k0}"


def test_general_rollout_above_the_offset_bound_equals_two_plain_launches():
    K = 410
    assert K * M * 10 >= 2**31 > (K // 2) * M * 10
    acts = _actions(K, 410)
    e1, e2 = _env(41), _env(41)
    whole = e1.rollout(K, acts)
    first = e2.rollout(K // 2, acts[:K // 2])
    _check(whole, first, 0)
    del first
    second = e2.rollout(K - K // 2, acts[K // 2:])
    _check(whole, second, K // 2)
    assert torch.equal(e1.state.blob, e2.state.blob), "state after the rollout differs"
    assert e1.stats()["episodes"] > B  # the auto-reset path ran


def test_plain_rollout_below_the_offset_bound_equals_the_general_instance():
    K = 409
    assert K * M * 10 < 2**31
    acts = _actions(K, 409)
    e1, e2 = _env(42), _env(42)
    plain = e1.rollout(K, acts)
    general = e2.rollout(K, acts, want_reset_mask=True)  # the reset mask makes it the general instance
    _check(general, plain, 0)
    assert torch.equal(e1.state.blob, e2.state.blob), "state after the rollout differs"
    assert e1.stats()["episodes"] > B
