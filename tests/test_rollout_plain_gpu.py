"""GPU: the plain `uavca_rollout` launch — no final_obs, reset_mask, action_out or score tracking, as the open-loop
driver loops and bench.py call it — against K single steps.

Such a launch runs its own kernel instances (the action source and the action mapping fixed at compile time), so it is
pinned here on its own: bit-identical observations, rewards, done flags and state to K calls of `step()` fed the same
actions, with an action block and with Philox actions, for full and ragged last warps."""
import pytest
import torch

from oracle import oracle as O

pytestmark = pytest.mark.gpu

# B is not a multiple of the envs per warp (32 // n) except at n = 32: the last warp of the shard is ragged.  n = 7 has no
# specialised kernel (the runtime-N instance).
SHAPES = [(5, 1027), (7, 2050), (8, 4099), (10, 1501), (16, 1001), (32, 515)]


def _pair(B, n, **kw):
    import gym_uav_collision_avoidance_b200 as G

    if (B * n * 10 * 4) % 16:
        B += 1  # K > 1 needs 16-byte aligned step blocks
    mk = lambda: G.BatchedMultiUAVWorld2D(B, num_agents=n, reset_mode=O.RESET_ON_DONE0, max_episode_steps=15,  # noqa: E731
                                         x_size=20.0, y_size=20.0, **kw)
    a, b = mk(), mk()
    a.reset()
    b.reset()
    return a, b, B


def _check(out, k, o, r, d):
    assert torch.equal(out["obs"][k], o), f"obs differs at step {k}"
    assert torch.equal(out["reward"][k], r) and torch.equal(out["done"][k], d), f"reward/done differ at step {k}"


@pytest.mark.parametrize("evaluate", [False, True])
@pytest.mark.parametrize("n,B", SHAPES)
def test_plain_rollout_with_action_block_equals_single_steps(n, B, evaluate):
    K = 37
    e1, e2, B = _pair(B, n, seed=150 + n)
    gen = torch.Generator(device="cuda").manual_seed(100 + n)
    acts = torch.rand((K, B, n, 2), generator=gen, device="cuda") * 20 - 10
    out = e1.rollout(K, acts, evaluate=evaluate)
    assert set(out) == {"obs", "reward", "done"}
    for k in range(K):
        o, r, d, _ = e2.step(acts[k], evaluate=evaluate)
        _check(out, k, o, r, d)
    assert torch.equal(e1.state.blob, e2.state.blob), "state after the rollout differs from K single steps"
    assert e1.stats()["episodes"] > B  # every env went through the step limit: the auto-reset path ran


@pytest.mark.parametrize("n,B", SHAPES)
def test_plain_rollout_with_philox_actions_equals_single_steps(n, B):
    K, seed, step0 = 40, 0x51A + n, 777  # odd step0: the first step uses the second half of a Philox block
    e1, e2, B = _pair(B, n, seed=250 + n)
    out = e1.rollout(K, None, action_seed=seed, step0=step0)  # "cartesian" Philox actions span the action box
    assert set(out) == {"obs", "reward", "done"}
    for k in range(K):
        o, r, d, _ = e2.step(e2.sample_actions(step0 + k, seed), action_mode="scaled")
        _check(out, k, o, r, d)
    assert torch.equal(e1.state.blob, e2.state.blob), "state after the rollout differs from K single steps"
    assert e1.stats()["episodes"] > B
