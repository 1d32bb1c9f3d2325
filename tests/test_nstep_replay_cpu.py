"""CPU: the n-step restatement of test_nstep_replay_gpu.py against a brute-force walk over each UAV's episodes, and the
C-ABI's n-step argument checks that run before any launch."""
import ctypes as C

import numpy as np
import pytest

from test_nstep_replay_gpu import restated_nstep, ring_owner, truth_nstep


def synthetic_acting(T, B, N, seed, p_done=0.05, p_reset=0.08, od=4):
    """T acting steps of B envs x N UAVs as the step kernels record them: obs acted on, next obs (before any reset),
    reward, done, and the env's auto-reset; the next step acts on next obs unless the env reset."""
    rng = np.random.default_rng(seed)
    M = B * N
    obs = np.empty((T, M, od), np.float32)
    nxt = rng.random((T, M, od), dtype=np.float32)
    rew = rng.standard_normal((T, M)).astype(np.float32)
    done = rng.random((T, M)) < p_done
    reset = np.repeat(rng.random((T, B)) < p_reset, N, axis=1)
    obs[0] = rng.random((M, od), dtype=np.float32)
    for t in range(1, T):
        obs[t] = np.where(reset[t - 1][:, None], rng.random((M, od), dtype=np.float32), nxt[t - 1])
    return obs, nxt, rew, done, reset


def fill_ring(cap, obs, nxt, rew, done):
    """The ring after appending each step's M transitions at the head, wrapping at cap."""
    T, M, od = obs.shape
    r_obs, r_nxt = np.zeros((cap, od), np.float32), np.zeros((cap, od), np.float32)
    r_rew, r_mask = np.zeros(cap, np.float32), np.zeros(cap, np.float32)
    for t in range(T):
        s = (t * M + np.arange(M)) % cap
        r_obs[s], r_nxt[s], r_rew[s], r_mask[s] = obs[t], nxt[t], rew[t], 1.0 - done[t]
    return r_obs, r_rew, r_nxt, r_mask, (T * M) % cap


def brute_force(rew, done, reset, t, m, n, gamma):
    """One UAV's n-step target by walking its episode one step at a time."""
    R, g, k = 0.0, 1.0, 0
    T = rew.shape[0]
    while True:
        R = R + g * float(rew[t + k, m])
        g = g * gamma
        k += 1
        if k == n or done[t + k - 1, m] or reset[t + k - 1, m] or t + k >= T:
            break
    return k, np.float32(R), np.float32(0.0) if done[t + k - 1, m] else np.float32(g)


@pytest.mark.parametrize("B,N,cap,n,gamma", [(7, 3, 97, 5, 0.99), (4, 10, 400, 16, 1.0), (50, 1, 333, 3, 0.0),
                                             (3, 5, 15, 4, 0.9)])
def test_restatement_equals_a_brute_force_episode_walk(B, N, cap, n, gamma):
    """On rings filled by synthetic acting logs (with wraps; a ring of exactly one step in the last case), the rule of
    include/uavca.h gives every filled slot the target of a walk over its UAV's episode."""
    T = 40
    M = B * N
    obs, nxt, rew, done, reset = synthetic_acting(T, B, N, seed=B * cap + n)
    r_obs, r_rew, r_nxt, r_mask, head = fill_ring(cap, obs, nxt, rew, done)
    owner = ring_owner(cap, M, T)
    slots = np.arange(cap)
    k, R, disc, last = restated_nstep(r_obs, r_rew, r_nxt, r_mask, head, slots, M, n, gamma)
    tk, tR, tdisc, tq = truth_nstep(rew, done, reset, owner[slots], n, gamma)
    assert np.array_equal(k, tk) and np.array_equal(R, tR) and np.array_equal(disc, tdisc)
    assert np.array_equal(last, tq % cap)
    for s in range(0, cap, max(1, cap // 50)):
        q = owner[s]
        bk, bR, bd = brute_force(rew, done, reset, q // M, q % M, n, gamma)
        assert (k[s], R[s], disc[s]) == (bk, bR, bd), s
    if cap > M:
        assert k.min() == 1 and k.max() >= min(n, cap // M)


def test_restatement_folds_in_float64_and_rounds_once():
    obs = np.zeros((4, 1), np.float32)
    nxt = np.zeros((4, 1), np.float32)
    rew = np.array([1.0, 2.0 ** -24, 2.0 ** -24, 0.0], np.float32)
    mask = np.array([1, 1, 1, 0], np.float32)
    k, R, disc, last = restated_nstep(obs, rew, nxt, mask, 0, np.array([0]), 1, 4, 1.0)
    # a float32 fold would round both 2^-24 terms away (ties to even); float64 keeps them and rounds 1 + 2^-23 once
    assert k[0] == 4 and R[0] == np.float32(1.0 + 2.0 ** -23) and disc[0] == 0.0 and last[0] == 3
    nxt[0, 0] = -0.0  # bit equality: -0.0 does not chain into +0.0
    k, R, disc, last = restated_nstep(obs, rew, nxt, mask, 0, np.array([0]), 1, 4, 0.5)
    assert k[0] == 1 and disc[0] == np.float32(0.5) and R[0] == 1.0


def test_bad_nstep_arguments_are_refused_before_any_launch():
    """n outside 1..16, stride outside 1..capacity, gamma NaN, negative or above 1 fail on the host (the fake pointers
    are never dereferenced), for both samplers."""
    from gym_uav_collision_avoidance_b200 import _capi, build

    build.build()
    lib = _capi.load()
    fake = C.c_void_p(256)
    cap = 1000

    def uniform(stride, n, gamma):
        return lib.uavca_replay_sample_nstep(fake, fake, fake, fake, fake, cap, 10, 2, fake, 8, 0, 0, 0, stride, n, gamma,
                                             fake, fake, fake, fake, fake, fake, None)

    def prioritized(stride, n, gamma):
        return lib.uavca_per_sample_nstep(fake, fake, fake, fake, fake, cap, 10, 2, fake, fake, 1024, 8, 0.4, stride, n,
                                          gamma, 0, 0, fake, fake, fake, fake, fake, fake, fake, None)

    for call in (uniform, prioritized):
        for args, text in (((10, 0, 0.9), "n = 0"), ((10, 17, 0.9), "n = 17"), ((0, 3, 0.9), "stride = 0"),
                           ((cap + 1, 3, 0.9), "stride = 1001"), ((10, 3, float("nan")), "gamma"),
                           ((10, 3, -0.01), "gamma"), ((10, 3, 1.0 + 2 ** -52), "gamma"), ((10, 3, float("inf")), "gamma")):
            assert call(*args) == -1, (call.__name__, args)
            assert text in _capi.last_error(), (call.__name__, args, _capi.last_error())
    assert lib.uavca_version() == 205
