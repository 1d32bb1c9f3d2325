"""n-step returns from the device ring (`replay_sample_nstep_kernel`, csrc/uavca_kernels.cu; `per_sample_kernel<true>`,
csrc/uavca_per.cu; the shared gather in csrc/uavca_nstep.cuh) against restatements kept in this file:

* `restated_nstep`: the rule of include/uavca.h (mask, age and bit-equality links, k, the float64 fold, the discount)
  in numpy, exact;
* `truth_nstep`: n-step targets formed from an acting log alone (per-step reward, done and reset mask), with the true
  episode structure and no observation test; on rings filled by real rollouts it must agree with the device exactly.

The slots come from the one-step samplers' restatements (test_acting_kernels_gpu.restated_slots,
test_prioritized_replay_gpu.restated_draws).  Tests without the `gpu` marker need no device."""
import numpy as np
import pytest
import torch

from test_acting_kernels_gpu import restated_slots
from test_prioritized_replay_gpu import WEIGHT_REL, restated_draws

gpu = pytest.mark.gpu

C4_B, C4_N = 16384, 10  # configs[4]
CAP = 1 << 20


# ---- restatements -------------------------------------------------------------------------------------------------------


def restated_nstep(obs, rew, nxt, mask, head, slots, stride, n, gamma):
    """The n-step rule of include/uavca.h on host copies of the ring (obs / nxt float32 [cap, od], rew / mask float32
    [cap]) for drawn `slots`.  -> (k int64, R float32, discount float32, last slot s_{k-1})."""
    cap = rew.size
    ob, nb = obs.view(np.uint32), nxt.view(np.uint32)
    slots = np.asarray(slots, np.int64)
    age = (head - 1 - slots) % cap
    k = np.ones(slots.shape, np.int64)
    alive = np.ones(slots.shape, bool)
    prev = slots
    for i in range(1, n):
        si = (slots + i * stride) % cap
        alive = alive & (mask[prev] != 0) & (i * stride <= age) & (ob[si] == nb[prev]).all(axis=1)
        k += alive
        prev = si
    R, g = np.zeros(slots.shape), np.ones(slots.shape)
    for i in range(n):
        on = i < k
        R = np.where(on, R + g * rew[(slots + i * stride) % cap].astype(np.float64), R)
        g = np.where(on, g * gamma, g)
    last = (slots + (k - 1) * stride) % cap
    disc = np.where(mask[last] != 0, g.astype(np.float32), np.float32(0.0))
    return k, R.astype(np.float32), disc, last


def truth_nstep(rew, done, reset, q, n, gamma):
    """n-step targets from an acting log alone: rew / done / reset [T, M] (reset: the UAV's env auto-reset after that
    step), q = t * M + m the transitions of the drawn slots.  The return continues from step t + i - 1 to t + i while
    that step was not terminal for the UAV, its env did not reset, and step t + i has been taken.  -> (k, R, discount,
    q of the last transition)."""
    T, M = rew.shape
    q = np.asarray(q, np.int64)
    t, m = q // M, q % M
    k = np.ones(q.shape, np.int64)
    alive = np.ones(q.shape, bool)
    for i in range(1, n):
        tp = t + i - 1
        alive = alive & (t + i < T) & ~done[np.minimum(tp, T - 1), m] & ~reset[np.minimum(tp, T - 1), m]
        k += alive
    R, g = np.zeros(q.shape), np.ones(q.shape)
    for i in range(n):
        on = i < k
        R = np.where(on, R + g * rew[np.minimum(t + i, T - 1), m].astype(np.float64), R)
        g = np.where(on, g * gamma, g)
    tl = t + k - 1
    disc = np.where(done[tl, m], np.float32(0.0), g.astype(np.float32))
    return k, R.astype(np.float32), disc, tl * M + m


def ring_owner(cap, M, T):
    """q = t * M + m of the transition each slot holds after T appends of M into an empty ring (-1: never written)."""
    owner = np.full(cap, -1, np.int64)
    q = np.arange(T * M, dtype=np.int64)
    owner[q % cap] = q  # later transitions overwrite earlier ones
    return owner


def host_ring(rb):
    return (rb.state.cpu().numpy(), rb.reward.cpu().numpy(), rb.next_state.cpu().numpy(), rb.mask.cpu().numpy())


# ---- a synthetic ring of configs[4] steps with episode structure -------------------------------------------------------


def fill_chained(rb, steps, B, N, g, p_done=0.03, p_reset=0.05, sizes=None):
    """Append `steps` acting steps of B envs x N UAVs: next step's observation = this step's next observation, except in
    envs that reset (a fresh observation); mask 0 with probability p_done.  The action row holds (UAV, step), so the
    transitions a return chains can be checked.  `sizes` (a list of UAV counts per step) makes mixed-size appends: only
    the first sizes[t] UAVs act at step t."""
    M = B * N
    obs = torch.rand((M, rb.obs_dim), generator=g, device="cuda")
    for t in range(steps):
        nxt = torch.rand((M, rb.obs_dim), generator=g, device="cuda")
        done = (torch.rand(M, generator=g, device="cuda") < p_done).to(torch.uint8)
        act = torch.stack([torch.arange(M, device="cuda", dtype=torch.float32), torch.full((M,), float(t), device="cuda")], 1)
        rew = torch.randn(M, generator=g, device="cuda") * 0.1
        m = M if sizes is None else sizes[t]
        rb.push(obs[:m], act[:m, :rb.act_dim], rew[:m], nxt[:m], done[:m])
        reset = (torch.rand(B, generator=g, device="cuda") < p_reset).repeat_interleave(N)
        obs = torch.where(reset[:, None], torch.rand((M, rb.obs_dim), generator=g, device="cuda"), nxt)


@pytest.fixture(scope="module")
def c4_ring():
    """A 2^20-slot prioritized ring filled by 11 configs[4]-shape appends (163,840 transitions each: it wraps), with
    priorities spread over 1e3."""
    import gym_uav_collision_avoidance_b200 as G

    rb = G.PrioritizedDeviceReplay(CAP, 10, 2, seed=21)
    g = torch.Generator(device="cuda").manual_seed(21)
    fill_chained(rb, 11, C4_B, C4_N, g)
    rb.update_priorities(torch.arange(CAP, device="cuda"), torch.exp(torch.rand(CAP, generator=g, device="cuda") * 7.0))
    torch.cuda.synchronize()
    return rb


def _check_draw(rb, host, sampler, batch, n, gamma, stride):
    """One n-step draw against the restatement: slots, state, action, next_state, R and discount exact, weights within
    the PER bound.  -> (k, slots)."""
    obs, rew, nxt, mask = host
    head, _, size, appends = (int(v) for v in rb.meta.tolist())
    if sampler == "prioritized":
        draw, tree = rb._per_draws, rb.tree.cpu().numpy()
        s, a, r, ns, d, idx, w = rb.sample_prioritized_nstep(batch, 0.4, n, gamma, stride)
        want_idx, want_w = restated_draws(tree, rb._sample_seed, draw + appends, batch, 0.4, size)
        got_w = w.cpu().numpy().astype(np.float64)
        assert (np.abs(got_w - want_w) <= WEIGHT_REL * want_w).all()
    else:
        draw = rb._draws
        s, a, r, ns, d, idx = rb.sample_nstep(batch, n, gamma, stride, recency_weighted=sampler == "recency", want_index=True)
        want_idx = restated_slots(rb._sample_seed, draw + appends, batch, head, size, rb.capacity, sampler == "recency")
    idx = idx.cpu().numpy()
    assert np.array_equal(idx, want_idx), (sampler, batch, n, gamma)
    k, R, disc, last = restated_nstep(obs, rew, nxt, mask, head, idx, stride, n, gamma)
    assert np.array_equal(s.cpu().numpy(), obs[idx]) and np.array_equal(ns.cpu().numpy(), nxt[last])
    assert np.array_equal(a.cpu().numpy(), rb.action[torch.from_numpy(idx).cuda()].cpu().numpy())
    assert np.array_equal(r.cpu().numpy().view(np.uint32), R.view(np.uint32)), (sampler, batch, n, gamma)
    assert np.array_equal(d.cpu().numpy().view(np.uint32), disc.view(np.uint32)), (sampler, batch, n, gamma)
    return k, idx


# ---- GPU ----------------------------------------------------------------------------------------------------------------


@gpu
@pytest.mark.parametrize("sampler", ["uniform", "recency", "prioritized"])
@pytest.mark.parametrize("n", [1, 2, 3, 5, 16])
def test_nstep_draws_match_the_restatement(c4_ring, sampler, n):
    rb = c4_ring
    host = host_ring(rb)
    act = rb.action.cpu().numpy()
    ks = []
    for gamma in (0.0, 0.99, 1.0):
        for batch in (1, 256, 4096):
            k, idx = _check_draw(rb, host, sampler, batch, n, gamma, C4_B * C4_N)
            # every chained successor is the same UAV's next step
            for i in range(1, n):
                on = i < k
                si = (idx[on] + i * C4_B * C4_N) % CAP
                assert np.array_equal(act[si, 0], act[idx[on], 0]) and np.array_equal(act[si, 1], act[idx[on], 1] + i)
            ks.append(k)
    ks = np.concatenate(ks)
    # the ring holds 6.4 steps: at most 7 transitions of one UAV can chain
    assert min(n, 6) <= ks.max() <= min(n, 7) and (n == 1 or ks.min() == 1)


@gpu
@pytest.mark.parametrize("gamma", [0.0, 0.99, 1.0])
def test_n1_equals_the_one_step_samplers(c4_ring, gamma):
    rb = c4_ring
    g32 = np.float32(gamma)
    for recency in (False, True):
        d0 = rb._draws
        one = rb.sample_fused(4096, recency_weighted=recency, want_index=True)
        rb._draws = d0
        nst = rb.sample_nstep(4096, 1, gamma, C4_B * C4_N, recency_weighted=recency, want_index=True)
        assert rb._draws == d0 + 1
        for i in (0, 1, 2, 3, 5):
            assert torch.equal(one[i], nst[i]), (recency, i)
        assert np.array_equal(nst[4].cpu().numpy(), g32 * one[4].cpu().numpy())
    d0 = rb._per_draws
    one = rb.sample_prioritized(4096, 0.6)
    rb._per_draws = d0
    nst = rb.sample_prioritized_nstep(4096, 0.6, 1, gamma, C4_B * C4_N)
    assert rb._per_draws == d0 + 1
    for i in (0, 1, 2, 3, 5, 6):
        assert torch.equal(one[i], nst[i]), i
    assert np.array_equal(nst[4].cpu().numpy(), g32 * one[4].cpu().numpy())


@gpu
def test_wrong_stride_yields_one_step_returns(c4_ring):
    rb = c4_ring
    _, rew, nxt, mask = host_ring(rb)
    for stride in (C4_B * C4_N + 1, C4_B * C4_N - C4_N, 1):
        s, a, r, ns, d, idx = rb.sample_nstep(4096, 5, 0.99, stride, want_index=True)
        idx = idx.cpu().numpy()
        assert np.array_equal(r.cpu().numpy(), rew[idx]) and np.array_equal(ns.cpu().numpy(), nxt[idx])
        assert np.array_equal(d.cpu().numpy(), np.float32(0.99) * mask[idx])


@gpu
def test_mixed_size_appends_only_truncate():
    """Every third append holds 600 transitions instead of 1,000: the stride no longer finds a UAV's successor across
    it.  The device still equals the restatement, and every transition it chains is the same UAV's next step."""
    import gym_uav_collision_avoidance_b200 as G

    B, N, cap = 100, 10, 9_973
    rb = G.DeviceReplay(cap, 10, 2, seed=3)
    g = torch.Generator(device="cuda").manual_seed(3)
    fill_chained(rb, 25, B, N, g, sizes=[1000 if t % 3 else 600 for t in range(25)])
    host = host_ring(rb)
    act = rb.action.cpu().numpy()
    ks = []
    for recency in ("uniform", "recency"):
        k, idx = _check_draw(rb, host, recency, 8192, 6, 0.97, B * N)
        for i in range(1, 6):
            on = i < k
            si = (idx[on] + i * B * N) % cap
            assert np.array_equal(act[si, 0], act[idx[on], 0]) and np.array_equal(act[si, 1], act[idx[on], 1] + i)
        ks.append(k)
    ks = np.concatenate(ks)
    assert (ks == 1).any() and (ks > 1).any() and ks.max() < 6  # never 5 full-size appends in a row


@gpu
def test_empty_ring_yields_slot_0_with_discount_0():
    import gym_uav_collision_avoidance_b200 as G

    rb = G.PrioritizedDeviceReplay(1000, 7, 3, seed=1)
    for recency in (False, True):
        s, a, r, ns, d, idx = rb.sample_nstep(300, 5, 0.99, 10, recency_weighted=recency, want_index=True)
        assert bool((idx == 0).all()) and not bool(d.any()) and not bool(s.any()) and not bool(ns.any()) and not bool(r.any())
    s, a, r, ns, d, idx, w = rb.sample_prioritized_nstep(300, 0.4, 16, 1.0, 1000)
    assert bool((idx == 0).all()) and not bool(d.any()) and not bool(w.any()) and not bool(r.any())
    assert rb.tree.abs().sum().item() == 0.0


def _make_env(world, N, mode, seed):
    import gym_uav_collision_avoidance_b200 as G

    if world == "single":
        return G.BatchedUAVWorld2D(256, reset_mode=mode, max_episode_steps=60, seed=seed)
    B = max(8, 2048 // N)
    return G.BatchedMultiUAVWorld2D(B, num_agents=N, reset_mode=mode, max_episode_steps=60, seed=seed,
                                    circular=world == "circular")


ROLLOUTS = [("fused", "multi", n) for n in (2, 8, 10, 20, 32)] + [("push", "single", 1), ("push", "multi", 40),
                                                                  ("push", "circular", 6)]


@gpu
@pytest.mark.parametrize("mode", ["done0", "all_done"])
@pytest.mark.parametrize("path,world,N", ROLLOUTS)
def test_rule_finds_the_true_episode_boundaries(path, world, N, mode):
    """A BatchedRollout with terminal ends, max_episode_steps truncations and auto-resets; the n-step targets of the
    drawn slots equal those formed from the acting log alone (truth_nstep), including the newest slots and slots whose
    successors wrap around the ring."""
    import gym_uav_collision_avoidance_b200 as G

    rmode = {"done0": G.RESET_ON_DONE0, "all_done": G.RESET_ON_ALL_DONE}[mode]
    env = _make_env(world, N, rmode, seed=N + 5)
    B = env.num_envs
    M = B * env.num_agents
    cap = 23 * M + 7
    rb = G.DeviceReplay(cap, env.obs_dim, 2, seed=N)
    ro = G.BatchedRollout(env, None, rb, action_mode="polar", warmup_uniform=True)
    assert ro.fused_append == (path == "fused")
    ro.reset()
    T = 150
    rew, done, reset = np.zeros((T, M), np.float32), np.zeros((T, M), bool), np.zeros((T, M), bool)
    for t in range(T):
        ro.step()
        rew[t] = env.reward.reshape(-1).cpu().numpy()
        done[t] = env.done.reshape(-1).cpu().numpy() != 0
        reset[t] = np.repeat(env.reset_mask.cpu().numpy() != 0, env.num_agents)
    assert int(rb.meta[3]) == T
    # truncations occur everywhere, terminal ends too (the float64 world's ring layout keeps its UAVs apart for 150 steps)
    assert (reset & ~done).any() and (done.any() or world == "circular")
    owner = ring_owner(cap, M, T)
    _, _, nxt, _ = host_ring(rb)
    head = int(rb.meta[0])
    for n, gamma in ((5, 0.99), (16, 1.0)):
        for recency in (False, True):
            s, a, r, ns, d, idx = rb.sample_nstep(8192, n, gamma, M, recency_weighted=recency, want_index=True)
            idx = idx.cpu().numpy()
            k, R, disc, ql = truth_nstep(rew, done, reset, owner[idx], n, gamma)
            assert np.array_equal(r.cpu().numpy().view(np.uint32), R.view(np.uint32)), (n, recency)
            assert np.array_equal(d.cpu().numpy().view(np.uint32), disc.view(np.uint32)), (n, recency)
            assert np.array_equal(ns.cpu().numpy(), nxt[ql % cap])
            age = (head - 1 - idx) % cap
            if recency:
                assert (age < (n - 1) * M).any()  # the newest slots: truncated by age
            else:
                assert ((idx + (k - 1) * M) >= cap).any()  # returns that wrap around the ring


PREMISE = [("warp", 8), ("cta", 11), ("cta", 20), ("single", 1), ("general", 40), ("circular", 6)]


@gpu
@pytest.mark.parametrize("family,N", PREMISE)
def test_final_obs_is_the_next_acted_on_obs_without_a_reset(family, N):
    """The episode test rests on this: for every env that did not reset, the step's final_obs (the ring's next_obs) is
    bit for bit the observation the next step acts on."""
    import gym_uav_collision_avoidance_b200 as G

    world = {"single": "single", "circular": "circular"}.get(family, "multi")
    env = _make_env(world, N, G.RESET_ON_DONE0, seed=N)
    env.enable_final_obs()
    env.reset()
    g = torch.Generator(device="cuda").manual_seed(N)
    resets = 0
    for t in range(120):
        a = torch.rand((env.num_envs, env.num_agents, 2), generator=g, device="cuda") * 2 - 1
        if world == "single":
            env.step(a.reshape(env.num_envs, 2), action_mode="polar")
        else:
            env.step(a, action_mode="polar")
        keep = env.reset_mask == 0
        resets += int((~keep).sum())
        fo, ob = env.final_obs.view(torch.int32), env.obs.view(torch.int32)
        assert torch.equal(fo[keep], ob[keep]), (family, t)
    assert resets > 0


@gpu
def test_captured_learner_step_draws_fresh_exact_batches():
    """An acting step (fused append + sync into a prioritized ring) and a learner step (sample_nstep and
    sample_prioritized_nstep into reused tensors), each captured once: every learner replay equals the restatement on
    the ring as the acting replays left it."""
    import gym_uav_collision_avoidance_b200 as G

    B, N = 512, 10
    M = B * N
    env = G.BatchedMultiUAVWorld2D(B, num_agents=N, reset_mode=G.RESET_ON_DONE0, max_episode_steps=40, seed=2)
    rb = G.PrioritizedDeviceReplay(M * 9 + 3, 10, 2, seed=8)
    ro = G.BatchedRollout(env, None, rb, action_mode="polar", warmup_uniform=True)
    assert ro.fused_append
    ro.reset()
    batch, n, gamma = 512, 3, 0.99
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        ro.run(4)
        uni = rb.sample_nstep(batch, n, gamma, M, want_index=True)
        per = rb.sample_prioritized_nstep(batch, 0.5, n, gamma, M)
    torch.cuda.current_stream().wait_stream(s)
    torch.cuda.synchronize()
    act, learn = torch.cuda.CUDAGraph(), torch.cuda.CUDAGraph()
    with torch.cuda.graph(act):
        ro.run(2)
    d_uni, d_per = rb._draws, rb._per_draws
    with torch.cuda.graph(learn):
        rb.sample_nstep(batch, n, gamma, M, out=uni)
        rb.sample_prioritized_nstep(batch, 0.5, n, gamma, M, out=per)
    torch.cuda.synchronize()
    seen = []
    for rnd in range(4):
        act.replay()
        torch.cuda.synchronize()
        head, _, size, appends = (int(v) for v in rb.meta.tolist())
        obs, rew, nxt, mask = host_ring(rb)
        tree = rb.tree.cpu().numpy()
        learn.replay()
        torch.cuda.synchronize()
        want = restated_slots(rb._sample_seed, d_uni + appends, batch, head, size, rb.capacity, False)
        want_p, want_w = restated_draws(tree, rb._sample_seed, d_per + appends, batch, 0.5, size)
        for out, w_idx in ((uni, want), (per, want_p)):
            assert np.array_equal(out[5].cpu().numpy(), w_idx), rnd
            k, R, disc, last = restated_nstep(obs, rew, nxt, mask, head, w_idx, M, n, gamma)
            assert np.array_equal(out[2].cpu().numpy(), R) and np.array_equal(out[4].cpu().numpy(), disc)
            assert np.array_equal(out[3].cpu().numpy(), nxt[last]) and np.array_equal(out[0].cpu().numpy(), obs[w_idx])
        got_w = per[6].cpu().numpy().astype(np.float64)
        assert (np.abs(got_w - want_w) <= WEIGHT_REL * want_w).all(), rnd
        seen.append(want)
    assert all(not np.array_equal(seen[i], seen[i + 1]) for i in range(len(seen) - 1))
