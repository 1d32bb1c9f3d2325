"""GPU: the rows either side of the hot path — B=1 drop-in classes (compat), device replay ring, batched acting
path — against the reference's golden vectors and plain PyTorch restatements."""
import numpy as np
import pytest
import torch

from _golden import Case, obs_close

pytestmark = pytest.mark.gpu
RTOL, ATOL = 1e-5, 1e-6


def _close(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return np.abs(a - b) <= RTOL * np.abs(b) + ATOL


# ---- compat: the reference's loop shape, lists in / lists out ------------------------------------------------------


def test_compat_multi_runs_the_reference_loop_on_golden_vectors():
    from gym_uav_collision_avoidance_b200 import compat

    case = Case("multi_n8")
    z, N = case.z, case.N
    for e in range(2):  # env e of the golden batch, through the B=1 class
        env = compat.MultiUAVWorld2D(num_agents=N)
        env.reset()
        for i, ag in enumerate(env.agent_list):  # state injection the way the scripts do it (attribute assignment)
            ag.location = z["init_pos"][e, i]
            ag.target_location = z["init_tgt"][e, i]
            ag.velocity = z["init_vel"][e, i]
            ag.init_distance = z["init_init"][e, i]
            ag.prev_distance = z["init_prev"][e, i]
            ag.done = bool(z["init_flags"][e, i] & 1)
            ag.collided = bool(z["init_flags"][e, i] & 2)
        env.steps = env.target_reach_count = env.collision_count = 0
        for t in range(60):
            actions = [z["action"][t, e, i].astype(np.float64) for i in range(N)]
            obs, rewards, dones, info = env.step(actions)
            assert isinstance(obs, list) and len(obs) == N and obs[0].shape == (10,) and obs[0].dtype == np.float64
            assert isinstance(rewards, list) and isinstance(rewards[0], float)
            assert isinstance(dones, list) and isinstance(dones[0], bool) and info == {"distance": 0}
            assert dones == [bool(d) for d in z["done"][t, e]], f"done flags env {e} step {t}"
            assert _close(rewards, z["reward"][t, e]).all()
            assert obs_close(np.stack(obs), z["obs"][t, e], RTOL, ATOL).all()
            assert np.array_equal(np.stack([a.location for a in env.agent_list]), z["pos"][t, e])
            assert env.steps == int(z["steps"][t, e]) and env.collision_count == int(z["coll"][t, e])
            assert env.target_reach_count == int(z["reach"][t, e])
        env.close()


def test_compat_keeps_float64_actions():
    """The reference's SAC loop builds float64 cartesian actions on the host (test_sac_multi.py:77-80) and UAVAgent.step
    consumes them in float64 (uav_agent.py:26): the drop-in hands them over unrounded (uavca_step_f64) — positions,
    velocities and flags bit-exact against a golden run of the literal reference whose actions float32 cannot hold."""
    from gym_uav_collision_avoidance_b200 import compat

    case = Case("f64act_multi_n5")
    z, N = case.z, case.N
    assert (z["action64"] != z["action64"].astype(np.float32)).mean() > 0.5
    for e in (0, 1):
        env = compat.MultiUAVWorld2D(num_agents=N)
        env.reset()
        for i, ag in enumerate(env.agent_list):
            ag.location, ag.target_location, ag.velocity = z["init_pos"][e, i], z["init_tgt"][e, i], z["init_vel"][e, i]
            ag.init_distance, ag.prev_distance = z["init_init"][e, i], z["init_prev"][e, i]
            ag.done, ag.collided = bool(z["init_flags"][e, i] & 1), bool(z["init_flags"][e, i] & 2)
        env.steps = env.target_reach_count = env.collision_count = 0
        for t in range(80):
            if z["reset_mask"][t, e]:
                break  # the golden harness restarts from its pool there
            obs, rewards, dones, _ = env.step([z["action64"][t, e, i] for i in range(N)])
            assert dones == [bool(d) for d in z["done"][t, e]], f"done flags env {e} step {t}"
            assert np.array_equal(np.stack([a.location for a in env.agent_list]), z["pos"][t, e]), f"positions env {e} step {t}"
            assert np.array_equal(np.stack([a.velocity for a in env.agent_list]), z["vel"][t, e]), f"velocities env {e} step {t}"
            assert _close(rewards, z["reward"][t, e]).all()
            assert obs_close(np.stack(obs), z["obs"][t, e], RTOL, ATOL).all()
        assert t >= 20
        env.close()
    # the single world: float64 actions from the first step on
    case = Case("f64act_single")
    z = case.z
    env = compat.UAVWorld2D()
    env.reset()
    env._agent_location, env._target_location = z["init_pos"][0, 0], z["init_tgt"][0, 0]
    env._agent_speed, env._init_target_distance, env._prev_distance = z["init_vel"][0, 0], z["init_init"][0, 0], z["init_prev"][0, 0]
    env.steps = 0
    for t in range(60):
        if z["reset_mask"][t, 0]:
            break
        obs, r, d, info = env.step(z["action64"][t, 0, 0])
        assert bool(d) == bool(z["done"][t, 0, 0])
        assert np.array_equal(env._agent_location, z["pos"][t, 0, 0]) and np.array_equal(env._agent_speed, z["vel"][t, 0, 0])
    env.close()


def test_compat_multi_surface():
    from gym_uav_collision_avoidance_b200 import compat

    env = compat.MultiUAVWorld2D(num_agents=5, seed=3)
    assert env.observation_space.shape[0] == 10 and env.action_space.shape[0] == 2
    assert np.allclose(np.linalg.norm(env.action_space.high), 200 ** 0.5)
    assert env.max_acceleratoin[0] == 5.0 and env.max_speed[0] == 10.0 and env.d_sense == 15 and env.collider_radius == 1.0
    obs, info = env.reset(return_info=True)
    assert len(obs) == 5 and info == {"distance": 0} and env.steps == 0
    loc = np.stack([a.location for a in env.agent_list])
    assert loc.dtype == np.float32 and (np.abs(loc) <= 25).all()
    obs2 = env.reset()
    assert not np.allclose(np.stack(obs), np.stack(obs2))  # a new episode is a new draw
    ring = env.reset(circular=True)  # multi_uav_world_2d.py:157-163: float64 locations from here to the next reset()
    loc = np.stack([a.location for a in env.agent_list])
    assert loc.dtype == np.float64 and np.allclose(np.linalg.norm(loc, axis=1), 20.0, atol=1e-12) and len(ring) == 5
    tgt = np.stack([a.target_location for a in env.agent_list])
    assert tgt.dtype == np.float64 and np.allclose(np.linalg.norm(tgt, axis=1), 23.0, atol=1e-12)
    env.agent_list[2].location = np.array([1.5, -2.5000000001])
    assert np.array_equal(env.agent_list[2].location, np.array([1.5, -2.5000000001]))
    for _ in range(3):
        env.step([env.action_space.sample() for _ in range(5)])
    assert env.steps == 3 and env.agent_list[0].location.dtype == np.float64
    env.render()
    env.reset()  # a plain reset leaves the float64 world
    assert env.agent_list[0].location.dtype == np.float32 and env.steps == 0
    env.close()


def test_compat_circular_episode_is_the_references_float64_world():
    """The plotting script's loop (test_sac_multi_plot_trajectory.py:40-68: reset(circular=True), step, read
    agent.location / .done) through the drop-in class, against the literal reference's golden vectors."""
    from gym_uav_collision_avoidance_b200 import compat

    case = Case("circular_n6")
    z, N = case.z, case.N
    env = compat.MultiUAVWorld2D(num_agents=N)
    obs = env.reset(circular=True)
    assert obs_close(np.stack(obs), z["obs0"][0], RTOL, ATOL).all()
    for t in range(150):
        if z["reset_mask"][t, 0]:
            break
        obs, rewards, dones, _ = env.step([z["action"][t, 0, i].astype(np.float64) for i in range(N)])
        assert dones == [bool(d) for d in z["done"][t, 0]]
        assert np.array_equal(np.stack([a.location for a in env.agent_list]), z["pos64"][t, 0]), f"float64 locations, step {t}"
        assert _close(rewards, z["reward"][t, 0]).all() and obs_close(np.stack(obs), z["obs"][t, 0], RTOL, ATOL).all()
        assert [a.done for a in env.agent_list] == [bool(f & 1) for f in z["flags"][t, 0]]
    assert t > 100
    env.close()


def test_compat_single_runs_the_reference_loop_on_golden_vectors():
    from gym_uav_collision_avoidance_b200 import compat

    for name, f32 in (("single_f64_actions", False), ("single_f32_actions", True)):
        case = Case(name)
        z = case.z
        env = compat.UAVWorld2D(float32_actions=f32)
        env.reset()
        e = 1
        env._agent_location = z["init_pos"][e, 0]
        env._target_location = z["init_tgt"][e, 0]
        env._agent_speed = z["init_vel"][e, 0]
        env._init_target_distance = z["init_init"][e, 0]
        env._prev_distance = z["init_prev"][e, 0]
        env.steps = 0
        for t in range(40):
            if z["reset_mask"][t, e]:
                break
            obs, reward, done, info = env.step(z["action"][t, e, 0])
            assert obs.shape == (4,) and obs.dtype == np.float64 and isinstance(done, bool)
            assert done == bool(z["done"][t, e, 0])
            assert _close(reward, z["reward"][t, e, 0]) and info["distance"] == z["distance"][t, e]
            assert obs_close(obs[None], case.final_obs(t)[e], RTOL, ATOL).all()
            assert np.array_equal(env._agent_location, z["pos"][t, e, 0])
            if done:
                break
        env.close()


# ---- replay ring ------------------------------------------------------------------------------------------------------


@pytest.mark.parametrize("obs_dim,act_dim", [(10, 2), (4, 2), (5, 3)])
def test_replay_push_wraps_like_a_ring(obs_dim, act_dim):
    import gym_uav_collision_avoidance_b200 as G

    cap, M = 1000, 384
    rb = G.DeviceReplay(cap, obs_dim, act_dim, seed=1)
    ref = dict(s=torch.zeros(cap, obs_dim), a=torch.zeros(cap, act_dim), r=torch.zeros(cap), n=torch.zeros(cap, obs_dim),
               m=torch.zeros(cap))
    gen = torch.Generator().manual_seed(0)
    pos = 0
    for k in range(7):
        s, a = torch.randn(M // 4, 4, obs_dim, generator=gen), torch.randn(M // 4, 4, act_dim, generator=gen)
        r, n = torch.randn(M // 4, 4, generator=gen), torch.randn(M // 4, 4, obs_dim, generator=gen)
        d = (torch.rand(M // 4, 4, generator=gen) < 0.3).to(torch.uint8)
        rb.push(s.cuda(), a.cuda(), r.cuda(), n.cuda(), d.cuda())
        idx = (pos + torch.arange(M)) % cap
        ref["s"][idx], ref["a"][idx], ref["r"][idx] = s.view(M, -1), a.view(M, -1), r.view(M)
        ref["n"][idx], ref["m"][idx] = n.view(M, -1), 1.0 - d.view(M).float()  # mask = float(not done)
        pos = (pos + M) % cap
        assert rb.position == pos and len(rb) == min(cap, (k + 1) * M)
    for name, t in (("s", rb.state), ("a", rb.action), ("r", rb.reward), ("n", rb.next_state), ("m", rb.mask)):
        assert torch.equal(t.cpu(), ref[name]), name
    st, ac, rw, nx, mk = rb.sample(256)
    assert st.shape == (256, obs_dim) and ac.shape == (256, act_dim) and rw.shape == (256,) and mk.shape == (256,)
    assert set(mk.unique().tolist()) <= {0.0, 1.0}
    with pytest.raises(ValueError):
        rb.push(torch.zeros(cap + 1, obs_dim).cuda(), torch.zeros(cap + 1, act_dim).cuda(), torch.zeros(cap + 1).cuda(),
                torch.zeros(cap + 1, obs_dim).cuda(), torch.zeros(cap + 1, dtype=torch.uint8).cuda())


def test_replay_recency_weighted_sampling_prefers_new_transitions():
    import gym_uav_collision_avoidance_b200 as G

    rb = G.DeviceReplay(4096, 4, 2, seed=5)
    for k in range(6):  # 6144 transitions through a ring of 4096: reward carries the insertion order
        r = torch.arange(k * 1024, (k + 1) * 1024, dtype=torch.float32).cuda()
        z = torch.zeros(1024, 4).cuda()
        rb.push(z, z[:, :2], r, z, torch.zeros(1024, dtype=torch.uint8).cuda())
    _, _, rw_u, _, _ = rb.sample(200000)
    _, _, rw_w, _, _ = rb.sample(200000, recency_weighted=True)
    assert rw_u.min() >= 2048 and rw_w.min() >= 2048  # only live transitions
    mid = 2048 + 2048
    assert abs((rw_u >= mid).float().mean().item() - 0.5) < 0.01
    assert abs((rw_w >= mid).float().mean().item() - 0.75) < 0.01  # p_i ~ i: the newer half carries 3/4 of the mass


# ---- batched acting path ----------------------------------------------------------------------------------------------


def test_replay_sample_fused_gathers_on_the_device():
    """`sample_fused` (uavca_replay_sample): one launch, no host sync — slots inside the filled part, rows equal to the ring's
    rows at the returned slots, uniform and recency-weighted laws, fresh draws per call and per CUDA-graph replay."""
    import gym_uav_collision_avoidance_b200 as G

    cap, M, od = 5000, 700, 10
    rb = G.DeviceReplay(cap, od, 2, seed=4)
    gen = torch.Generator(device="cuda").manual_seed(0)
    pushed = 0

    def push():
        nonlocal pushed
        tag = torch.arange(pushed, pushed + M, device="cuda", dtype=torch.float32)  # insertion order, kept in `reward`
        rb.push(torch.rand((M, od), generator=gen, device="cuda"), torch.rand((M, 2), generator=gen, device="cuda"), tag,
                torch.rand((M, od), generator=gen, device="cuda"), (torch.rand(M, generator=gen, device="cuda") < 0.1).to(torch.uint8))
        pushed += M

    for _ in range(3):  # partly filled: 2,100 of 5,000
        push()
    s, a, r, n, m, idx = rb.sample_fused(4096, want_index=True)
    assert int(idx.min()) >= 0 and int(idx.max()) < 2100 and idx.unique().numel() > 1500
    assert torch.equal(s, rb.state[idx]) and torch.equal(a, rb.action[idx]) and torch.equal(n, rb.next_state[idx])
    assert torch.equal(r, rb.reward[idx]) and torch.equal(m, rb.mask[idx])
    assert abs(float(idx.float().mean()) / 2100 - 0.5) < 0.03  # uniform over the filled slots
    idx2 = rb.sample_fused(4096, want_index=True)[5]
    assert not torch.equal(idx, idx2)  # every call draws afresh
    for _ in range(6):  # wrapped: 6,300 pushed into 5,000 slots
        push()
    assert rb.size == cap
    r_u = rb.sample_fused(20000)[2]
    r_w = rb.sample_fused(20000, recency_weighted=True)[2]
    oldest = pushed - cap
    assert float(r_u.min()) >= oldest and float(r_w.min()) >= oldest  # nothing overwritten is ever returned
    age_u, age_w = (pushed - 1 - r_u) / cap, (pushed - 1 - r_w) / cap  # 0 = newest, 1 = oldest
    assert abs(float(age_u.mean()) - 0.5) < 0.02 and abs(float(age_w.mean()) - 1 / 3) < 0.02  # p ~ recency: E[age] = 1/3
    # captured once, replayed while the ring grows: the draws follow the ring's append counter
    out = rb.sample_fused(512, want_index=True)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        rb.sample_fused(512, out=out)
    seen = []
    for _ in range(3):
        push()
        g.replay()
        torch.cuda.synchronize()
        seen.append(out[5].clone())
        assert torch.equal(out[0], rb.state[out[5]])
    assert not torch.equal(seen[0], seen[1]) and not torch.equal(seen[1], seen[2])


def test_rollout_feeds_the_replay_ring_with_the_steps_own_transitions():
    import gym_uav_collision_avoidance_b200 as G

    torch.manual_seed(0)
    B, N = 64, 10
    env = G.BatchedMultiUAVWorld2D(B, num_agents=N, reset_mode=G.RESET_ON_DONE0, max_episode_steps=25, seed=11)
    policy = G.GaussianPolicy(10, 2).cuda()
    rb = G.DeviceReplay(B * N * 8, 10, 2, seed=0)
    ro = G.BatchedRollout(env, policy, rb, action_mode="polar", fused_append=False)
    obs0 = ro.reset().clone()
    ro.step()
    # the first B*N slots: state = reset observation, next_state = the step's own (pre-reset) observation
    assert torch.equal(rb.state[:B * N].view(B, N, 10), obs0)
    assert torch.equal(rb.next_state[:B * N].view(B, N, 10), env.final_obs)
    assert torch.equal(rb.reward[:B * N].view(B, N), env.reward)
    assert torch.equal(rb.mask[:B * N].view(B, N), 1.0 - env.done.float())
    assert (rb.action[:B * N].abs() <= 1).all()  # the policy's squashed action, mapped to cartesian inside the step
    ro.run(40)
    assert len(rb) == B * N * 8 and ro.steps == 41
    sr, cr, episodes = ro.success_collision_rates()
    assert episodes > 0 and 0.0 <= sr <= 1.0 and cr >= 0.0
    # where an env auto-reset, the policy's next observation differs from the stored terminal observation
    m = env.reset_mask.bool()
    if m.any():
        assert not torch.equal(env.obs[m], env.final_obs[m])


@pytest.mark.parametrize("N,B", [(2, 37), (5, 64), (8, 50), (10, 64), (16, 33), (20, 21), (32, 19)])
def test_step_with_the_replay_append_folded_in_equals_step_then_push(N, B):
    """uavca_step_multi_replay (one launch) against uavca_step_multi + uavca_replay_push_dev on twin envs: identical env
    outputs and state, identical ring contents, head and counters, across ring wraps (capacity is not a multiple of B*N),
    auto-resets (dones[0] / a 25-step limit) and ragged last warps."""
    import gym_uav_collision_avoidance_b200 as G

    kw = dict(num_agents=N, reset_mode=G.RESET_ON_DONE0, max_episode_steps=25, seed=5, x_size=30.0, y_size=30.0)
    M = B * N
    cap = M * 3 + 7
    envs = [G.BatchedMultiUAVWorld2D(B, **kw) for _ in range(2)]
    rings = [G.DeviceReplay(cap, 10, 2, seed=0) for _ in range(2)]
    ros = [G.BatchedRollout(e, None, r, action_mode="polar", warmup_uniform=True, fused_append=f)
           for e, r, f in zip(envs, rings, (True, False))]
    assert ros[0].fused_append and not ros[1].fused_append and envs[0].final_obs is None
    for ro in ros:
        ro.reset()
    gen = torch.Generator(device="cuda").manual_seed(3)
    for step in range(60):
        a = torch.rand((B, N, 2), generator=gen, device="cuda") * 2 - 1
        for ro in ros:
            ro.action.copy_(a)
            ro.state = ro.env.obs
            ro._env_step()
            if not ro.fused_append:
                ro.replay.push(ro.state, ro.action, ro.env.reward, ro.env.final_obs, ro.env.done)
        e0, e1 = envs
        assert torch.equal(e0.obs, e1.obs) and torch.equal(e0.reward, e1.reward) and torch.equal(e0.done, e1.done), step
        assert torch.equal(e0.reset_mask, e1.reset_mask) and torch.equal(e0.state.blob, e1.state.blob), step
        r0, r1 = rings
        assert torch.equal(r0.meta[[0, 2, 3]], r1.meta[[0, 2, 3]]) and int(r0.meta[1]) == 0, step
        for name in ("state", "action", "reward", "next_state", "mask"):
            assert torch.equal(getattr(r0, name), getattr(r1, name)), (step, name)
    assert len(rings[0]) == cap and rings[0].position == (60 * M) % cap
    assert envs[0].stats()["episodes"] > 0


def test_step_replay_and_push_share_one_ring():
    """uavca_step_multi_replay and uavca_replay_push_dev keep the ring head the same way: mixed on ONE ring (a second env
    appending with push between the first env's fused steps) they produce what push alone produces."""
    import gym_uav_collision_avoidance_b200 as G

    B, N = 48, 5
    M = B * N
    kw = dict(num_agents=N, reset_mode=G.RESET_ON_DONE0, max_episode_steps=30, seed=3)
    cap = 7 * M + 11

    def run(fused):
        a_env, b_env = G.BatchedMultiUAVWorld2D(B, **kw), G.BatchedMultiUAVWorld2D(B, **dict(kw, seed=4))
        ring = G.DeviceReplay(cap, 10, 2, seed=0)
        b_env.enable_final_obs()
        if not fused:
            a_env.enable_final_obs()
        a_env.reset(); b_env.reset()
        spare = torch.zeros_like(a_env.obs)
        gen = torch.Generator(device="cuda").manual_seed(8)
        for _ in range(25):
            act = torch.rand((B, N, 2), generator=gen, device="cuda") * 2 - 1
            prev = a_env.obs
            a_env.set_obs_buffer(spare)
            if fused:
                a_env.step_replay(act, prev, ring, action_mode="polar")
            else:
                a_env.step(act, action_mode="polar")
                ring.push(prev, act, a_env.reward, a_env.final_obs, a_env.done)
            spare = prev
            prev_b = b_env.obs.clone()
            b_env.step(act, action_mode="scaled")
            ring.push(prev_b, act, b_env.reward, b_env.final_obs, b_env.done)
        return ring

    r0, r1 = run(True), run(False)
    assert torch.equal(r0.meta, r1.meta) and r0.size == cap and int(r0.meta[3]) == 50
    for name in ("state", "action", "reward", "next_state", "mask"):
        assert torch.equal(getattr(r0, name), getattr(r1, name)), name


def test_step_with_the_replay_append_replays_from_a_cuda_graph():
    """A captured acting step (uniform actions, fused append) appends where the previous replay stopped."""
    import gym_uav_collision_avoidance_b200 as G

    B, N = 256, 10
    env = G.BatchedMultiUAVWorld2D(B, num_agents=N, reset_mode=G.RESET_ON_DONE0, max_episode_steps=40, seed=2)
    rb = G.DeviceReplay(B * N * 5, 10, 2, seed=0)
    ro = G.BatchedRollout(env, None, rb, action_mode="polar", warmup_uniform=True)
    assert ro.fused_append
    ro.reset()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        ro.run(2)
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        ro.run(2)  # an even number of steps: the env alternates between two observation buffers
    torch.cuda.synchronize()
    assert rb.position == 2 * B * N  # capturing launches nothing
    for _ in range(3):
        g.replay()
    torch.cuda.synchronize()
    assert rb.size == B * N * 5 and rb.position == (8 * B * N) % (B * N * 5) and int(rb.meta[3]) == 8
    # consecutive steps chain: the observation stored as `state` at step t+1 is the policy-side observation of step t,
    # which equals next_state of step t wherever the env did not auto-reset
    M = B * N
    nxt, st, mask = rb.next_state[0:M], rb.state[M:2 * M], rb.mask[0:M]  # steps 5 and 6 (slots wrap at 5 steps)
    same = (nxt == st).all(dim=1)
    assert same.float().mean() > 0.9 and same[mask.bool()].float().mean() > 0.9


def test_gaussian_policy_matches_the_reference_formulas():
    import gym_uav_collision_avoidance_b200 as G

    torch.manual_seed(1)
    p = G.GaussianPolicy(10, 2).cuda()
    assert [n for n, _ in p.named_parameters()] == [
        "linear1.weight", "linear1.bias", "linear2.weight", "linear2.bias", "mean_linear.weight", "mean_linear.bias",
        "log_std_linear.weight", "log_std_linear.bias"]  # pytorch_sac_temp/model.py:68-72: checkpoints load unchanged
    x = torch.randn(512, 10).cuda()
    mean, log_std = p(x)
    assert (log_std >= -20).all() and (log_std <= 2).all()
    torch.manual_seed(2)
    a, logp, _ = p.sample(x)
    torch.manual_seed(2)
    normal = torch.distributions.Normal(mean, log_std.exp())
    x_t = mean + log_std.exp() * torch.randn_like(mean)
    ref_logp = (normal.log_prob(x_t) - torch.log(1 - torch.tanh(x_t).pow(2) + 1e-6)).sum(1, keepdim=True)
    assert torch.allclose(a, torch.tanh(x_t)) and torch.allclose(logp, ref_logp, atol=1e-5)


# ---- fused tcgen05 acting kernel ----------------------------------------------------------------------------------------


def test_fused_policy_philox_noise_is_standard_normal_and_counter_keyed():
    import gym_uav_collision_avoidance_b200 as G

    p = G.GaussianPolicy(10, 2).cuda()
    with torch.no_grad():
        for prm in p.parameters():
            prm.zero_()  # mean = 0, log_std = 0: action = tanh(eps)
    f = G.FusedGaussianPolicy(p, seed=1234)
    obs = torch.zeros(200000, 10, device="cuda")
    a0 = f.act(obs).clone()
    a1 = f.act(obs).clone()
    assert not torch.equal(a0, a1)  # the call counter advances the stream
    f.counter.zero_()
    assert torch.equal(f.act(obs), a0)  # same (seed, row, counter) -> same draw
    g = torch.cuda.CUDAGraph()  # captured once, replayed: the device-side counter keeps the draws fresh
    out = torch.empty_like(a0)
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        f.act(obs, out=out)
    torch.cuda.synchronize()
    with torch.cuda.graph(g, stream=s):
        f.act(obs, out=out)
    g.replay(); torch.cuda.synchronize(); r1 = out.clone()
    g.replay(); torch.cuda.synchronize()
    assert not torch.equal(out, r1)
    eps = torch.atanh(a0.double().clamp(-1 + 1e-12, 1 - 1e-12))
    assert abs(eps.mean().item()) < 0.01 and abs(eps.std().item() - 1.0) < 0.01
    assert abs((eps ** 4).mean().item() - 3.0) < 0.1 and abs((eps[:, 0] * eps[:, 1]).mean().item()) < 0.01


def test_rollout_with_the_fused_policy():
    import gym_uav_collision_avoidance_b200 as G

    torch.manual_seed(0)
    env = G.BatchedMultiUAVWorld2D(512, num_agents=10, reset_mode=G.RESET_ON_DONE0, max_episode_steps=50, seed=2)
    ro = G.BatchedRollout(env, G.GaussianPolicy(10, 2).cuda(), G.DeviceReplay(512 * 10 * 4, 10, 2), precision="fused")
    ro.reset()
    ro.run(20)
    assert len(ro.replay) == 512 * 10 * 4 and ro.action.abs().max().item() <= 1.0 and bool(torch.isfinite(env.obs).all())


def test_fused_policy_accepts_a_td3_style_deterministic_actor():
    """pytorch_td3_temp/td3.py:14-27 — l1 10->256, l2 256->256, l3 256->2, tanh — through the same tcgen05 kernel."""
    import torch.nn as nn
    import torch.nn.functional as F
    import gym_uav_collision_avoidance_b200 as G

    class Actor(nn.Module):
        def __init__(self):
            super().__init__()
            self.l1, self.l2, self.l3 = nn.Linear(10, 256), nn.Linear(256, 256), nn.Linear(256, 2)

        def forward(self, s):
            return torch.tanh(self.l3(F.relu(self.l2(F.relu(self.l1(s))))))

    torch.manual_seed(5)
    actor = Actor().cuda()
    f = G.FusedGaussianPolicy(actor)
    obs = torch.rand(5000, 10, device="cuda") * 2 - 1
    with torch.no_grad():
        ref = actor(obs)
    a0, a1 = f.act(obs).clone(), f.act(obs).clone()
    assert (a0 - ref).abs().max().item() < 5e-3 and (a0 - a1).abs().max().item() < 1e-6  # deterministic up to e^-20 noise


def test_rollout_example_runs():
    import importlib.util
    import os

    path = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "examples", "rollout_sac_multi.py")
    spec = importlib.util.spec_from_file_location("rollout_sac_multi", path)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    sr, cr, episodes = mod.main(["--envs", "256", "--agents", "10", "--steps", "30", "--warmup-steps", "5", "--eval-envs", "64"])
    assert episodes >= 64 and 0.0 <= sr <= 1.0 and cr >= 0.0


def test_config5_rollout_env_parity_under_policy_actions():
    """BASELINE config 5's shape (B=16,384 x N=10, actions from a PyTorch GaussianPolicy through the polar map, reset on
    dones[0]): the env under policy-shaped actions against the oracle.  The polar map runs once on the device
    (`map_action`); both sides then step on the same cartesian actions, so flags and state must be bit-exact; the
    fused polar step must equal map + cartesian step bit for bit."""
    import gym_uav_collision_avoidance_b200 as G
    from oracle import oracle as O
    from test_cuda_parity import assert_outputs, assert_state_equal

    torch.manual_seed(4)
    B, N = 16384, 10
    kw = dict(reset_mode=O.RESET_ON_DONE0, max_episode_steps=120, seed=55)
    env = G.BatchedMultiUAVWorld2D(B, num_agents=N, **kw)
    fused = G.BatchedMultiUAVWorld2D(B, num_agents=N, **kw)
    orc = O.Oracle(O.multi_config(B, N, **kw), nthreads=O.max_threads())
    policy = G.GaussianPolicy(10, 2).cuda()
    obs = env.reset()
    fused.reset()
    orc.reset()
    for t in range(200):
        with torch.no_grad():
            a = policy.act(obs.view(-1, 10)).view(B, N, 2).contiguous()
        mapped = env.map_action(a, "polar")
        obs, rew, done, info = env.step(mapped)
        fused.step(a, action_mode="polar")
        out = orc.step(mapped.cpu().numpy())
        assert np.array_equal(done.cpu().numpy(), out["done"]), f"done flags differ at step {t}"
        assert np.array_equal(info["reset_mask"].cpu().numpy(), out["reset_mask"]), f"reset mask differs at step {t}"
        if t % 20 == 19:
            assert_outputs(env, out, f"(config 5, step {t})")
            assert_state_equal(env, orc.state, f"(config 5, step {t})")
            assert torch.equal(fused.state.blob, env.state.blob) and torch.equal(fused.obs, env.obs)
    assert env.stats()["episodes"] == int(orc.state.stats[0]) > B


# ---- episode scores, non-finite counter, trajectory export (SURVEY.md 8f rows 3 and 4) --------------------------------


@pytest.mark.parametrize("kind,n", [("multi", 5), ("multi", 8), ("multi", 32), ("single", 1)])
def test_score_accumulators_match_the_oracle(kind, n):
    """`score += rewards[0]` (test_sac_multi.py:105) and `total_score += rewards[i] * (1 - dones[i])` (:152-156) kept per
    env on the device and folded into the totals at every auto-reset — against the oracle's float64 accumulation."""
    import gym_uav_collision_avoidance_b200 as G
    from oracle import oracle as O

    B, steps = 600, 150
    if kind == "single":
        kw = dict(reset_mode=O.RESET_ON_ANY_DONE, max_episode_steps=45, seed=7)
        env = G.BatchedUAVWorld2D(B, track_scores=True, **kw)
        cfg = O.single_config(B, track_scores=1, **kw)
        amax = 12.0
    else:
        kw = dict(reset_mode=O.RESET_ON_DONE0, max_episode_steps=45, seed=7, x_size=18.0, y_size=18.0)
        env = G.BatchedMultiUAVWorld2D(B, num_agents=n, track_scores=True, **kw)
        cfg = O.multi_config(B, n, track_scores=1, **kw)
        amax = 10.0
    orc = O.Oracle(cfg, nthreads=4)
    env.reset()
    orc.reset()
    gen = torch.Generator(device="cuda").manual_seed(n)
    for t in range(steps):
        a = torch.rand((B, n, 2), generator=gen, device="cuda") * 2 * amax - amax
        if kind == "multi" and t % 2:  # head for the targets: reaches (+10) and collisions (-2) enter the scores
            a = ((env.state.tgt - env.state.pos) * 2).clamp(-amax, amax).contiguous()
        env.step(a)
        orc.step(a.cpu().numpy())
        if t % 10 == 0 or t == steps - 1:
            sc, so = env.score.cpu().numpy(), orc.state.score
            assert np.allclose(sc, so, rtol=2e-5, atol=2e-4), f"running scores differ at step {t}: {np.abs(sc - so).max()}"
    s = env.stats()
    of = orc.state.stats.view(np.float64)
    assert s["episodes"] == int(orc.state.stats[0]) > B
    assert np.isclose(s["score0_sum"], of[4], rtol=1e-5, atol=1e-2) and np.isclose(s["score_live_sum"], of[5], rtol=1e-5, atol=1e-2)
    assert s["nonfinite"] == int(orc.state.stats[6]) == 0
    if kind == "multi":
        ro = G.BatchedRollout(env, None)
        ev = ro.evaluation_summary()
        assert np.isclose(ev["Avg_Score"], of[5] / (n * s["episodes"]), rtol=1e-5)
        assert np.isclose(ev["mean_episode_score"], of[4] / s["episodes"], rtol=1e-5)
        assert ev["SR"] == s["reach"] / (n * s["episodes"]) and ev["CR"] == s["collisions"] / (n * s["episodes"])


def test_scores_are_off_by_default_and_nonfinite_steps_are_counted():
    import gym_uav_collision_avoidance_b200 as G
    from oracle import oracle as O

    B, N = 64, 4
    env = G.BatchedMultiUAVWorld2D(B, num_agents=N, seed=1)
    orc = O.Oracle(O.multi_config(B, N, seed=1))
    env.reset()
    orc.reset()
    # the reference divides by init_distance (multi_uav_world_2d.py:189-194): a UAV injected ON its target with
    # init_distance 0 gets a NaN reward (0 * inf), which the reference silently propagates
    env.state.tgt[:8, 0] = env.state.pos[:8, 0]
    env.state.init[:8, 0] = 0.0
    env.state.prev[:8, 0] = 0.0
    orc.state.tgt[:8, 0] = orc.state.pos[:8, 0]
    orc.state.init[:8, 0] = 0.0
    orc.state.prev[:8, 0] = 0.0
    zero = torch.zeros((B, N, 2), device="cuda")
    env.step(zero)
    out = orc.step(zero.cpu().numpy())
    bad_ref = int((~np.isfinite(out["reward"])).sum())
    assert bad_ref == 8 and int(orc.state.stats[6]) == 8
    assert env.stats()["nonfinite"] == 8 and int((~torch.isfinite(env.reward)).sum()) == 8
    assert float(env.score.abs().sum()) == 0.0  # track_scores is off: nothing accumulated


def test_export_trajectory_is_the_plotting_scripts_record():
    """pos / target / done per step for an env slice (test_sac_multi_plot_trajectory.py:46-68), equal to stepping by hand."""
    import gym_uav_collision_avoidance_b200 as G

    B, N, T = 128, 6, 40
    kw = dict(num_agents=N, seed=5, reset_mode=G.RESET_ON_DONE0, max_episode_steps=25)
    e1, e2 = G.BatchedMultiUAVWorld2D(B, **kw), G.BatchedMultiUAVWorld2D(B, **kw)
    e1.reset()
    e2.reset()
    gen = torch.Generator(device="cuda").manual_seed(0)
    acts = torch.rand((T, B, N, 2), generator=gen, device="cuda") * 20 - 10
    tr = e1.export_trajectory(slice(10, 14), T, actions=acts)
    assert tr["pos"].shape == (T + 1, 4, N, 2) and tr["target"].shape == (T + 1, 4, N, 2) and tr["done"].shape == (T, 4, N)
    assert tr["reset"].shape == (T, 4) and tr["done_step"].shape == (4, N) and list(tr["env_index"]) == [10, 11, 12, 13]
    assert np.array_equal(tr["pos"][0], e2.state.pos[10:14].cpu().numpy())
    for t in range(T):
        _, r, d, info = e2.step(acts[t])
        assert np.array_equal(tr["pos"][t + 1], e2.state.pos[10:14].cpu().numpy())
        assert np.array_equal(tr["target"][t + 1], e2.state.tgt[10:14].cpu().numpy())
        assert np.array_equal(tr["done"][t], d[10:14].cpu().numpy().astype(bool)) and np.array_equal(tr["reward"][t], r[10:14].cpu().numpy())
        assert np.array_equal(tr["reset"][t], info["reset_mask"][10:14].cpu().numpy().astype(bool))
    assert tr["reset"].any(), "the slice should have gone through an auto-reset (25-step limit)"
    ds = tr["done_step"]
    assert ((ds == -1) | (tr["done"][np.clip(ds, 0, T - 1), np.arange(4)[:, None], np.arange(N)[None, :]])).all()
    # random-stream and policy-driven variants run too
    tr2 = e1.export_trajectory(3, 5)
    assert tr2["pos"].shape == (6, 1, N, 2)
    tr3 = e1.export_trajectory(slice(0, 2), 5, policy=lambda obs: torch.zeros((B, N, 2), device="cuda"))
    assert tr3["velocity"].shape == (6, 2, N, 2)


def test_compat_render_records_a_trajectory():
    from gym_uav_collision_avoidance_b200 import compat

    env = compat.MultiUAVWorld2D(num_agents=3, seed=2)
    env.reset()
    for _ in range(5):
        env.step([np.array([1.0, 0.0])] * 3)
        assert env.render() is None
    tr = env.export_trajectory()
    assert tr["pos"].shape == (5, 3, 2) and tr["target"].shape == (5, 3, 2) and tr["done"].shape == (5, 3)
    assert list(tr["step"]) == [1, 2, 3, 4, 5]
    assert np.array_equal(tr["pos"][-1], np.stack([a.location for a in env.agent_list]))
    env.close()
