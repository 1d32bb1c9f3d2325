"""GPU: the CUDA path (through the C-ABI / torch custom ops) against the oracle and the reference's golden vectors.

Bar (BASELINE.json north_star): done / collision / reset flags, counters and env indexing bit-exact; positions
(float32) and velocities (float64) bit-exact as well (they feed the flags); rewards and observations within
1e-5 relative (+1e-6 absolute floor for values that cancel to ~0), angle features compared on the circle.
"""
import numpy as np
import pytest
import torch

from oracle import oracle as O

from _golden import Case, golden_names, obs_close

pytestmark = pytest.mark.gpu

RTOL, ATOL = 1e-5, 1e-6


def _b200():
    import gym_uav_collision_avoidance_b200 as G

    return G


def close(a, b, rtol=RTOL, atol=ATOL):
    a = np.asarray(a, np.float64)
    b = np.asarray(b, np.float64)
    return np.abs(a - b) <= rtol * np.abs(b) + atol


def make_env(cfg: O.Config, **kw):
    G = _b200()
    common = dict(seed=int(cfg.seed), reset_mode=cfg.reset_mode, max_episode_steps=cfg.max_episode_steps,
                  reset_source=cfg.reset_source, env_index_base=int(cfg.env_index_base))
    common.update(kw)
    if cfg.kind == O.KIND_SINGLE:
        return G.BatchedUAVWorld2D(cfg.num_envs, x_size=cfg.x_size, y_size=cfg.y_size, max_speed=cfg.max_speed,
                                   max_acceleration=cfg.max_acceleration,
                                   float32_first_step=bool(cfg.single_f32_first_step), **common)
    return G.BatchedMultiUAVWorld2D(cfg.num_envs, x_size=cfg.x_size, y_size=cfg.y_size, max_speed=cfg.max_speed,
                                    max_acceleration=cfg.max_acceleration, num_agents=cfg.num_agents,
                                    collider_radius=cfg.collider_radius, d_sense=cfg.d_sense,
                                    hard_collision_radius=cfg.hard_collision_radius, circular=bool(cfg.circular), **common)


def load_state(blob, st: O.State):
    blob.load_arrays(pos=st.pos, vel=st.vel, tgt=st.tgt, init=st.init, prev=st.prev, flags=st.flags, steps=st.steps,
                     reach=st.reach, coll=st.coll, episode=st.episode.astype(np.int64))


def assert_state_equal(env, st: O.State, where=""):
    h = env.state.to_host()
    for f in ("pos", "vel", "tgt", "init", "prev", "flags", "steps", "reach", "coll"):
        assert np.array_equal(h[f], getattr(st, f)), f"state field {f} differs {where}"
    assert np.array_equal(h["episode"].astype(np.uint32), st.episode), f"episode counter differs {where}"


def assert_outputs(env, out, where="", obs_ref=None):
    obs_ref = out["obs"] if obs_ref is None else obs_ref
    assert np.array_equal(env.done.cpu().numpy(), out["done"]), f"done flags differ {where}"
    assert np.array_equal(env.reset_mask.cpu().numpy(), out["reset_mask"]), f"reset mask differs {where}"
    rew = env.reward.cpu().numpy()
    ok = close(rew, out["reward"])
    assert ok.all(), f"reward outside tolerance {where}: {rew[~ok][:4]} vs {out['reward'][~ok][:4]}"
    obs = env.obs.cpu().numpy()
    ok = obs_close(obs, obs_ref, RTOL, ATOL)
    assert ok.all(), f"obs outside tolerance {where}: idx {np.argwhere(~ok)[:4].tolist()} {obs[~ok][:4]} vs {obs_ref[~ok][:4]}"


# ---- golden vectors produced by the literal reference ----------------------------------------------------------


@pytest.mark.parametrize("name", golden_names())
def test_cuda_matches_reference_golden(name):
    case = Case(name)
    cfg = case.config()
    env = make_env(cfg)
    env.enable_final_obs()
    load_state(env.state, case.init_state())
    pool_host = case.pool_state()
    load_state(env.make_pool(pool_host.B), pool_host)
    z = case.z
    obs0 = env.observe().cpu().numpy()
    assert obs_close(obs0, z["obs0"], RTOL, ATOL).all()
    for t in range(case.T):
        if "action64" in z.files:  # f64act_*: float64 actions that float32 cannot hold, through uavca_step_f64
            env.step_f64(torch.from_numpy(z["action64"][t]).cuda(), evaluate=case.evaluate)
        else:
            a = torch.from_numpy(z["action"][t]).cuda()
            if case.kind == "single":
                env.step(a)
            else:
                env.step(a, evaluate=case.evaluate)
        w = f"({name}, step {t})"
        assert np.array_equal(env.done.cpu().numpy(), z["done"][t]), f"done flags differ {w}"
        assert np.array_equal(env.reset_mask.cpu().numpy(), z["reset_mask"][t]), f"reset mask differs {w}"
        h = env.state.to_host()
        assert np.array_equal(h["pos"], z["pos"][t]), f"positions differ {w}"
        assert np.array_equal(h["vel"], z["vel"][t]), f"velocities differ {w}"
        assert np.array_equal(h["prev"], z["prev"][t]), f"prev_distance differs {w}"
        assert np.array_equal(h["steps"], z["steps"][t]), f"env.steps differs {w}"
        if case.kind == "multi":
            assert np.array_equal(h["flags"], z["flags"][t]), f"parked/collided latches differ {w}"
            assert np.array_equal(h["reach"], z["reach"][t]), f"target_reach_count differs {w}"
            assert np.array_equal(h["coll"], z["coll"][t]), f"collision_count differs {w}"
        else:
            assert np.array_equal(env.distance.cpu().numpy(), z["distance"][t]), f"info distance differs {w}"
        assert close(env.reward.cpu().numpy(), z["reward"][t]).all(), f"reward {w}"
        assert obs_close(env.obs.cpu().numpy(), z["obs"][t], RTOL, ATOL).all(), f"obs {w}"
        assert obs_close(env.final_obs.cpu().numpy(), case.final_obs(t), RTOL, ATOL).all(), f"final obs {w}"


@pytest.mark.parametrize("N,circular", [(5, False), (32, False), (40, False), (6, True)])
def test_float64_actions_that_float32_holds_step_like_float32_actions(N, circular):
    """uavca_step_f64 on every kernel that serves it (warp kernel, general kernel for N > 32 and for the float64 world):
    float64 actions whose values float32 holds exactly must give the very state the float32 entry point gives."""
    G = _b200()
    B = 64
    kw = dict(num_agents=N, reset_mode=G.RESET_ON_DONE0, max_episode_steps=40, seed=17, circular=circular)
    e32, e64 = G.BatchedMultiUAVWorld2D(B, **kw), G.BatchedMultiUAVWorld2D(B, **kw)
    e32.reset(); e64.reset()
    gen = torch.Generator(device="cuda").manual_seed(5)
    for t in range(120):
        a = (torch.rand((B, N, 2), generator=gen, device="cuda") * 20 - 10)
        e32.step(a)
        e64.step_f64(a.double())
        assert torch.equal(e32.state.blob, e64.state.blob), f"state differs at step {t}"
        assert torch.equal(e32.done, e64.done) and torch.equal(e32.reset_mask, e64.reset_mask)
        assert torch.equal(e32.obs, e64.obs) and torch.equal(e32.reward, e64.reward)
    assert e32.stats()["episodes"] > 0


# ---- rollouts against the oracle, with Philox auto-reset on both sides ----------------------------------------


def rollout_vs_oracle(cfg: O.Config, steps, seed, evaluate=False, crowd=None, nthreads=8, check_every=1):
    """Device and oracle start from the same Philox reset and see the same actions; compare every step."""
    env = make_env(cfg)
    orc = O.Oracle(cfg, nthreads=nthreads)
    obs_dev = env.reset().cpu().numpy()
    obs_orc = orc.reset()
    assert_state_equal(env, orc.state, "after reset")
    assert obs_close(obs_dev, obs_orc, RTOL, ATOL).all()
    gen = torch.Generator(device="cuda").manual_seed(seed)
    B, N = cfg.num_envs, cfg.num_agents
    amax = float(cfg.max_speed)
    events = dict(done=0, resets=0)
    for t in range(steps):
        a = (torch.rand((B, N, 2), generator=gen, device="cuda") * 2 - 1) * amax
        if crowd is not None:  # pull UAVs towards the origin so that they meet
            a = (a * 0.3 - env.state.pos * crowd).clamp(-amax, amax).contiguous()
        if cfg.kind == O.KIND_SINGLE:
            env.step(a)
        else:
            env.step(a, evaluate=evaluate)
        out = orc.step(a.cpu().numpy(), evaluate=evaluate)
        events["done"] += int(out["done"].sum())
        events["resets"] += int(out["reset_mask"].sum())
        if t % check_every == 0 or t == steps - 1:
            assert_outputs(env, out, f"(step {t})")
            assert_state_equal(env, orc.state, f"(step {t})")
    st = env.stats()
    assert st["episodes"] == int(orc.state.stats[0]) and st["reach"] == int(orc.state.stats[1])
    assert st["collisions"] == int(orc.state.stats[2]) and st["steps"] == int(orc.state.stats[3])
    assert st["live_steps"] == int(orc.state.steps.sum())
    return events, orc


@pytest.mark.parametrize("n,B", [pytest.param(n, 257, id=str(n)) for n in [1, 2, 3, 4, 5, 7, 8, 9, 10, 11, 12, 13, 16, 17, 24, 31, 32]]
                         + [(7, 1), (16, 3)])
def test_multi_rollout_all_agent_counts(n, B):
    """Every N in 1..32 maps to a different lane layout (specialised or generic kernel, ragged last warp).  B = 257 is not
    a multiple of any envs-per-warp; B = 1 and B = 3 fill less than one CTA (a partial warp, then idle warps)."""
    cfg = O.multi_config(B, n, reset_mode=O.RESET_ON_DONE0, max_episode_steps=40, seed=1000 + n, x_size=24.0, y_size=24.0)
    ev, _ = rollout_vs_oracle(cfg, steps=120, seed=n, crowd=0.4)
    assert ev["resets"] > 0


@pytest.mark.parametrize("n", [2, 5, 8, 16, 32])
@pytest.mark.parametrize("mode", [O.RESET_ON_ANY_DONE, O.RESET_ON_ALL_DONE, O.RESET_ON_ANY_DONE | O.RESET_ON_DONE0])
def test_multi_rollout_reset_modes(n, mode):
    """any(dones) / all(dones) with several envs per warp: an env's reset decision must only see its own done bits
    (reset_mask, episode and step counters bit-exact against the oracle's want_reset)."""
    # a small box and random actions: UAVs leave it all the time (done = out of bounds), one by one
    cfg = O.multi_config(515, n, reset_mode=mode, max_episode_steps=60, seed=300 + n, x_size=9.0, y_size=9.0,
                         collider_radius=0.3, hard_collision_radius=0.15)
    ev, orc = rollout_vs_oracle(cfg, steps=150, seed=40 + n)
    assert ev["resets"] > 515 and ev["done"] > 0
    if mode & O.RESET_ON_ANY_DONE:
        assert int(orc.state.stats[3]) < 60 * int(orc.state.stats[0]), "some episodes should end before the step limit"


def test_multi_rollout_crowded_collisions_and_reaches():
    cfg = O.multi_config(2048, 8, reset_mode=O.RESET_ON_ALL_DONE, max_episode_steps=300, seed=77, x_size=16.0, y_size=16.0)
    ev, orc = rollout_vs_oracle(cfg, steps=400, seed=3, crowd=1.2)
    assert int(orc.state.stats[2]) + int(orc.state.coll.sum()) > 100, "scenario should produce hard collisions"


def test_multi_rollout_evaluate_mode():
    cfg = O.multi_config(1024, 5, reset_mode=O.RESET_ON_ALL_DONE, max_episode_steps=200, seed=5)
    rollout_vs_oracle(cfg, steps=250, seed=4, evaluate=True)


def test_multi_c3_1000_step_rollout_subset():
    """BASELINE config 3 (N=8, B=65,536) for 1,000 steps on the GPU; the oracle follows a contiguous 1,024-env
    window (envs are independent and the Philox streams are keyed by the global env index)."""
    G = _b200()
    B, N, W, START = 65536, 8, 1024, 30000
    kw = dict(reset_mode=O.RESET_ON_DONE0, max_episode_steps=1500, seed=0x5EED)
    env = G.BatchedMultiUAVWorld2D(B, num_agents=N, **kw)
    cfg = O.multi_config(W, N, env_index_base=START, **kw)
    orc = O.Oracle(cfg, nthreads=8)
    env.reset()
    orc.reset()
    gen = torch.Generator(device="cuda").manual_seed(1234)
    sl = slice(START, START + W)
    mism = 0
    for t in range(1000):
        a = (torch.rand((B, N, 2), generator=gen, device="cuda") * 20 - 10)
        obs, rew, done, info = env.step(a)
        out = orc.step(a[sl].cpu().numpy())
        assert np.array_equal(done[sl].cpu().numpy(), out["done"]), f"done flags differ at step {t}"
        assert np.array_equal(info["reset_mask"][sl].cpu().numpy(), out["reset_mask"]), f"reset mask differs at step {t}"
        if t % 10 == 0 or t == 999:
            assert np.array_equal(env.state.pos[sl].cpu().numpy(), orc.state.pos), f"positions differ at step {t}"
            assert np.array_equal(env.state.vel[sl].cpu().numpy(), orc.state.vel), f"velocities differ at step {t}"
            mism += int((~close(rew[sl].cpu().numpy(), out["reward"])).sum())
            mism += int((~obs_close(obs[sl].cpu().numpy(), out["obs"], RTOL, ATOL)).sum())
    assert mism == 0
    assert int(orc.state.stats[0]) > 100, "the window should have gone through many episodes"


def test_multi_c3_full_batch_1000_steps():
    """The north-star criterion taken literally: BASELINE config 3 — ALL 65,536 envs x 8 UAVs — for 1,000 steps with
    auto-reset, against the oracle on identical states and actions: done flags and reset masks bit-exact at every step,
    positions / velocities / latches / counters bit-exact and rewards / observations within 1e-5 at checkpoints."""
    G = _b200()
    B, N = 65536, 8
    kw = dict(reset_mode=O.RESET_ON_DONE0, max_episode_steps=400, seed=0xC3)
    env = G.BatchedMultiUAVWorld2D(B, num_agents=N, **kw)
    orc = O.Oracle(O.multi_config(B, N, **kw), nthreads=O.max_threads())
    env.reset()
    orc.reset()
    gen = torch.Generator(device="cuda").manual_seed(77)
    flagged = 0
    for t in range(1000):
        a = torch.rand((B, N, 2), generator=gen, device="cuda") * 20 - 10
        obs, rew, done, info = env.step(a)
        out = orc.step(a.cpu().numpy())
        assert np.array_equal(done.cpu().numpy(), out["done"]), f"done flags differ at step {t}"
        assert np.array_equal(info["reset_mask"].cpu().numpy(), out["reset_mask"]), f"reset mask differs at step {t}"
        flagged += int(out["done"].sum())
        if t % 50 == 49 or t < 3:
            assert_state_equal(env, orc.state, f"(step {t})")
            assert close(rew.cpu().numpy(), out["reward"]).all(), f"reward at step {t}"
            assert obs_close(obs.cpu().numpy(), out["obs"], RTOL, ATOL).all(), f"observation at step {t}"
    st = env.stats()
    assert st["episodes"] == int(orc.state.stats[0]) > 2 * B and st["collisions"] == int(orc.state.stats[2]) > 0
    assert flagged > 100000


def test_multi_c3_full_batch_short():
    """All 65,536 envs of config 3 against the oracle for 30 steps."""
    cfg = O.multi_config(65536, 8, reset_mode=O.RESET_ON_DONE0, max_episode_steps=20, seed=9)
    rollout_vs_oracle(cfg, steps=30, seed=11, check_every=5)


def test_multi_n32_rollout():
    cfg = O.multi_config(4096, 32, reset_mode=O.RESET_ON_DONE0, max_episode_steps=100, seed=32)
    rollout_vs_oracle(cfg, steps=150, seed=6, check_every=3)


@pytest.mark.parametrize("limit", [1500, 60])
def test_multi_c4_shard_1000_step_window(limit):
    """BASELINE configs[3] at the size one of eight GPUs holds (N=32, 131,072 envs) for 1,000 steps; the oracle follows a
    4,096-env window keyed by the global env index.  N=32 is where the key-based neighbour selection falls back to the
    exact one most often and where collisions, parking and resets interact: done flags and reset masks bit-exact at every
    step, state bit-exact and outputs within tolerance at checkpoints; with the reference's 1,500-step limit and with a
    short one (many auto-resets)."""
    G = _b200()
    B, N, W, START, BASE = 131072, 32, 4096, 70000, 5 * 131072  # the shard of rank 5 of 8
    kw = dict(reset_mode=O.RESET_ON_DONE0, max_episode_steps=limit, seed=0xC4 + limit)
    env = G.BatchedMultiUAVWorld2D(B, num_agents=N, env_index_base=BASE, **kw)
    orc = O.Oracle(O.multi_config(W, N, env_index_base=BASE + START, **kw), nthreads=O.max_threads())
    env.reset()
    orc.reset()
    sl = slice(START, START + W)
    gen = torch.Generator(device="cuda").manual_seed(limit)
    events = 0
    for t in range(1000):
        a = torch.rand((B, N, 2), generator=gen, device="cuda") * 20 - 10
        if t % 3 == 0:  # every third step steer towards the targets, so that UAVs meet, park and get hit
            a = ((env.state.tgt - env.state.pos) * 2.0 + a * 0.1).clamp(-10, 10).contiguous()
        obs, rew, done, info = env.step(a)
        out = orc.step(a[sl].cpu().numpy())
        assert np.array_equal(done[sl].cpu().numpy(), out["done"]), f"done flags differ at step {t}"
        assert np.array_equal(info["reset_mask"][sl].cpu().numpy(), out["reset_mask"]), f"reset mask differs at step {t}"
        events += int(out["done"].sum())
        if t % 20 == 0 or t == 999:
            assert np.array_equal(env.state.pos[sl].cpu().numpy(), orc.state.pos), f"positions differ at step {t}"
            assert np.array_equal(env.state.vel[sl].cpu().numpy(), orc.state.vel), f"velocities differ at step {t}"
            assert np.array_equal(env.state.flags[sl].cpu().numpy(), orc.state.flags), f"latches differ at step {t}"
            assert np.array_equal(env.state.coll[sl].cpu().numpy(), orc.state.coll), f"collision counts differ at step {t}"
            assert close(rew[sl].cpu().numpy(), out["reward"]).all(), f"reward at step {t}"
            assert obs_close(obs[sl].cpu().numpy(), out["obs"], RTOL, ATOL).all(), f"observation at step {t}"
    assert events > 1000 and int(orc.state.stats[0]) >= (W * (1000 // limit) if limit < 1000 else 1)
    assert int(orc.state.stats[2]) + int(orc.state.coll.sum()) > 0, "the window should have seen hard collisions"


@pytest.mark.parametrize("trial", range(16))
def test_multi_rollout_random_constructor_arguments(trial):
    """Non-default worlds: box, speed / acceleration bounds, collider and hard-collision radii and sensing range drawn
    at random (including a sensing range shorter than the collision distance).  Every threshold the kernel tests in
    squared-distance space is derived on the host from these; the oracle uses the reference's own comparisons."""
    rng = np.random.default_rng(7000 + trial)
    n = int(rng.choice([2, 3, 5, 8, 11, 16, 32]))
    r = float(rng.uniform(0.3, 3.0))
    kw = dict(x_size=float(rng.uniform(8, 120)), y_size=float(rng.uniform(8, 120)), max_speed=float(rng.uniform(2, 30)),
              max_acceleration=float(rng.uniform(1, 20)), collider_radius=r,
              hard_collision_radius=float(rng.uniform(0.1, 1.0) * r),
              d_sense=float(rng.choice([rng.uniform(0.5, 2.0) * r, rng.uniform(5, 60)])))
    cfg = O.multi_config(300, n, reset_mode=O.RESET_ON_DONE0, max_episode_steps=80, seed=trial, **kw)
    ev, _ = rollout_vs_oracle(cfg, steps=100, seed=trial, crowd=float(rng.choice([0.0, 0.5, 1.5])) or None, check_every=2)
    assert ev["resets"] > 0


def test_multi_c4_full_size_properties_and_window():
    """BASELINE config 4's shape on ONE GPU (N=32, B=1,048,576: 33.5 M UAVs, ~3.2 GB): a 2,048-env window against the
    oracle plus size-independent properties over the whole batch (flag ranges, observation bounds, reset mask ==
    dones[0] | step limit, counters conserved, auto-reset envs respect the reference's separation constraints)."""
    G = _b200()
    B, N, W, START = 1048576, 32, 2048, 777777
    kw = dict(reset_mode=O.RESET_ON_DONE0, max_episode_steps=6, seed=0xC4)
    env = G.BatchedMultiUAVWorld2D(B, num_agents=N, **kw)
    orc = O.Oracle(O.multi_config(W, N, env_index_base=START, **kw), nthreads=8)
    env.reset()
    orc.reset()
    sl = slice(START, START + W)
    gen = torch.Generator(device="cuda").manual_seed(4)
    total_steps = 0
    for t in range(8):
        a = torch.rand((B, N, 2), generator=gen, device="cuda") * 20 - 10
        steps_prev = env.state.steps.clone()
        obs, rew, done, info = env.step(a)
        out = orc.step(a[sl].cpu().numpy())
        assert np.array_equal(done[sl].cpu().numpy(), out["done"]) and np.array_equal(info["reset_mask"][sl].cpu().numpy(), out["reset_mask"])
        assert np.array_equal(env.state.pos[sl].cpu().numpy(), orc.state.pos)
        assert close(rew[sl].cpu().numpy(), out["reward"]).all() and obs_close(obs[sl].cpu().numpy(), out["obs"], RTOL, ATOL).all()
        # whole batch
        assert int(env.state.flags.max()) <= 3 and int(done.max()) <= 1
        assert bool(torch.isfinite(obs).all()) and bool(torch.isfinite(rew).all())
        assert float(obs[..., 0].min()) >= 0 and float(obs[..., 0].max()) <= 1.0 + 1e-6  # speed / ||v_max||
        for k in (1, 3, 5, 6, 8, 9):
            assert float(obs[..., k].abs().max()) <= 1.0 + 1e-6
        expect = (done[:, 0] != 0) | (steps_prev + 1 >= 6)  # training protocol: dones[0] or the step limit
        assert torch.equal(info["reset_mask"].bool(), expect)
        assert torch.equal(env.state.steps, torch.where(expect, torch.zeros_like(steps_prev), steps_prev + 1))
        total_steps += B
    st = env.stats()
    assert st["steps"] + st["live_steps"] == total_steps and st["episodes"] >= B  # every env hit the 6-step limit once
    # envs that auto-reset start again from separated positions (multi_uav_world_2d.py:127-137)
    m = info["reset_mask"].bool()
    p = env.state.pos[m][:4096].double()
    d = (p[:, :, None, :] - p[:, None, :, :]).norm(dim=-1) + torch.eye(N, device="cuda", dtype=torch.float64) * 1e3
    assert float(d.min()) > 2.0 - 1e-6
    assert_state_equal_window = env.state.vel[sl].cpu().numpy()
    assert np.array_equal(assert_state_equal_window, orc.state.vel)


@pytest.mark.parametrize("n", [11, 17, 20, 24, 25])
def test_cta_packed_kernel_and_warp_kernel_agree(monkeypatch, n):
    """17 <= N <= 25 runs step_multi_cta_kernel (envs packed across the warps of a CTA) by default and the one-env-per-
    warp kernel under UAVCA_STEP_PATH=plain (which uavca_rollout also uses): both against the oracle, all three reset
    triggers, and bit for bit against each other (scores included) on a batch with a ragged last CTA."""
    for mode in (O.RESET_ON_DONE0, O.RESET_ON_ANY_DONE, O.RESET_ON_ALL_DONE):
        for path in ("lanes", "plain"):
            monkeypatch.setenv("UAVCA_STEP_PATH", path)
            cfg = O.multi_config(1031, n, reset_mode=mode, max_episode_steps=30, seed=300 + n + mode)
            ev, _ = rollout_vs_oracle(cfg, steps=45, seed=n + mode, check_every=3)
            assert ev["resets"] > 0
    G = _b200()
    B = 40003
    kw = dict(num_agents=n, seed=99, reset_mode=O.RESET_ON_DONE0, max_episode_steps=9, track_scores=True)
    monkeypatch.setenv("UAVCA_STEP_PATH", "plain")
    e1 = G.BatchedMultiUAVWorld2D(B, **kw)
    monkeypatch.setenv("UAVCA_STEP_PATH", "lanes")
    e2 = G.BatchedMultiUAVWorld2D(B, **kw)
    e1.reset()
    e2.reset()
    gen = torch.Generator(device="cuda").manual_seed(6)
    for t in range(12):
        a = torch.rand((B, n, 2), generator=gen, device="cuda") * 20 - 10
        e1.step(a)
        e2.step(a)
        assert torch.equal(e1.obs, e2.obs) and torch.equal(e1.reward, e2.reward) and torch.equal(e1.done, e2.done)
        assert torch.equal(e1.reset_mask, e2.reset_mask)
    h1, h2 = e1.state.to_host(), e2.state.to_host()
    for f in e1.state.FIELDS:
        assert np.array_equal(h1[f], h2[f]), f"state field {f} differs"
    assert torch.equal(e1.score, e2.score)  # per-env running scores: same summation order in both kernels
    s1, s2 = e1.stats(), e2.stats()
    for k in s1:  # the score totals are double atomics over all envs: equal up to the order of the additions
        assert s1[k] == s2[k] or (k.startswith("score") and abs(s1[k] - s2[k]) <= 1e-9 * abs(s1[k])), k


@pytest.mark.parametrize("f32", [0, 1])
def test_single_rollout(f32):
    cfg = O.single_config(65536, reset_mode=O.RESET_ON_ANY_DONE, max_episode_steps=500, seed=21 + f32,
                          single_f32_first_step=f32)
    ev, _ = rollout_vs_oracle(cfg, steps=300, seed=8 + f32, check_every=10)
    assert ev["resets"] > 100


def test_single_1000_step_rollout():
    """BASELINE config 2 (single UAV, B=65,536) for 1,000 steps; oracle follows a 4,096-env window."""
    G = _b200()
    B, W, START = 65536, 65536, 0  # BASELINE config 2, the whole batch
    kw = dict(reset_mode=O.RESET_ON_ANY_DONE, seed=77)
    env = G.BatchedUAVWorld2D(B, **kw)
    orc = O.Oracle(O.single_config(W, env_index_base=START, **kw), nthreads=8)
    env.reset()
    orc.reset()
    gen = torch.Generator(device="cuda").manual_seed(99)
    sl = slice(START, START + W)
    for t in range(1000):
        a = torch.rand((B, 1, 2), generator=gen, device="cuda") * 24 - 12
        obs, rew, done, info = env.step(a)
        out = orc.step(a[sl].cpu().numpy())
        assert np.array_equal(done[sl].cpu().numpy(), out["done"]), f"done flags differ at step {t}"
        if t % 10 == 0 or t == 999:
            assert np.array_equal(env.state.pos[sl].cpu().numpy(), orc.state.pos)
            assert np.array_equal(env.state.vel[sl].cpu().numpy(), orc.state.vel)
            assert close(rew[sl].cpu().numpy(), out["reward"]).all()
            assert obs_close(obs[sl].cpu().numpy(), out["obs"], RTOL, ATOL).all()
            assert np.array_equal(info["distance"][sl].cpu().numpy(), out["distance"])


def _edge_states(B, N, radius, rng, spread_ulps=6):
    """Stationary UAVs whose pair distances sit within a few float32 ulps of `radius` (zero velocity + zero action
    keep every position fixed, so the step tests exactly these distances)."""
    st = O.State(B, N)
    centre = rng.uniform(-6.0, 6.0, size=(B, 1, 2))
    phi = rng.uniform(0, 2 * np.pi, size=(B, N))
    # UAV 0 in the middle, the others on a circle of ~radius around it (their mutual distances are arbitrary)
    r = radius * (1.0 + rng.integers(-spread_ulps, spread_ulps + 1, size=(B, N)) * 2.0 ** -24)
    off = np.stack([r * np.cos(phi), r * np.sin(phi)], axis=-1)
    off[:, 0] = 0.0
    st.pos[...] = (centre + off).astype(np.float32)
    st.tgt[...] = (st.pos.astype(np.float64) + rng.uniform(5.0, 7.0, size=(B, N, 2))).astype(np.float32)
    d = st.tgt - st.pos
    st.init[...] = np.sqrt(d[..., 0] * d[..., 0] + d[..., 1] * d[..., 1], dtype=np.float32)
    st.prev[...] = st.init
    return st


@pytest.mark.parametrize("radius,n", [(2.0, 2), (1.0, 2), (15.0, 2), (2.0, 5), (1.0, 8), (2.0, 32)])
def test_threshold_edges_are_bit_exact(radius, n):
    """Soft collision (d <= 2.0), hard collision (d <= 1.0) and sensing range (d < 15) decided on distances within
    a few ulps of the threshold: the float32 norm must be formed exactly as the reference does (products and sum
    rounded separately; a fused multiply-add flips ~8 % of these)."""
    B = 131072 if n <= 8 else 8192
    cfg = O.multi_config(B, n, x_size=60.0, y_size=60.0, seed=3)
    rng = np.random.default_rng(int(radius * 10) + n)
    st = _edge_states(B, n, radius, rng)
    d01 = st.pos[:, 1] - st.pos[:, 0]
    s01 = (d01[:, 0] * d01[:, 0] + d01[:, 1] * d01[:, 1]).astype(np.float32)
    lo, hi = np.float32(radius) ** 2 * np.float32(1 - 2e-6), np.float32(radius) ** 2 * np.float32(1 + 2e-6)
    assert ((s01 > lo) & (s01 < hi)).all(), "the crafted distances should hug the threshold"
    env = make_env(cfg)
    orc = O.Oracle(cfg, nthreads=8)
    orc.state = st.copy()
    load_state(env.state, st)
    zero = torch.zeros((B, n, 2), device="cuda")
    for t in range(2):  # second step: the collided latch is set, collision_count must not grow again
        env.step(zero)
        out = orc.step(zero.cpu().numpy())
        assert_outputs(env, out, f"(edge {radius}, step {t})")
        assert_state_equal(env, orc.state, f"(edge {radius}, step {t})")
    if radius == 2.0 and n == 2:
        hit = int((out["reward"] == -2.0).sum())
        assert 0 < hit < B * n, "the edge cases should fall on both sides of the threshold"


@pytest.mark.parametrize("n,spread", [(3, 40), (4, 24), (8, 64), (10, 100), (32, 48), (32, 400)])
def test_neighbour_order_across_the_key_granularity(n, spread):
    """The two nearest neighbours are picked with integer keys that keep 19 bits of the squared distance; lanes
    whose three best keys share truncated bits fall back to the exact selection.  Neighbour distances spread over
    a few tens of ulps around one radius sit on both sides of that granularity (32 ulps of the square): the order —
    hence observation features 4..9 — must still be the reference's."""
    B = 32768 if n <= 10 else 4096
    cfg = O.multi_config(B, n, x_size=60.0, y_size=60.0, seed=5)
    rng = np.random.default_rng(1000 * n + spread)
    st = _edge_states(B, n, 7.0, rng, spread_ulps=spread)
    env = make_env(cfg)
    orc = O.Oracle(cfg, nthreads=8)
    orc.state = st.copy()
    load_state(env.state, st)
    zero = torch.zeros((B, n, 2), device="cuda")
    env.step(zero)
    out = orc.step(zero.cpu().numpy())
    # exact ties have no defined order in the reference (SURVEY.md 7.3-4): compare only envs without one around UAV 0
    d = st.pos[:, 1:] - st.pos[:, :1]
    s = (d[..., 0] * d[..., 0] + d[..., 1] * d[..., 1]).astype(np.float32)
    srt = np.sort(s, axis=1)
    untied = (np.diff(srt[:, :4], axis=1) != 0).all(axis=1) if n > 2 else np.ones(B, bool)  # the three smallest (+1) differ
    assert untied.mean() > 0.5
    obs = env.obs.cpu().numpy()
    ok = obs_close(obs[untied, 0], out["obs"][untied, 0], RTOL, ATOL)
    assert ok.all(), f"UAV 0 neighbour features differ in {int((~ok.all(axis=-1)).sum())} envs"
    assert_state_equal(env, orc.state, "(key granularity)")
    assert np.array_equal(env.done.cpu().numpy(), out["done"])


def test_crafted_corner_states_match_the_oracle():
    """Hand-built states for the reference's quirks (SURVEY.md 8c): zero velocity (heading atan2(0,0) = 0), a UAV exactly
    on its target, denormal-tiny velocities, parked UAVs earning +10 and being hit by a neighbour, out-of-bounds UAVs
    that fly back in (done is not latched), UAVs with no neighbour in sensing range, evaluate=True."""
    N = 3
    scen = []

    def add(pos, vel, tgt, flags=(0, 0, 0), act=((0, 0),) * 3):
        scen.append(dict(pos=pos, vel=vel, tgt=tgt, flags=flags, act=act))

    far = [(-20.0, -20.0), (20.0, 20.0), (-20.0, 20.0)]  # nobody senses anybody (d_sense = 15)
    add(far, [(0, 0)] * 3, [(5, 5), (-5, -5), (0, 0)])                                   # zero velocity, zero action
    add(far, [(0, 0)] * 3, far, act=((1, 0), (0, 0), (-3, 2)))                            # sitting exactly on the target
    add(far, [(1e-40, 0), (0, -1e-39), (1e-41, 1e-41)], [(5, 5), (-5, -5), (0, 0)], act=((1e-40, 0), (0, -1e-39), (1e-41, 1e-41)))
    add([(0.1, 0.0), (1.5, 0.0), (20, 20)], [(0.05, 0), (-3, 0), (0, 0)], [(0.0, 0.0), (-10, 0), (0, 0)],
        flags=(1, 0, 0), act=((0, 0), (-10, 0), (0, 0)))                                  # parked UAV 0 gets hit by UAV 1
    add([(0.2, 0.1), (10, 10), (-10, 5)], [(0.1, 0.05), (0, 0), (0, 0)], [(0.0, 0.0), (0, 0), (0, 0)],
        act=((0, 0), (1, 1), (0, 0)))                                                     # UAV 0 reaches: slow and close
    add([(25.05, 0.0), (-25.2, 3.0), (0.0, 25.0)], [(-8, 0), (9, 0), (0, 5)], [(0, 0)] * 3,
        act=((-10, 0), (10, 0), (0, 10)))                                                 # outside flying in / on the edge flying out
    add([(0, 0), (1.0, 0.0), (0.0, 0.99)], [(0, 0)] * 3, [(9, 9), (-9, 9), (9, -9)], flags=(0, 2, 0))  # hard collisions, latch set on UAV 1
    add([(0, 0), (14.99, 0.0), (0.0, 15.0)], [(0, 0)] * 3, [(9, 9), (-9, 9), (9, -9)])     # sensing range: just inside / exactly on it
    B = len(scen)
    for evaluate in (False, True):
        cfg = O.multi_config(B, N, seed=1)
        st = O.State(B, N)
        for b, sc in enumerate(scen):
            st.pos[b] = np.asarray(sc["pos"], np.float32)
            st.vel[b] = np.asarray(sc["vel"], np.float64)
            st.tgt[b] = np.asarray(sc["tgt"], np.float32)
            st.flags[b] = np.asarray(sc["flags"], np.uint8)
        d = st.tgt - st.pos
        st.init[...] = np.maximum(np.sqrt(d[..., 0] * d[..., 0] + d[..., 1] * d[..., 1], dtype=np.float32), np.float32(3.0))
        st.prev[...] = np.sqrt(d[..., 0] * d[..., 0] + d[..., 1] * d[..., 1], dtype=np.float32)
        st.prev[st.flags & 1 == 1] = 0.0
        env = make_env(cfg)
        orc = O.Oracle(cfg)
        orc.state = st.copy()
        load_state(env.state, st)
        obs0 = env.observe().cpu().numpy()
        assert obs_close(obs0, orc.observe(), RTOL, ATOL).all(), "observation of the crafted states"
        act = torch.tensor([sc["act"] for sc in scen], dtype=torch.float32, device="cuda")
        for t in range(4):
            env.step(act, evaluate=evaluate)
            out = orc.step(act.cpu().numpy(), evaluate=evaluate)
            assert_outputs(env, out, f"(crafted, evaluate={evaluate}, step {t})")
            assert_state_equal(env, orc.state, f"(crafted, evaluate={evaluate}, step {t})")
        if not evaluate:
            assert out["done"][4, 0] == 1 and (orc.state.flags[4, 0] & 1)      # the slow, close UAV parked
            assert (orc.state.flags[6] & 2).all() and orc.state.coll[6] >= 2   # hard collisions counted once per UAV


# ---- reset ------------------------------------------------------------------------------------------------------


@pytest.mark.parametrize("n", [1, 6, 8, 32])
def test_reset_constraints_and_philox_parity(n):
    """Device reset == oracle reset (same Philox stream) bit-for-bit, and the reference's separation constraints
    (multi_uav_world_2d.py:126-153) hold."""
    B = 1000
    cfg = O.multi_config(B, n, seed=4242, x_size=20.0, y_size=20.0)
    env = make_env(cfg)
    orc = O.Oracle(cfg)
    obs = env.reset().cpu().numpy()
    obs_o = orc.reset()
    assert_state_equal(env, orc.state, "after reset")
    assert obs_close(obs, obs_o, RTOL, ATOL).all()
    pos, tgt = env.state.pos.cpu().numpy(), env.state.tgt.cpu().numpy()
    assert (np.abs(pos) <= 10).all() and (np.abs(tgt) <= 10).all()
    d_own = np.linalg.norm(tgt - pos, axis=-1)
    assert (d_own > 2.0).all()
    if n > 1:
        iu = np.triu_indices(n, 1)
        dp = np.linalg.norm(pos[:, :, None] - pos[:, None, :], axis=-1)[:, iu[0], iu[1]]
        dt = np.linalg.norm(tgt[:, :, None] - tgt[:, None, :], axis=-1)[:, iu[0], iu[1]]
        assert (dp > 2.0).all() and (dt > 2.0).all()
    # masked reset: only the chosen envs change, and their episode counter advances
    before = env.state.to_host()
    mask = np.zeros(B, np.uint8)
    mask[::3] = 1
    env.reset(torch.from_numpy(mask))
    orc.reset(mask)
    assert_state_equal(env, orc.state, "after masked reset")
    after = env.state.to_host()
    assert np.array_equal(after["pos"][mask == 0], before["pos"][mask == 0])
    assert (after["episode"][mask == 1] == 2).all() and (after["episode"][mask == 0] == 1).all()


def test_reset_is_uniform_over_the_box():
    G = _b200()
    env = G.BatchedMultiUAVWorld2D(200000, num_agents=1, seed=3)
    env.reset()
    pos = env.state.pos.cpu().numpy().reshape(-1, 2)
    assert abs(pos.mean()) < 0.1 and abs(pos.std() - 50 / np.sqrt(12)) < 0.1
    hist, _ = np.histogram(pos[:, 0], bins=10, range=(-25, 25))
    assert (np.abs(hist / len(pos) - 0.1) < 0.005).all()


def assert_state_equal_f64(env, st: O.State, where=""):
    h = env.state.to_host()
    for f in ("pos64", "tgt64", "init64", "prev64", "vel", "flags", "steps", "reach", "coll", "pos", "tgt", "init", "prev"):
        assert np.array_equal(h[f], getattr(st, f)), f"state field {f} differs {where}"


@pytest.mark.parametrize("n", [2, 6, 12, 24, 40])
def test_circular_reset_is_the_float64_ring(n):
    cfg = O.multi_config(64, n, circular=1, seed=1)
    env = make_env(cfg)
    orc = O.Oracle(cfg)
    obs = env.reset().cpu().numpy()
    obs_o = orc.reset()
    assert env.state.float64_world and env.state.pos64.dtype == torch.float64
    assert_state_equal_f64(env, orc.state, "after circular reset")
    assert obs_close(obs, obs_o, RTOL, ATOL).all()
    assert np.allclose(np.linalg.norm(env.state.pos64.cpu().numpy(), axis=-1), 20.0, atol=1e-12)


@pytest.mark.parametrize("name", golden_names("circular"))
def test_cuda_matches_reference_golden_circular(name):
    """Episodes started by reset(circular=True) against the LITERAL reference: it keeps float64 locations there
    (multi_uav_world_2d.py:157-163), so does the float64 world of the CUDA path — positions, velocities, prev
    distances, latches, counters and every flag bit-exact; rewards / observations within tolerance."""
    case = Case(name)
    env = make_env(case.config())
    env.enable_final_obs()
    z = case.z
    assert obs_close(env.reset().cpu().numpy(), z["obs0"], RTOL, ATOL).all()
    for t in range(case.T):
        env.step(torch.from_numpy(z["action"][t]).cuda(), evaluate=case.evaluate)
        w = f"({name}, step {t})"
        assert np.array_equal(env.done.cpu().numpy(), z["done"][t]), f"done flags differ {w}"
        assert np.array_equal(env.reset_mask.cpu().numpy(), z["reset_mask"][t]), f"reset mask differs {w}"
        h = env.state.to_host()
        assert np.array_equal(h["pos64"], z["pos64"][t]), f"float64 positions differ {w}"
        assert np.array_equal(h["vel"], z["vel"][t]), f"velocities differ {w}"
        assert np.array_equal(h["prev64"], z["prev64"][t]), f"prev_distance differs {w}"
        assert np.array_equal(h["flags"], z["flags"][t]), f"latches differ {w}"
        keep = z["reset_mask"][t] == 0
        assert np.array_equal(h["reach"][keep], z["reach"][t][keep]) and np.array_equal(h["coll"][keep], z["coll"][t][keep])
        assert close(env.reward.cpu().numpy(), z["reward"][t]).all(), f"reward {w}"
        assert obs_close(env.obs.cpu().numpy(), z["obs"][t], RTOL, ATOL).all(), f"obs {w}"
        assert obs_close(env.final_obs.cpu().numpy(), z["final_obs"][t], RTOL, ATOL).all(), f"final obs {w}"


def test_circular_rollout_vs_oracle_with_scores():
    """A batch of float64-world envs (different actions per env) against the oracle's float64 world, auto-resets on."""
    B, n = 300, 10
    cfg = O.multi_config(B, n, circular=1, reset_mode=O.RESET_ON_ALL_DONE, max_episode_steps=260, seed=2, track_scores=1)
    G = _b200()
    env = G.BatchedMultiUAVWorld2D(B, num_agents=n, circular=True, reset_mode=O.RESET_ON_ALL_DONE, max_episode_steps=260, seed=2,
                                   track_scores=True)
    orc = O.Oracle(cfg, nthreads=4)
    env.reset()
    orc.reset()
    gen = torch.Generator(device="cuda").manual_seed(3)
    gain = torch.linspace(0.3, 2.0, B, device="cuda").view(B, 1, 1)
    for t in range(400):
        a = ((env.state.tgt - env.state.pos) * gain + torch.randn((B, n, 2), generator=gen, device="cuda") * 0.5).clamp(-10, 10).contiguous()
        env.step(a, evaluate=True)
        out = orc.step(a.cpu().numpy(), evaluate=True)
        assert np.array_equal(env.done.cpu().numpy(), out["done"]) and np.array_equal(env.reset_mask.cpu().numpy(), out["reset_mask"])
        if t % 20 == 0 or t == 399:
            assert_state_equal_f64(env, orc.state, f"(step {t})")
            assert close(env.reward.cpu().numpy(), out["reward"]).all() and obs_close(env.obs.cpu().numpy(), out["obs"], RTOL, ATOL).all()
            assert np.allclose(env.score.cpu().numpy(), orc.state.score, rtol=2e-5, atol=2e-4)
    st = env.stats()
    assert st["episodes"] == int(orc.state.stats[0]) >= B and st["reach"] == int(orc.state.stats[1])
    assert st["collisions"] == int(orc.state.stats[2]) > 0
    out = env.rollout(4, None)  # the float64 world has no K loop: the same call issues K launches (tests/test_rollout_gpu.py)
    assert out["obs"].shape == (4, B, n, 10) and torch.isfinite(out["reward"]).all()


@pytest.mark.parametrize("n", [33, 40, 64, 100])
def test_more_agents_than_a_warp_holds(n):
    """`num_agents` is unbounded in the reference (multi_uav_world_2d.py:13,36-41): envs wider than a warp run on the
    general one-thread-per-env kernel, same float32 semantics, same oracle."""
    cfg = O.multi_config(130, n, reset_mode=O.RESET_ON_DONE0, max_episode_steps=30, seed=500 + n, x_size=60.0, y_size=60.0)
    ev, _ = rollout_vs_oracle(cfg, steps=70, seed=n, crowd=0.4, check_every=3)
    assert ev["resets"] > 0


# ---- sharding, action modes, host path, graphs -----------------------------------------------------------------


def test_shard_invariance():
    """Env b behaves identically whichever shard it lands in (Philox keyed by the global env index)."""
    G = _b200()
    B, N, steps = 512, 8, 60
    kw = dict(num_agents=N, seed=31, reset_mode=O.RESET_ON_DONE0, max_episode_steps=25)
    full = G.BatchedMultiUAVWorld2D(B, **kw)
    shards = [G.BatchedMultiUAVWorld2D(B // 4, env_index_base=k * (B // 4), **kw) for k in range(4)]
    full.reset()
    for s in shards:
        s.reset()
    gen = torch.Generator(device="cuda").manual_seed(5)
    for t in range(steps):
        a = torch.rand((B, N, 2), generator=gen, device="cuda") * 20 - 10
        full.step(a)
        for k, s in enumerate(shards):
            s.step(a[k * (B // 4):(k + 1) * (B // 4)].contiguous())
    for k, s in enumerate(shards):
        sl = slice(k * (B // 4), (k + 1) * (B // 4))
        assert torch.equal(s.state.pos, full.state.pos[sl]) and torch.equal(s.state.vel, full.state.vel[sl])
        assert torch.equal(s.obs, full.obs[sl]) and torch.equal(s.done, full.done[sl])
        assert torch.equal(s.state.episode, full.state.episode[sl])


@pytest.mark.parametrize("mode", ["polar", "scaled"])
def test_action_modes(mode):
    """Fused mapping == map_action kernel followed by a cartesian step (bit-exact); mapping ~= the callers' NumPy
    formula (test_sac_multi.py:77-80, test_pytorch_multi.py:80)."""
    G = _b200()
    B, N = 300, 5
    e1 = G.BatchedMultiUAVWorld2D(B, num_agents=N, seed=2)
    e2 = G.BatchedMultiUAVWorld2D(B, num_agents=N, seed=2)
    e1.reset()
    e2.reset()
    gen = torch.Generator(device="cuda").manual_seed(1)
    for _ in range(20):
        a = torch.rand((B, N, 2), generator=gen, device="cuda") * 2 - 1
        mapped = e2.map_action(a, mode)
        e1.step(a, action_mode=mode)
        e2.step(mapped)
        assert torch.equal(e1.state.pos, e2.state.pos) and torch.equal(e1.obs, e2.obs)
        an = a.cpu().numpy()
        if mode == "polar":
            v = (an[..., 0] / 2 + 0.5) * np.float32(np.linalg.norm(e1.action_space.high))
            th = an[..., 1] * np.float32(np.pi)
            ref = np.stack([v * np.cos(th.astype(np.float64)), v * np.sin(th.astype(np.float64))], -1)
        else:
            ref = an * e1.action_space.high
        orc = O.Oracle(O.multi_config(B, N))
        assert np.allclose(mapped.cpu().numpy(), ref, rtol=1e-5, atol=2e-6)
        assert np.allclose(orc.map_action(an, O.ACTION_POLAR if mode == "polar" else O.ACTION_SCALED), ref, rtol=1e-5, atol=2e-6)


@pytest.mark.parametrize("pinned", [True, False, "dma"])
@pytest.mark.parametrize("kind", ["multi", "single"])
def test_step_host_matches_device_step(kind, pinned, monkeypatch):
    """Host-buffer step: pinned buffers take the zero-copy path (the kernel reads/writes mapped host memory through
    PCIe) or, for very large outputs (forced here), the DMA pipeline; pageable buffers the staged chunked-copy
    pipeline; all must equal the device-resident step."""
    if pinned == "dma":
        monkeypatch.setenv("UAVCA_HOST_PATH", "dma")
    G = _b200()
    B = 5000
    pin = (lambda t: t.pin_memory()) if pinned else (lambda t: t)
    if kind == "multi":
        mk = lambda: G.BatchedMultiUAVWorld2D(B, num_agents=7, seed=8, reset_mode=O.RESET_ON_DONE0, max_episode_steps=30)  # noqa: E731
        N, D = 7, 10
    else:
        mk = lambda: G.BatchedUAVWorld2D(B, seed=8, reset_mode=O.RESET_ON_ANY_DONE, max_episode_steps=30)  # noqa: E731
        N, D = 1, 4
    e1, e2 = mk(), mk()
    e1.reset()
    e2.reset()
    act = pin(torch.empty((B, N, 2), dtype=torch.float32))
    obs = pin(torch.empty((B, N, D), dtype=torch.float32))
    rew = pin(torch.empty((B, N), dtype=torch.float32))
    done = pin(torch.empty((B, N), dtype=torch.uint8))
    g = torch.Generator().manual_seed(0)
    for _ in range(50):
        act.copy_(torch.rand((B, N, 2), generator=g) * 20 - 10)
        e1.step(act.cuda())
        torch.cuda.synchronize()
        e2.step_host(act, obs, rew, done)
        assert torch.equal(obs, e1.obs.cpu()) and torch.equal(rew, e1.reward.cpu()) and torch.equal(done, e1.done.cpu())
    assert torch.equal(e1.state.blob, e2.state.blob)


def test_custom_op_route_equals_the_direct_route():
    """step() calls the C-ABI directly in eager code and through torch.ops.uavca.* when asked to (or under
    torch.compile): same entry point, same results; the ops are registered with their mutation signatures."""
    G = _b200()
    for kind in ("multi", "single"):
        mk = (lambda: G.BatchedMultiUAVWorld2D(3000, num_agents=6, seed=4, reset_mode=O.RESET_ON_DONE0, max_episode_steps=25)) \
            if kind == "multi" else (lambda: G.BatchedUAVWorld2D(3000, seed=4, reset_mode=O.RESET_ON_ANY_DONE, max_episode_steps=25))
        e1, e2 = mk(), mk()
        e2.use_custom_ops = True
        e1.enable_final_obs(); e2.enable_final_obs()
        e1.reset(); e2.reset()
        gen = torch.Generator(device="cuda").manual_seed(2)
        for _ in range(40):
            a = torch.rand((3000, e1.num_agents, 2), generator=gen, device="cuda") * 20 - 10
            e1.step(a); e2.step(a)
        assert torch.equal(e1.state.blob, e2.state.blob) and torch.equal(e1.obs, e2.obs) and torch.equal(e1.final_obs, e2.final_obs)
        assert torch.equal(e1.reward, e2.reward) and torch.equal(e1.done, e2.done) and torch.equal(e1.reset_mask, e2.reset_mask)
    assert hasattr(torch.ops.uavca, "step_multi") and hasattr(torch.ops.uavca, "step_single") and hasattr(torch.ops.uavca, "policy_act")


def test_checkpoint_resume_is_bit_identical():
    G = _b200()
    mk = lambda: G.BatchedMultiUAVWorld2D(2000, num_agents=9, seed=12, reset_mode=O.RESET_ON_DONE0, max_episode_steps=15)  # noqa: E731
    env = mk()
    env.reset()
    gen = torch.Generator(device="cuda").manual_seed(3)
    acts = [torch.rand((2000, 9, 2), generator=gen, device="cuda") * 20 - 10 for _ in range(40)]
    for a in acts[:20]:
        env.step(a)
    sd = env.state_dict()
    for a in acts[20:]:
        env.step(a)
    final_blob, final_obs = env.state.blob.clone(), env.obs.clone()
    fresh = mk()  # a new handle: nothing but the checkpoint carries over (auto-resets keep drawing the same episodes)
    fresh.load_state_dict(sd)
    assert torch.equal(fresh.obs, torch.as_tensor(sd["obs"]).cuda())
    for a in acts[20:]:
        fresh.step(a)
    assert torch.equal(fresh.state.blob, final_blob) and torch.equal(fresh.obs, final_obs)
    with pytest.raises(ValueError):
        G.BatchedMultiUAVWorld2D(2000, num_agents=9, seed=13).load_state_dict(sd)


def test_step_in_cuda_graph():
    """The custom op captures into a CUDA graph (how bench.py and rollouts replay it)."""
    G = _b200()
    B, N = 4096, 8
    kw = dict(num_agents=N, seed=4, reset_mode=O.RESET_ON_DONE0, max_episode_steps=50)
    eager, graphed = G.BatchedMultiUAVWorld2D(B, **kw), G.BatchedMultiUAVWorld2D(B, **kw)
    eager.reset()
    graphed.reset()
    a = torch.zeros((B, N, 2), device="cuda")
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        graphed.step(a)  # warm-up outside capture
    torch.cuda.synchronize()
    graphed.state.blob.copy_(eager.state.blob)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        graphed.step(a)
    gen = torch.Generator(device="cuda").manual_seed(2)
    for _ in range(80):
        a.copy_(torch.rand((B, N, 2), generator=gen, device="cuda") * 20 - 10)
        g.replay()
        eager.step(a)
    torch.cuda.synchronize()
    assert torch.equal(eager.state.blob, graphed.state.blob) and torch.equal(eager.obs, graphed.obs)


def test_misaligned_tensors_are_rejected():
    G = _b200()
    from gym_uav_collision_avoidance_b200 import _capi

    env = G.BatchedMultiUAVWorld2D(64, num_agents=5)
    env.reset()
    a = torch.zeros(64 * 5 * 2 + 1, device="cuda")[1:].view(64, 5, 2)  # 4-byte aligned only
    assert a.data_ptr() % 8 == 4
    rc = env._lib.uavca_step_multi(env._h, env.state.blob.data_ptr(), a.data_ptr(), 0, 0, env.obs.data_ptr(), env.reward.data_ptr(),
                                   env.done.data_ptr(), None, None, None)
    assert rc == -1 and "misaligned" in _capi.last_error()
    env.step(a)  # ... while the class realigns such a view by copying it
    assert env.steps.min().item() == 1


def test_errors_are_loud():
    G = _b200()
    with pytest.raises(G.UavcaError):
        G.BatchedMultiUAVWorld2D(16, num_agents=1025)
    env = G.BatchedMultiUAVWorld2D(16, num_agents=4)
    with pytest.raises(ValueError):
        env.step(torch.zeros((16, 3, 2), device="cuda"))
    env2 = G.BatchedMultiUAVWorld2D(16, num_agents=4, reset_mode=1, reset_source=G.SOURCE_POOL)
    with pytest.raises(G.UavcaError):
        env2.step(torch.zeros((16, 4, 2), device="cuda"))
