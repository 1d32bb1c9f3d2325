"""Generate tests/golden/*.npz by executing the UNMODIFIED reference.  TEST INFRASTRUCTURE ONLY.

Run in the build container (where /root/reference exists):

    python -m oracle.gen_golden            # rewrites tests/golden/*.npz
    python -m oracle.gen_golden live       # rewrites tests/golden/live_reference_digests.json (oracle only)

Every file holds seeded initial states, the float32 actions that were fed (to the reference as float64
up-casts, SURVEY.md §8c), and what the literal reference returned at every step: float64 observations and
rewards, done flags, and the float32 positions / float64 velocities / flags / counters after the step.
tests/test_oracle_golden.py replays the same inputs through oracle/uav_oracle.c and demands exact equality;
the GPU parity tests replay them through the CUDA path.

Scenarios mix wide-box random actions (out-of-bounds events) with a noisy go-to-goal controller in a crowded
region (soft/hard collisions, goal reaches, parked UAVs being hit), both env kinds, evaluate=True, and the
"reset when dones[0]" training protocol with host-supplied reset states (pool).
"""
from __future__ import annotations

import json
import math
import os

import numpy as np

from . import oracle as O
from . import ref_loader as R

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "tests", "golden")

MULTI_CASES = [
    # name, N, envs, steps, seed, evaluate, reset_mode, max_episode_steps
    dict(name="multi_n1", N=1, E=6, T=200, seed=101, evaluate=0, reset_mode=0, max_steps=0),
    dict(name="multi_n2", N=2, E=6, T=250, seed=102, evaluate=0, reset_mode=0, max_steps=0),
    dict(name="multi_n5_reset_done0", N=5, E=8, T=400, seed=105, evaluate=0, reset_mode=O.RESET_ON_DONE0, max_steps=150),
    dict(name="multi_n8", N=8, E=8, T=400, seed=108, evaluate=0, reset_mode=0, max_steps=0),
    dict(name="multi_n10_eval_reset_all", N=10, E=4, T=300, seed=110, evaluate=1, reset_mode=O.RESET_ON_ALL_DONE, max_steps=0),
    dict(name="multi_n32", N=32, E=2, T=120, seed=132, evaluate=0, reset_mode=0, max_steps=0),
    # more UAVs than a warp holds: the general one-thread-per-env kernel (num_agents is unbounded in the reference)
    dict(name="multi_n40_reset_done0", N=40, E=2, T=90, seed=140, evaluate=0, reset_mode=O.RESET_ON_DONE0, max_steps=60),
]
# float64 actions that float32 cannot hold — what the reference's SAC loop builds on the host (test_sac_multi.py:77-80: a
# uniform policy output mapped to polar coordinates in float64) and a float64 go-to-goal controller in the crowded envs
F64ACT_CASES = [
    dict(name="f64act_multi_n5", N=5, E=6, T=300, seed=405, evaluate=0, reset_mode=O.RESET_ON_DONE0, max_steps=120, f64act=1),
    dict(name="f64act_multi_n12_eval", N=12, E=4, T=250, seed=412, evaluate=1, reset_mode=O.RESET_ON_ALL_DONE, max_steps=0, f64act=1),
]
F64ACT_SINGLE_CASES = [
    dict(name="f64act_single", E=8, T=300, seed=451, f32=0, f64act=1),
]
SINGLE_CASES = [
    dict(name="single_f64_actions", E=12, T=400, seed=201, f32=0),
    dict(name="single_f32_actions", E=12, T=400, seed=202, f32=1),
]
CIRCULAR_CASES = [
    # reset(circular=True): float64 locations on a ring, targets across it — everybody meets in the middle
    dict(name="circular_n6", N=6, E=3, T=600, seed=306, evaluate=0, max_steps=0),
    dict(name="circular_n12_eval", N=12, E=2, T=700, seed=312, evaluate=1, max_steps=0),
    dict(name="circular_n5_limit", N=5, E=3, T=500, seed=305, evaluate=0, max_steps=170),
]
POOL = 16


def _actions_multi(rng, st: O.State, b: int, N: int, controller: bool):
    if controller:
        a = (st.tgt[b] - st.pos[b]) * 1.5 + rng.normal(0, 0.3, size=(N, 2))
        return np.clip(a, -10, 10).astype(np.float32)
    return rng.uniform(-10, 10, size=(N, 2)).astype(np.float32)


def _actions_multi_f64(rng, st: O.State, b: int, N: int, controller: bool):
    if controller:
        return np.clip((st.tgt[b].astype(np.float64) - st.pos[b]) * 1.5 + rng.normal(0, 0.3, size=(N, 2)), -10, 10)
    u = rng.uniform(-1, 1, size=(N, 2))  # the policy-space action of test_sac_multi.py:72-80
    v = (u[:, 0] / 2 + 0.5) * np.linalg.norm(np.full(2, 10.0, np.float32))
    th = u[:, 1] * math.pi
    return np.stack([v * np.cos(th), v * np.sin(th)], axis=1).astype(np.float64)


def _init_and_pool(case, rng):
    """Seeded initial states and reset pool of a multi case: odd envs in a crowded region, even envs in the full box."""
    N, E = case["N"], case["E"]
    regions = [None if b % 2 == 0 else max(3.0, 0.75 * N ** 0.5 * 2.0) for b in range(E)]
    init = O.State(E, N)
    for b in range(E):
        s = O.sample_multi_states(1, N, rng, region=regions[b])
        for f in ("pos", "vel", "tgt", "init", "prev", "flags"):
            getattr(init, f)[b] = getattr(s, f)[0]
    pool = O.State(POOL, N)
    for p in range(POOL):
        s = O.sample_multi_states(1, N, rng, region=regions[p % E])
        for f in ("pos", "vel", "tgt", "init", "prev", "flags"):
            getattr(pool, f)[p] = getattr(s, f)[0]
    return init, pool


def run_reference_multi(case) -> dict:
    _, MultiUAVWorld2D = R.load_reference()
    N, E, T = case["N"], case["E"], case["T"]
    rng = np.random.default_rng(case["seed"])
    # odd envs: crowded region + controller; even envs: full box + random actions
    init, pool = _init_and_pool(case, rng)

    envs = [MultiUAVWorld2D(num_agents=N) for _ in range(E)]
    cur = init.copy()
    for b, env in enumerate(envs):
        env.reset()
        R.inject_multi(env, cur.pos[b], cur.vel[b], cur.tgt[b], cur.init[b], cur.prev[b], cur.flags[b])
    episode = np.ones(E, np.int64)  # episode counter after the initial "reset" (matches the oracle/device: 1)
    out = dict(
        action=np.zeros((T, E, N, 2), np.float32), obs=np.zeros((T, E, N, 10)), final_obs=np.zeros((T, E, N, 10)),
        reward=np.zeros((T, E, N)), done=np.zeros((T, E, N), np.uint8), reset_mask=np.zeros((T, E), np.uint8),
        pos=np.zeros((T, E, N, 2), np.float32), vel=np.zeros((T, E, N, 2)), flags=np.zeros((T, E, N), np.uint8),
        prev=np.zeros((T, E, N), np.float32), steps=np.zeros((T, E), np.int32), reach=np.zeros((T, E), np.int32),
        coll=np.zeros((T, E), np.int32),
    )
    obs0 = np.stack([np.stack([env._get_obs(a) for a in env.agent_list]) for env in envs])
    for t in range(T):
        for b, env in enumerate(envs):
            if case.get("f64act"):
                a = _actions_multi_f64(rng, cur, b, N, controller=(b % 2 == 1))
                out.setdefault("action64", np.zeros((T, E, N, 2), np.float64))[t, b] = a
            else:
                a = _actions_multi(rng, cur, b, N, controller=(b % 2 == 1))
            out["action"][t, b] = a
            o, r, d, _ = env.step([a[i].astype(np.float64) for i in range(N)], evaluate=bool(case["evaluate"]))
            o = np.stack(o)
            out["final_obs"][t, b] = o
            out["reward"][t, b] = np.array(r, dtype=np.float64)
            out["done"][t, b] = np.array(d, dtype=np.uint8)
            rs = False
            if case["reset_mode"] & O.RESET_ON_DONE0:
                rs |= bool(d[0])
            if case["reset_mode"] & O.RESET_ON_ALL_DONE:
                rs |= all(d)
            if case["max_steps"] > 0:
                rs |= env.steps >= case["max_steps"]
            if rs:
                p = (b + int(episode[b])) % POOL
                env.reset()  # zeroes the counters exactly as the reference does (:166-168)
                R.inject_multi(env, pool.pos[p], pool.vel[p], pool.tgt[p], pool.init[p], pool.prev[p], pool.flags[p])
                episode[b] += 1
                o = np.stack([env._get_obs(ag) for ag in env.agent_list])
            out["reset_mask"][t, b] = rs
            out["obs"][t, b] = o
            pos, vel, tgt, ini, prv, flg = R.extract_multi(env)
            cur.pos[b], cur.vel[b], cur.tgt[b], cur.init[b], cur.prev[b], cur.flags[b] = pos, vel, tgt, ini, prv, flg
            out["pos"][t, b], out["vel"][t, b], out["flags"][t, b], out["prev"][t, b] = pos, vel, flg, prv
            out["steps"][t, b], out["reach"][t, b], out["coll"][t, b] = env.steps, env.target_reach_count, env.collision_count
    meta = dict(kind="multi", **case, pool=POOL)
    res = dict(meta=np.array(json.dumps(meta)), obs0=obs0)
    for f in ("pos", "vel", "tgt", "init", "prev", "flags"):
        res["init_" + f] = getattr(init, f)
        res["pool_" + f] = getattr(pool, f)
    res.update(out)
    return res


def run_reference_circular(case) -> dict:
    """Episodes started by reset(circular=True) (multi_uav_world_2d.py:157-163): the locations are float64 arrays from
    then on.  Env e flies a go-to-goal controller of gain 0.5 + 0.4 e with noise; the episode restarts (circular again)
    when dones[0] (training protocol), when all(dones) under evaluate, or at the step limit."""
    _, MultiUAVWorld2D = R.load_reference()
    N, E, T = case["N"], case["E"], case["T"]
    rng = np.random.default_rng(case["seed"])
    envs = [MultiUAVWorld2D(num_agents=N) for _ in range(E)]
    obs0 = np.stack([np.stack(env.reset(circular=True)) for env in envs])
    out = dict(
        action=np.zeros((T, E, N, 2), np.float32), obs=np.zeros((T, E, N, 10)), final_obs=np.zeros((T, E, N, 10)),
        reward=np.zeros((T, E, N)), done=np.zeros((T, E, N), np.uint8), reset_mask=np.zeros((T, E), np.uint8),
        pos64=np.zeros((T, E, N, 2)), vel=np.zeros((T, E, N, 2)), flags=np.zeros((T, E, N), np.uint8),
        prev64=np.zeros((T, E, N)), steps=np.zeros((T, E), np.int32), reach=np.zeros((T, E), np.int32),
        coll=np.zeros((T, E), np.int32),
    )
    for t in range(T):
        for b, env in enumerate(envs):
            loc = np.stack([a.location for a in env.agent_list])
            tgt = np.stack([a.target_location for a in env.agent_list])
            a = np.clip((tgt - loc) * (0.5 + 0.4 * b) + rng.normal(0, 0.6, size=(N, 2)), -10, 10).astype(np.float32)
            out["action"][t, b] = a
            o, r, d, _ = env.step([a[i].astype(np.float64) for i in range(N)], evaluate=bool(case["evaluate"]))
            o = np.stack(o)
            out["final_obs"][t, b] = o
            out["reward"][t, b] = np.array(r, dtype=np.float64)
            out["done"][t, b] = np.array(d, dtype=np.uint8)
            rs = all(d) if case["evaluate"] else bool(d[0])
            if case["max_steps"] > 0:
                rs |= env.steps >= case["max_steps"]
            # the counters are read before the restart zeroes them, like the scripts do (test_sac_multi.py:164-166)
            out["steps"][t, b], out["reach"][t, b], out["coll"][t, b] = env.steps, env.target_reach_count, env.collision_count
            if rs:
                o = np.stack(env.reset(circular=True))
            out["reset_mask"][t, b] = rs
            out["obs"][t, b] = o
            assert all(ag.location.dtype == np.float64 for ag in env.agent_list)
            out["pos64"][t, b] = np.stack([ag.location for ag in env.agent_list])
            out["vel"][t, b] = np.stack([ag.velocity for ag in env.agent_list])
            out["prev64"][t, b] = np.array([ag.prev_distance for ag in env.agent_list], dtype=np.float64)
            out["flags"][t, b] = np.array([(1 if ag.done else 0) | (2 if ag.collided else 0) for ag in env.agent_list], np.uint8)
    meta = dict(kind="circular", **case, reset_mode=(O.RESET_ON_ALL_DONE if case["evaluate"] else O.RESET_ON_DONE0))
    res = dict(meta=np.array(json.dumps(meta)), obs0=obs0)
    res.update(out)
    return res


def run_reference_single(case) -> dict:
    UAVWorld2D, _ = R.load_reference()
    E, T = case["E"], case["T"]
    rng = np.random.default_rng(case["seed"])
    init = O.sample_single_states(E, rng)
    pool = O.sample_single_states(POOL, rng)
    envs = [UAVWorld2D() for _ in range(E)]
    cur = init.copy()
    for b, env in enumerate(envs):
        env.reset()
        R.inject_single(env, cur.pos[b, 0], cur.vel[b, 0], cur.tgt[b, 0], cur.init[b, 0], cur.prev[b, 0], vel_f32=True)
    episode = np.ones(E, np.int64)
    out = dict(
        action=np.zeros((T, E, 1, 2), np.float32), obs=np.zeros((T, E, 1, 4)), final_obs=np.zeros((T, E, 1, 4)),
        reward=np.zeros((T, E, 1)), done=np.zeros((T, E, 1), np.uint8), reset_mask=np.zeros((T, E), np.uint8),
        pos=np.zeros((T, E, 1, 2), np.float32), vel=np.zeros((T, E, 1, 2)), prev=np.zeros((T, E, 1), np.float32),
        steps=np.zeros((T, E), np.int32), distance=np.zeros((T, E), np.float32),
    )
    obs0 = np.stack([env._get_obs() for env in envs])[:, None, :]
    for t in range(T):
        for b, env in enumerate(envs):
            if b % 2 == 1:
                a = np.clip((cur.tgt[b, 0] - cur.pos[b, 0]) * 0.8 + rng.normal(0, 0.5, 2), -12, 12).astype(np.float32)
            else:
                a = rng.uniform(-12, 12, 2).astype(np.float32)
            if case.get("f64act"):  # the same controller / random actions, not rounded to float32
                a = (np.clip((cur.tgt[b, 0].astype(np.float64) - cur.pos[b, 0]) * 0.8 + rng.normal(0, 0.5, 2), -12, 12)
                     if b % 2 == 1 else rng.uniform(-12, 12, 2))
                out.setdefault("action64", np.zeros((T, E, 1, 2), np.float64))[t, b, 0] = a
            out["action"][t, b, 0] = a
            o, r, d, info = env.step(a if case["f32"] else a.astype(np.float64))
            out["final_obs"][t, b, 0] = o
            out["reward"][t, b, 0] = np.float64(r)
            out["done"][t, b, 0] = d
            out["distance"][t, b] = info["distance"]
            if d:
                p = (b + int(episode[b])) % POOL
                env.reset()
                R.inject_single(env, pool.pos[p, 0], pool.vel[p, 0], pool.tgt[p, 0], pool.init[p, 0], pool.prev[p, 0],
                                vel_f32=True)
                episode[b] += 1
                o = env._get_obs()
            out["reset_mask"][t, b] = d
            out["obs"][t, b, 0] = o
            pos, vel, tgt, ini, prv = R.extract_single(env)
            cur.pos[b, 0], cur.vel[b, 0], cur.tgt[b, 0], cur.init[b, 0], cur.prev[b, 0] = pos, vel, tgt, ini, prv
            out["pos"][t, b, 0], out["vel"][t, b, 0], out["prev"][t, b, 0] = pos, vel, prv
            out["steps"][t, b] = env.steps
    meta = dict(kind="single", **case, pool=POOL, reset_mode=O.RESET_ON_ANY_DONE)
    res = dict(meta=np.array(json.dumps(meta)), obs0=obs0)
    for f in ("pos", "vel", "tgt", "init", "prev", "flags"):
        res["init_" + f] = getattr(init, f)
        res["pool_" + f] = getattr(pool, f)
    res.update(out)
    return res


# ---- the live checks of tests/test_oracle_golden.py, kept runnable without the reference ---------------------------
# Their inputs come from seeded NumPy generators and from the state of the world being stepped, never from the reference
# itself, so the oracle regenerates them exactly.  LIVE_DIGESTS stores, per step, a digest of the exact bytes of those
# inputs and of everything the checks compare; where the reference is present the tests still compare it live as well.
LIVE_DIGESTS = os.path.join(GOLDEN_DIR, "live_reference_digests.json")
LIVE_MULTI_N = (3, 7)
RANDOM_WORLD_TRIALS = 6


def digest(*arrays) -> str:
    """First 128 bits of SHA-256 over the exact bytes of `arrays` (None skipped)."""
    import hashlib

    h = hashlib.sha256()
    for a in arrays:
        if a is not None:
            h.update(np.ascontiguousarray(a).tobytes())
    return h.hexdigest()[:32]


def live_multi_case(n: int) -> dict:
    return dict(name="live", N=n, E=4, T=120, seed=900 + n, evaluate=0, reset_mode=O.RESET_ON_DONE0, max_steps=60)


def oracle_live_multi(case):
    """The oracle's side of run_reference_multi(case): the same initial states, pool and action draws (made from the
    oracle's state, which is the reference's as long as the two agree).  Yields (action, step outputs, state) per step."""
    N, E = case["N"], case["E"]
    rng = np.random.default_rng(case["seed"])
    init, pool = _init_and_pool(case, rng)
    orc = O.Oracle(O.multi_config(E, N, reset_mode=case["reset_mode"], max_episode_steps=case["max_steps"],
                                  reset_source=O.SOURCE_POOL))
    for f in ("pos", "vel", "tgt", "init", "prev", "flags"):
        getattr(orc.state, f)[...] = getattr(init, f)
    orc.state.episode[...] = 1
    orc.set_pool(pool)
    for _ in range(case["T"]):
        a = np.stack([_actions_multi(rng, orc.state, b, N, controller=(b % 2 == 1)) for b in range(E)])
        yield a, orc.step(a, evaluate=bool(case["evaluate"]), want_final_obs=True), orc.state


def live_multi_digest(a, out, st) -> str:
    return digest(a, out["done"], out["reset_mask"], out["reward"], out["obs"], out["final_obs"], st.pos, st.vel)


def oracle_random_world(trial: int):
    """A non-default world drawn at random (box, speed / acceleration bounds, collider radius, sensing range, N), crowded
    enough for collisions, goal reaches and parked UAVs, stepped 250 times by the oracle.  Yields first the setup
    dict(n, kw, state, obs0, evaluate, f64), then (action, step outputs, state) per step; half of the trials feed float64
    actions that float32 cannot hold."""
    rng = np.random.default_rng(4100 + trial)
    n = int(rng.choice([2, 3, 6, 9, 12, 17]))
    kw = dict(x_size=float(rng.uniform(10, 40)), y_size=float(rng.uniform(10, 40)), max_speed=float(rng.uniform(3, 20)),
              max_acceleration=float(rng.uniform(1, 12)), collider_radius=float(rng.uniform(0.3, 1.5)),
              d_sense=float(rng.choice([rng.uniform(1.0, 4.0), rng.uniform(6, 40)])))
    st = O.sample_multi_states(1, n, rng, x_size=kw["x_size"], y_size=kw["y_size"], collider_radius=kw["collider_radius"],
                               region=min(kw["x_size"], kw["y_size"]) / 3)
    orc = O.Oracle(O.multi_config(1, n, **kw))
    orc.state = st.copy()
    evaluate, f64 = bool(trial % 2), trial >= 3
    yield dict(n=n, kw=kw, state=st, obs0=orc.observe()[0], evaluate=evaluate, f64=f64)
    for t in range(250):
        if t % 3:
            a = np.clip((orc.state.tgt[0] - orc.state.pos[0]) * 1.2 + rng.normal(0, 0.4, (n, 2)), -kw["max_speed"], kw["max_speed"])
        else:
            a = rng.uniform(-kw["max_speed"], kw["max_speed"], (n, 2))
        a = a.astype(np.float64) if f64 else a.astype(np.float32)
        out = orc.step_f64(a[None], evaluate=evaluate) if f64 else orc.step(a[None], evaluate=evaluate)
        yield a, out, orc.state


def random_world_setup_digest(setup) -> str:
    st = setup["state"]
    return digest(np.array(json.dumps(setup["kw"], sort_keys=True)), st.pos, st.vel, st.tgt, st.init, st.prev, st.flags, setup["obs0"])


def random_world_digest(a, out, st) -> str:
    return digest(a, out["done"], out["reward"], out["obs"], st.pos, st.vel, st.prev, st.flags, st.coll, st.reach)


def record_live_digests() -> str:
    """Write LIVE_DIGESTS from the oracle (`python -m oracle.gen_golden live`)."""
    rec = {"about": "Per-step digests (first 128 bits of SHA-256 over the exact bytes) of oracle/uav_oracle.c on the inputs of "
                     "the live checks in tests/test_oracle_golden.py, recorded by `python -m oracle.gen_golden live`.  Those "
                     "checks demand exact equality with the reference at every step; where the reference is present they "
                     "still run it live beside these digests.",
           "live_multi": {}, "random_world": {}}
    for n in LIVE_MULTI_N:
        rec["live_multi"][str(n)] = [live_multi_digest(*s) for s in oracle_live_multi(live_multi_case(n))]
    for trial in range(RANDOM_WORLD_TRIALS):
        gen = oracle_random_world(trial)
        setup = next(gen)
        rec["random_world"][str(trial)] = {"n": setup["n"], "kw": setup["kw"], "setup": random_world_setup_digest(setup),
                                           "steps": [random_world_digest(*s) for s in gen]}
    with open(LIVE_DIGESTS, "w") as f:
        json.dump(rec, f, indent=0)
        f.write("\n")
    return LIVE_DIGESTS


def main():
    import sys

    os.makedirs(GOLDEN_DIR, exist_ok=True)
    only = sys.argv[1] if len(sys.argv) > 1 else None  # "circular" or a case name: regenerate just those cases
    if only == "live":
        print(record_live_digests())
        return
    if only and only not in ("circular", "f64act"):
        for case in MULTI_CASES:
            if case["name"] == only:
                res = run_reference_multi(case)
                path = os.path.join(GOLDEN_DIR, case["name"] + ".npz")
                if res["reset_mask"].sum() == 0:
                    del res["final_obs"]
                np.savez_compressed(path, **res)
                print(f"{case['name']}: done-events={int(res['done'].sum())} resets={int(res['reset_mask'].sum())} "
                      f"reach={int(res['reach'].max())} coll={int(res['coll'].max())} -> {os.path.getsize(path) / 1e6:.2f} MB")
        return
    if only == "f64act":
        for case in F64ACT_CASES:
            res = run_reference_multi(case)
            path = os.path.join(GOLDEN_DIR, case["name"] + ".npz")
            np.savez_compressed(path, **res)
            lost = int((res["action64"] != res["action"]).sum())
            print(f"{case['name']}: done-events={int(res['done'].sum())} resets={int(res['reset_mask'].sum())} "
                  f"reach={int(res['reach'].max())} coll={int(res['coll'].max())} actions float32 cannot hold={lost} "
                  f"-> {os.path.getsize(path) / 1e6:.2f} MB")
        for case in F64ACT_SINGLE_CASES:
            res = run_reference_single(case)
            path = os.path.join(GOLDEN_DIR, case["name"] + ".npz")
            np.savez_compressed(path, **res)
            print(f"{case['name']}: resets={int(res['reset_mask'].sum())} -> {os.path.getsize(path) / 1e6:.2f} MB")
        return
    if only == "circular":
        for case in CIRCULAR_CASES:
            res = run_reference_circular(case)
            path = os.path.join(GOLDEN_DIR, case["name"] + ".npz")
            np.savez_compressed(path, **res)
            print(f"{case['name']}: done-events={int(res['done'].sum())} resets={int(res['reset_mask'].sum())} "
                  f"reach={int(res['reach'].max())} coll={int(res['coll'].max())} parked-steps={int((res['flags'] & 1).sum())} "
                  f"-> {os.path.getsize(path) / 1e6:.2f} MB")
        return
    for case in MULTI_CASES:
        res = run_reference_multi(case)
        path = os.path.join(GOLDEN_DIR, case["name"] + ".npz")
        if res["reset_mask"].sum() == 0:
            del res["final_obs"]  # identical to obs when nothing reset
        np.savez_compressed(path, **res)
        print(f"{case['name']}: done-events={int(res['done'].sum())} resets={int(res['reset_mask'].sum())} "
              f"reach={int(res['reach'].max())} coll={int(res['coll'].max())} -> {os.path.getsize(path) / 1e6:.2f} MB")
    for case in CIRCULAR_CASES:
        res = run_reference_circular(case)
        path = os.path.join(GOLDEN_DIR, case["name"] + ".npz")
        np.savez_compressed(path, **res)
        print(f"{case['name']}: done-events={int(res['done'].sum())} resets={int(res['reset_mask'].sum())} "
              f"reach={int(res['reach'].max())} coll={int(res['coll'].max())} parked-steps={int((res['flags'] & 1).sum())} "
              f"-> {os.path.getsize(path) / 1e6:.2f} MB")
    for case in SINGLE_CASES + F64ACT_SINGLE_CASES:
        res = run_reference_single(case)
        path = os.path.join(GOLDEN_DIR, case["name"] + ".npz")
        np.savez_compressed(path, **res)
        print(f"{case['name']}: resets={int(res['reset_mask'].sum())} -> {os.path.getsize(path) / 1e6:.2f} MB")
    for case in F64ACT_CASES:
        res = run_reference_multi(case)
        np.savez_compressed(os.path.join(GOLDEN_DIR, case["name"] + ".npz"), **res)


if __name__ == "__main__":
    main()
