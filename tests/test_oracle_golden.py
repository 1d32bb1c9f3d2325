"""CPU: oracle/uav_oracle.c replayed against the golden vectors the literal reference produced
(oracle/gen_golden.py).  Everything is compared for EXACT equality — flags, float32 positions, float64
velocities, float64 rewards and float64 observations."""
import json

import numpy as np
import pytest

from oracle import oracle as O
from oracle import ref_loader as R

from _golden import Case, golden_names


@pytest.mark.parametrize("name", golden_names())
def test_oracle_matches_reference_golden(name):
    case = Case(name)
    orc = O.Oracle(case.config())
    orc.state = case.init_state()
    orc.set_pool(case.pool_state())
    z = case.z
    assert np.array_equal(orc.observe(), z["obs0"]), "reset observation"
    for t in range(case.T):
        if "action64" in z.files:  # f64act_*: float64 actions that float32 cannot hold
            out = orc.step_f64(z["action64"][t], evaluate=case.evaluate, want_final_obs=True)
        else:
            out = orc.step(z["action"][t], evaluate=case.evaluate, want_final_obs=True)
        assert np.array_equal(out["done"], z["done"][t]), f"done flags, step {t}"
        assert np.array_equal(out["reset_mask"], z["reset_mask"][t]), f"reset mask, step {t}"
        assert np.array_equal(out["reward"], z["reward"][t]), f"reward, step {t}"
        assert np.array_equal(out["final_obs"], case.final_obs(t)), f"terminal observation, step {t}"
        assert np.array_equal(out["obs"], z["obs"][t]), f"observation, step {t}"
        assert np.array_equal(orc.state.pos, z["pos"][t]), f"position, step {t}"
        assert np.array_equal(orc.state.vel, z["vel"][t]), f"velocity, step {t}"
        assert np.array_equal(orc.state.prev, z["prev"][t]), f"prev_distance, step {t}"
        assert np.array_equal(orc.state.steps, z["steps"][t]), f"env.steps, step {t}"
        if case.kind == "multi":
            assert np.array_equal(orc.state.flags, z["flags"][t]), f"parked/collided latches, step {t}"
            assert np.array_equal(orc.state.reach, z["reach"][t]), f"target_reach_count, step {t}"
            assert np.array_equal(orc.state.coll, z["coll"][t]), f"collision_count, step {t}"
        else:
            assert np.array_equal(out["distance"], z["distance"][t]), f"info distance, step {t}"


@pytest.mark.parametrize("name", golden_names("circular"))
def test_oracle_matches_reference_golden_circular(name):
    """Episodes started by reset(circular=True): the reference keeps float64 locations (multi_uav_world_2d.py:157-163), the
    oracle's float64 world must reproduce them bit for bit — positions, velocities, rewards, observations, flags."""
    case = Case(name)
    orc = O.Oracle(case.config())
    z = case.z
    assert np.array_equal(orc.reset(), z["obs0"]), "reset(circular=True) observation"
    assert np.allclose(np.linalg.norm(orc.state.pos64, axis=-1), 20.0, atol=1e-12)
    for t in range(case.T):
        steps_before = orc.state.steps.copy()
        out = orc.step(z["action"][t], evaluate=case.evaluate, want_final_obs=True)
        assert np.array_equal(out["done"], z["done"][t]), f"done flags, step {t}"
        assert np.array_equal(out["reset_mask"], z["reset_mask"][t]), f"reset mask, step {t}"
        assert np.array_equal(out["reward"], z["reward"][t]), f"reward, step {t}"
        assert np.array_equal(out["final_obs"], z["final_obs"][t]), f"terminal observation, step {t}"
        assert np.array_equal(out["obs"], z["obs"][t]), f"observation, step {t}"
        assert np.array_equal(orc.state.pos64, z["pos64"][t]), f"position, step {t}"
        assert np.array_equal(orc.state.vel, z["vel"][t]), f"velocity, step {t}"
        assert np.array_equal(orc.state.prev64, z["prev64"][t]), f"prev_distance, step {t}"
        assert np.array_equal(orc.state.flags, z["flags"][t]), f"parked/collided latches, step {t}"
        keep = z["reset_mask"][t] == 0  # the golden counters were read before a restart zeroed them
        assert np.array_equal(orc.state.steps[keep], z["steps"][t][keep]) and np.array_equal(steps_before + 1, z["steps"][t])
        assert np.array_equal(orc.state.reach[keep], z["reach"][t][keep]) and np.array_equal(orc.state.coll[keep], z["coll"][t][keep])
        assert np.array_equal(orc.state.pos, z["pos64"][t].astype(np.float32))  # the float32 mirrors follow


def test_golden_cases_exercise_the_interesting_events():
    ev = dict(done=0, resets=0, reach=0, coll=0, parked=0)
    for name in golden_names("multi"):
        z = Case(name).z
        ev["done"] += int(z["done"].sum())
        ev["resets"] += int(z["reset_mask"].sum())
        ev["reach"] += int(z["reach"].max())
        ev["coll"] += int(z["coll"].max())
        ev["parked"] += int((z["flags"] & 1).sum())
    assert ev["done"] > 1000 and ev["resets"] > 10 and ev["reach"] > 10 and ev["coll"] > 10 and ev["parked"] > 1000


def _live_digests():
    from oracle import gen_golden as G

    with open(G.LIVE_DIGESTS) as f:
        return json.load(f)


@pytest.mark.parametrize("n", [3, 7])
def test_oracle_matches_live_reference(n):
    """A small pool-reset case on fresh seeds: where the reference is present it runs live and every step is compared
    exactly; everywhere, every step must reproduce the stored digest of the exact input and output bytes."""
    from oracle import gen_golden as G

    case = G.live_multi_case(n)
    res = G.run_reference_multi(case) if R.reference_available() else None
    want = _live_digests()["live_multi"][str(n)]
    for t, (a, out, st) in enumerate(G.oracle_live_multi(case)):
        if res is not None:
            assert np.array_equal(a, res["action"][t])
            assert np.array_equal(out["done"], res["done"][t])
            assert np.array_equal(out["reward"], res["reward"][t])
            assert np.array_equal(out["obs"], res["obs"][t])
            assert np.array_equal(out["final_obs"], res["final_obs"][t])
            assert np.array_equal(st.pos, res["pos"][t])
            assert np.array_equal(st.vel, res["vel"][t])
        assert G.live_multi_digest(a, out, st) == want[t], f"step {t} differs from the stored record"
    assert t + 1 == len(want) == case["T"]


@pytest.mark.parametrize("trial", range(6))
def test_oracle_matches_live_reference_with_random_constructor_arguments(trial):
    """Non-default worlds: box, speed / acceleration bounds, collider radius, sensing range and N drawn at random (crowded
    enough for collisions, goal reaches and parked UAVs).  Where the reference is present it is stepped live beside the
    oracle and every output and the whole state are compared for exact equality at every step; everywhere, the drawn
    world and every step must reproduce the stored digest of the exact bytes.  (HARD_COLLISION_RADIUS is a module
    constant of the reference, multi_uav_world_2d.py:8, so it stays 0.5.)"""
    from oracle import gen_golden as G

    want = _live_digests()["random_world"][str(trial)]
    gen = G.oracle_random_world(trial)
    setup = next(gen)
    n, kw, st = setup["n"], setup["kw"], setup["state"]
    assert (n, kw) == (want["n"], want["kw"]) and G.random_world_setup_digest(setup) == want["setup"]
    env = None
    if R.reference_available():
        _, MultiUAVWorld2D = R.load_reference()
        env = MultiUAVWorld2D(num_agents=n, **kw)
        env.reset()
        R.inject_multi(env, st.pos[0], st.vel[0], st.tgt[0], st.init[0], st.prev[0], st.flags[0])
        assert np.array_equal(setup["obs0"], np.stack([env._get_obs(a) for a in env.agent_list]))
    events = 0
    for t, (a, out, s) in enumerate(gen):
        if env is not None:
            o, r, d, _ = env.step([a[i].astype(np.float64) for i in range(n)], evaluate=setup["evaluate"])
            assert np.array_equal(out["done"][0], np.array(d, np.uint8)), f"done flags, step {t}"
            assert np.array_equal(out["reward"][0], np.array(r, np.float64)), f"reward, step {t}"
            assert np.array_equal(out["obs"][0], np.stack(o)), f"observation, step {t}"
            pos, vel, tgt, ini, prv, flg = R.extract_multi(env)
            assert np.array_equal(s.pos[0], pos) and np.array_equal(s.vel[0], vel), f"state, step {t}"
            assert np.array_equal(s.prev[0], prv) and np.array_equal(s.flags[0], flg), f"latches, step {t}"
            assert int(s.coll[0]) == env.collision_count and int(s.reach[0]) == env.target_reach_count
        assert G.random_world_digest(a, out, s) == want["steps"][t], f"step {t} differs from the stored record"
        events += int(out["done"].sum()) + int(s.flags.sum())
    assert t + 1 == len(want["steps"]) and events > 0
