"""Prioritized replay on one GPU: sum-tree sync, priority update and prioritized sampling against the PyTorch ways of
drawing from a priority vector, what the sync adds to the configs[4] acting step, and the n-step samplers against the
one-step draws and against the same n-step rule written with torch indexing.  CUDA events; ring of 1,048,576 slots
(2^20 leaves).
    python tools/per_bench.py [--reps N]"""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

import gym_uav_collision_avoidance_b200 as G  # noqa: E402
from gym_uav_collision_avoidance_b200 import ops  # noqa: E402

CAP = 1 << 20
B4, N4 = 16384, 10  # BASELINE configs[4]


def card():
    name = torch.cuda.get_device_name()
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i",
                            str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30)
        power = q.stdout.strip() or "unknown"
    except (OSError, subprocess.SubprocessError):
        power = "unknown"
    return name, power


def graph_us(fn, n=20, reps=5):
    """us per call of fn, replayed from a CUDA graph of n calls (device time without host launch overhead)."""
    st = torch.cuda.Stream()
    st.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(st):
        for _ in range(3):
            fn()
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=st):
        for _ in range(n):
            fn()
    g.replay()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with torch.cuda.stream(st):
        e0.record(st)
        for _ in range(reps):
            g.replay()
        e1.record(st)
    st.synchronize()
    return e0.elapsed_time(e1) * 1e3 / (reps * n)


def torch_nstep(rb, idx, n, gamma, stride):
    """The n-step rule of include/uavca.h (uavca_replay_sample_nstep) for slots `idx`, written with torch indexing: what a
    learner would run without the fused sampler.  No host synchronisation, so it can be captured too."""
    cap = rb.capacity
    age = torch.remainder(rb.meta[0] - 1 - idx, cap)
    ob, nb = rb.state.view(torch.int32), rb.next_state.view(torch.int32)
    k = torch.ones_like(idx)
    alive = torch.ones_like(idx, dtype=torch.bool)
    prev = idx
    for i in range(1, n):
        si = torch.remainder(idx + i * stride, cap)
        alive = alive & (rb.mask[prev] != 0) & (age >= i * stride) & (ob[si] == nb[prev]).all(1)
        k = k + alive
        prev = si
    R = torch.zeros(idx.shape, dtype=torch.float64, device=idx.device)
    g = torch.ones_like(R)
    for i in range(n):
        on = k > i
        R = torch.where(on, R + g * rb.reward[torch.remainder(idx + i * stride, cap)].double(), R)
        g = torch.where(on, g * gamma, g)
    last = torch.remainder(idx + (k - 1) * stride, cap)
    disc = torch.where(rb.mask[last] != 0, g.float(), torch.zeros_like(rb.mask[last]))
    return rb.state[idx], rb.action[idx], R.float(), rb.next_state[last], disc


def nstep_rows(res):
    """The n-step samplers on a 2^20-slot prioritized ring filled by configs[4] acting steps (fused append + sync)."""
    env = G.BatchedMultiUAVWorld2D(B4, num_agents=N4, reset_mode=G.RESET_ON_DONE0, max_episode_steps=100, seed=3)
    rb = G.PrioritizedDeviceReplay(CAP, 10, 2, seed=0)
    ro = G.BatchedRollout(env, None, rb, action_mode="polar", warmup_uniform=True)
    ro.reset()
    ro.run(8)  # 8 x 163,840 transitions: the ring is full and has wrapped
    stride, gamma = B4 * N4, 0.99
    for b in (256, 4096):
        uni = rb.sample_fused(b, want_index=True)
        res[f"nstep_sample_fused_{b}_us"] = graph_us(lambda: rb.sample_fused(b, out=uni))
        per = rb.sample_prioritized(b, 0.4)
        res[f"nstep_sample_prioritized_{b}_us"] = graph_us(lambda: rb.sample_prioritized(b, 0.4, out=per))
        for n in (1, 3, 5):
            un = rb.sample_nstep(b, n, gamma, stride, want_index=True)
            res[f"sample_nstep_n{n}_{b}_us"] = graph_us(lambda: rb.sample_nstep(b, n, gamma, stride, out=un))
            pn = rb.sample_prioritized_nstep(b, 0.4, n, gamma, stride)
            res[f"sample_prioritized_nstep_n{n}_{b}_us"] = graph_us(
                lambda: rb.sample_prioritized_nstep(b, 0.4, n, gamma, stride, out=pn))

            def torch_rule():
                rb.sample_fused(b, out=uni)
                return torch_nstep(rb, uni[5], n, gamma, stride)

            res[f"torch_nstep_n{n}_{b}_us"] = graph_us(torch_rule)
    # the fused sampler and the torch rule agree on the same slots
    d0 = rb._draws
    got = rb.sample_nstep(4096, 3, gamma, stride, want_index=True)
    rb._draws = d0
    ref = torch_nstep(rb, rb.sample_fused(4096, want_index=True)[5], 3, gamma, stride)
    res["nstep_torch_rule_agrees"] = all(torch.equal(x, y) for x, y in zip(got[:5], ref))
    del env, rb, ro


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=50)
    args = ap.parse_args()
    name, power = card()
    res = {"card": name, "power_limit": power, "capacity": CAP}
    rb = G.PrioritizedDeviceReplay(CAP, 10, 2, seed=0)
    M = B4 * N4
    x = torch.rand((M, 10), device="cuda")
    a = torch.rand((M, 2), device="cuda")
    r = torch.rand(M, device="cuda")
    d = torch.zeros(M, dtype=torch.uint8, device="cuda")
    for _ in range(8):  # fill the ring
        rb.push(x, a, r, x, d)
    # sync after one configs[4] append: events around the sync alone, an append before each
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    total = 0.0
    for i in range(args.reps + 3):
        G.DeviceReplay.push(rb, x, a, r, x, d)
        e0.record()
        rb.sync()
        e1.record()
        e1.synchronize()
        if i >= 3:
            total += e0.elapsed_time(e1) * 1e3
    res["sync_c4_append_us"] = total / args.reps
    res["idle_sync_us"] = graph_us(rb.sync)
    gen = torch.Generator(device="cuda").manual_seed(0)
    for n in (256, 4096):
        idx = torch.randint(0, CAP, (n,), generator=gen, device="cuda")
        td = torch.randn(n, generator=gen, device="cuda")
        p = (td.double().abs() + rb.eps).pow(rb.alpha)
        res[f"update_kernel_{n}_us"] = graph_us(lambda: ops.per_update(rb.tree, rb.per_meta, idx, p, CAP))
        res[f"update_priorities_{n}_us"] = graph_us(lambda: rb.update_priorities(idx, td))
        out = rb.sample_prioritized(n, 0.4)
        res[f"sample_prioritized_{n}_us"] = graph_us(lambda: rb.sample_prioritized(n, 0.4, out=out))
        prio = rb.tree[rb.leaves:rb.leaves + CAP].clone()
        res[f"torch_multinomial_{n}_us"] = graph_us(lambda: torch.multinomial(prio, n, replacement=True))
        u = torch.rand(n, dtype=torch.float64, device="cuda")

        def cumsum_search():
            cs = torch.cumsum(prio, 0)
            return torch.searchsorted(cs, u * cs[-1], right=True)

        res[f"torch_cumsum_searchsorted_{n}_us"] = graph_us(cumsum_search)
        uni = rb.sample_fused(n, want_index=True)
        res[f"uniform_sample_fused_{n}_us"] = graph_us(lambda: rb.sample_fused(n, out=uni))
    # the configs[4] acting step (fused policy, fused append) on a uniform and on a prioritized ring
    torch.manual_seed(0)
    pol = G.GaussianPolicy(10, 2).cuda()
    for kind, cls in (("uniform", G.DeviceReplay), ("prioritized", G.PrioritizedDeviceReplay)):
        env = G.BatchedMultiUAVWorld2D(B4, num_agents=N4, reset_mode=G.RESET_ON_DONE0, max_episode_steps=100, seed=1)
        ring = cls(CAP, 10, 2, seed=0)
        ro = G.BatchedRollout(env, pol, ring, precision="fused")
        ro.reset()
        res[f"acting_step_{kind}_us"] = graph_us(lambda: ro.run(2), n=10) / 2
        del env, ring, ro
    res["acting_step_sync_overhead_us"] = res["acting_step_prioritized_us"] - res["acting_step_uniform_us"]
    nstep_rows(res)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
