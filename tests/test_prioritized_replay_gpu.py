"""Prioritized replay (csrc/uavca_per.cu: `per_sync_kernel`, `per_update_kernel`, `per_sample_kernel`) against a numpy
restatement kept in this file:

* the sum-tree in float64 with the same pairwise additions (node k = tree[2k] + tree[2k+1]), so the whole device tree is
  compared bit for bit after every call;
* the sync rule (new slots from the ring's head, or every filled slot when more than one append went unsynced), the
  update rule (last occurrence wins, a bad entry drops the whole update);
* the stratified draws: Philox4x32-10 on stream tag 6, the same u53 uniform, the same float64 descent, so the slots are
  restated exactly; the weights within a bound derived below from the error of the device's `pow`.

Tests without the `gpu` marker need no device."""
import math

import numpy as np
import pytest
import torch

from test_acting_kernels_gpu import (TAG_ACT, TAG_POLICY, TAG_POS, TAG_SAMPLE, TAG_TGT, TAG_VEL, action_counter,
                                     indexed_counter, philox4x32_10, reset_counter)

gpu = pytest.mark.gpu

TAG_PER = 6
C4_M = 16384 * 10  # transitions of one configs[4] acting step (B = 16,384 envs x N = 10 UAVs)


# ---- restatement ------------------------------------------------------------------------------------------------------


def leaves_for(capacity):
    return 1 << (capacity - 1).bit_length()


def build_tree(leaves):
    """float64 [2L] sum-tree of `leaves` (L a power of two): node k = tree[2k] + tree[2k+1], one IEEE addition each."""
    L = leaves.size
    tree = np.zeros(2 * L, np.float64)
    tree[L:] = leaves
    k = L
    while k > 1:
        tree[k // 2:k] = tree[k:2 * k:2] + tree[k + 1:2 * k:2]
        k //= 2
    return tree


def u53(a, b):
    """The kernel's 53-bit uniform of two Philox words: ((a >> 5) * 2^26 + (b >> 6)) * 2^-53, exact in float64."""
    return ((a >> np.uint64(5)).astype(np.float64) * 67108864.0 + (b >> np.uint64(6)).astype(np.float64)) * 2.0 ** -53


def per_block(seed, samples, ctr):
    return philox4x32_10(*indexed_counter(TAG_PER, samples, ctr), seed & 0xFFFFFFFF, seed >> 32)


def descend(tree, u):
    """From node 1: left when u < tree[2k] or tree[2k+1] == 0, else u -= tree[2k] and right.  -> leaf node indices."""
    L = tree.size // 2
    node = np.ones(u.shape, np.int64)
    u = u.copy()
    while L > 1:
        left, right = tree[2 * node], tree[2 * node + 1]
        go_right = ~(u < left) & (right != 0)
        u = np.where(go_right, u - left, u)
        node = 2 * node + go_right
        L //= 2
    return node


def restated_draws(tree, seed, ctr, batch, beta, size):
    """-> (slots int64, weights float64) of per_sample_kernel for one call."""
    L = tree.size // 2
    total = tree[1]
    if total == 0:
        return np.zeros(batch, np.int64), np.zeros(batch)
    j = np.arange(batch, dtype=np.uint64)
    w0, w1, _, _ = per_block(seed, j, ctr)
    u = (j.astype(np.float64) + u53(w0, w1)) / float(batch) * total
    slots = descend(tree, u) - L
    w = (float(size) * (tree[L + slots] / total)) ** -beta
    return slots, w / w.max()


class Model:
    """The tree and per_meta as the three calls leave them, restated."""

    def __init__(self, capacity):
        self.cap, self.L = capacity, leaves_for(capacity)
        self.leaves = np.zeros(self.L)
        self.seen_appends, self.seen_head, self.maxp, self.missed, self.refused = 0, 0, 1.0, 0, 0

    def sync(self, ring_meta):
        head, _, size, appends = (int(v) for v in ring_meta)
        d = appends - self.seen_appends
        if d == 1:
            n = (head - self.seen_head) % self.cap or self.cap
            self.leaves[(self.seen_head + np.arange(n)) % self.cap] = self.maxp
        elif d != 0:
            self.leaves[:size] = self.maxp
            self.missed += 1
        self.seen_appends, self.seen_head = appends, head

    def synced_appends(self, ring_meta, m):
        """Several appends of m transitions, each followed by its sync, with no update in between."""
        head, _, _, appends = (int(v) for v in ring_meta)
        n = (appends - self.seen_appends) * m
        self.leaves[(self.seen_head + np.arange(n)) % self.cap] = self.maxp
        self.seen_appends, self.seen_head = appends, head

    def update(self, index, priority):
        index, priority = np.asarray(index, np.int64), np.asarray(priority, np.float64)
        if ((index < 0) | (index >= self.cap)).any() or not (np.isfinite(priority) & (priority >= 0)).all():
            self.refused += 1
            return
        for i, p in zip(index.tolist(), priority.tolist()):  # sequential: the last occurrence wins
            self.leaves[i] = p
        if index.size:
            self.maxp = max(self.maxp, float(priority.max()))

    def tree(self):
        return build_tree(self.leaves)


def assert_matches(rb, model, what=""):
    got = rb.tree.cpu().numpy()
    want = model.tree()
    assert np.array_equal(got.view(np.int64), want.view(np.int64)), \
        f"{what}: {int((got.view(np.int64) != want.view(np.int64)).sum())} tree elements differ"
    meta = rb.per_meta.cpu().numpy()
    assert meta[0] == model.seen_appends and meta[1] == model.seen_head, what
    assert meta[2:3].view(np.float64)[0] == model.maxp and meta[3] == model.missed and meta[4] == model.refused, what


# ---- the restatement itself and the stream tag (no device) -----------------------------------------------------------


def test_per_stream_tag_is_disjoint_from_the_other_device_streams():
    """Tag 6 joins the six layouts of test_device_philox_streams_are_pairwise_disjoint: over every layout's documented
    domain the upper half of counter word 2 is one constant per consumer, and the seven constants differ."""
    rng = np.random.default_rng(6)
    n = 4096

    def words(bits, edges):
        return np.concatenate([np.array(edges, np.uint64),
                               rng.integers(0, 2 ** min(bits, 63), n - len(edges), dtype=np.uint64) << np.uint64(max(bits - 63, 0))])

    w32 = lambda: words(32, [0, 1, 2 ** 31, 2 ** 32 - 1])
    w16 = lambda: words(16, [0, 1, 2 ** 15, 2 ** 16 - 1])
    w48 = lambda: words(48, [0, 2 ** 32 - 1, 2 ** 32, 2 ** 48 - 1])
    w64 = lambda: words(64, [0, 2 ** 32 - 1, 2 ** 32, 2 ** 64 - 1])
    layouts = {
        "reset pos": reset_counter(w32(), w32(), TAG_POS, w16(), w32()),
        "reset tgt": reset_counter(w32(), w32(), TAG_TGT, w16(), w32()),
        "reset vel": reset_counter(w32(), w32(), TAG_VEL, w16(), w32()),
        "rollout actions": action_counter(w32(), w16(), w64()),
        "policy": indexed_counter(TAG_POLICY, w48(), w64()),
        "sampler": indexed_counter(TAG_SAMPLE, w48(), w64()),
        "prioritized sampler": indexed_counter(TAG_PER, w48(), w64()),
    }
    tags = {}
    for name, ctr in layouts.items():
        ctr = np.broadcast_arrays(*(np.asarray(w, np.uint64) for w in ctr))
        assert all((w <= np.uint64(0xFFFFFFFF)).all() for w in ctr), name
        t = np.unique(ctr[2] >> np.uint64(16))
        assert t.size == 1, name
        tags[name] = int(t[0])
    assert tags["prioritized sampler"] == TAG_PER and len(set(tags.values())) == len(tags), tags


# ---- GPU ----------------------------------------------------------------------------------------------------------------


def _push(rb, m, g, sync=True):
    """Append m random transitions (obs_dim / act_dim of the ring); sync=False appends without the tree's sync."""
    import gym_uav_collision_avoidance_b200 as G

    args = (torch.rand((m, rb.obs_dim), generator=g, device="cuda"), torch.rand((m, rb.act_dim), generator=g, device="cuda"),
            torch.rand(m, generator=g, device="cuda"), torch.rand((m, rb.obs_dim), generator=g, device="cuda"),
            (torch.rand(m, generator=g, device="cuda") < 0.1).to(torch.uint8))
    (rb.push if sync else lambda *a: G.DeviceReplay.push(rb, *a))(*args)


def _priorities(rb, td):
    """(|td| + eps)^alpha exactly as update_priorities forms it (same torch ops on the same device)."""
    return (td.to(torch.float64).abs() + rb.eps).pow(rb.alpha).cpu().numpy()


@gpu
@pytest.mark.parametrize("capacity", [C4_M, 500_000, 1_000_003])
def test_sync_after_configs4_appends_matches_the_restatement(capacity):
    """Appends of one configs[4] step into rings that are not powers of two (and one exactly one step long: every append
    is a full-capacity append, n == 0), with learner updates in between so the appended slots take a moving maximum."""
    import gym_uav_collision_avoidance_b200 as G

    rb = G.PrioritizedDeviceReplay(capacity, 10, 2, seed=5)
    model = Model(capacity)
    g = torch.Generator(device="cuda").manual_seed(capacity)
    assert_matches(rb, model, "fresh")
    for step in range(9):
        _push(rb, C4_M, g)
        model.sync(rb.meta.tolist())
        assert_matches(rb, model, f"append {step}")
        idx = torch.randint(0, rb.size, (256,), generator=g, device="cuda")
        td = torch.randn(256, generator=g, device="cuda") * (1 + step)
        rb.update_priorities(idx, td)
        model.update(idx.cpu().numpy(), _priorities(rb, td))
        assert_matches(rb, model, f"update {step}")
    assert rb.missed_syncs == 0 and rb.refused_updates == 0


@gpu
def test_two_appends_between_syncs_refill_every_filled_slot():
    import gym_uav_collision_avoidance_b200 as G

    cap = 300_001
    rb = G.PrioritizedDeviceReplay(cap, 10, 2, seed=1)
    model = Model(cap)
    g = torch.Generator(device="cuda").manual_seed(3)
    _push(rb, 70_000, g)
    model.sync(rb.meta.tolist())
    rb.update_priorities(torch.arange(0, 70_000, 7, device="cuda"), torch.full((10_000,), 4.0, device="cuda"))
    model.update(np.arange(0, 70_000, 7), _priorities(rb, torch.full((10_000,), 4.0, device="cuda")))
    for _ in range(2):
        _push(rb, 100_000, g, sync=False)
    rb.sync()
    model.sync(rb.meta.tolist())
    assert_matches(rb, model, "two appends")
    assert rb.missed_syncs == 1 and bool((rb.tree[rb.leaves:rb.leaves + 270_000] == rb.max_priority).all())
    for _ in range(3):  # wraps, still unsynced: every slot is filled now
        _push(rb, 100_000, g, sync=False)
    rb.sync()
    model.sync(rb.meta.tolist())
    assert_matches(rb, model, "three appends, wrapped")
    assert rb.missed_syncs == 2
    rb.sync()  # nothing new
    assert_matches(rb, model, "idle sync")


@gpu
@pytest.mark.parametrize("n", [1, 256, 65_536])
def test_update_priorities_with_duplicates_matches_a_sequential_loop(n):
    import gym_uav_collision_avoidance_b200 as G

    cap = 1_000_000
    rb = G.PrioritizedDeviceReplay(cap, 4, 2, seed=2)
    model = Model(cap)
    g = torch.Generator(device="cuda").manual_seed(n)
    _push(rb, cap, g)  # full-capacity append into an empty ring
    model.sync(rb.meta.tolist())
    for rnd in range(3):
        # draw from a narrow range so that many slots repeat, in both orders of their priorities
        hi = max(1, n // 4) if rnd < 2 else cap
        idx = torch.randint(0, hi, (n,), generator=g, device="cuda")
        td = torch.randn(n, generator=g, device="cuda") * 10.0 ** rnd
        rb.update_priorities(idx, td)
        model.update(idx.cpu().numpy(), _priorities(rb, td))
        assert_matches(rb, model, f"n={n} round {rnd}")
    assert rb.refused_updates == 0


@gpu
@pytest.mark.parametrize("fused_append", [True, False])
def test_rollout_appends_keep_the_tree_in_step(fused_append):
    """BatchedRollout on a prioritized ring: the step kernel's own append (step_replay + sync) and the separate push
    (push + sync) both leave the tree equal to the restatement, with no missed sync."""
    import gym_uav_collision_avoidance_b200 as G

    B, N = 2048, 10
    env = G.BatchedMultiUAVWorld2D(B, num_agents=N, reset_mode=G.RESET_ON_DONE0, max_episode_steps=40, seed=4)
    rb = G.PrioritizedDeviceReplay(3 * B * N + 17, 10, 2, seed=4)
    ro = G.BatchedRollout(env, None, rb, action_mode="polar", warmup_uniform=True, fused_append=fused_append)
    assert ro.fused_append == fused_append
    model = Model(rb.capacity)
    ro.reset()
    g = torch.Generator(device="cuda").manual_seed(9)
    for step in range(7):
        ro.step()
        model.sync(rb.meta.tolist())
        assert_matches(rb, model, f"step {step}")
        assert int(rb.meta[3]) == step + 1
        idx = torch.randint(0, rb.size, (512,), generator=g, device="cuda")
        td = torch.randn(512, generator=g, device="cuda")
        rb.update_priorities(idx, td)
        model.update(idx.cpu().numpy(), _priorities(rb, td))
    assert rb.missed_syncs == 0


# weights: the device forms x = size * (leaf / total) and w = pow(x, -beta) / max pow(x, -beta) in float64 and rounds to
# float32; the restatement forms the same x (IEEE: identical) and numpy's pow.  CUDA's double pow has at most 2 ulp of
# error and glibc's under 1 ulp, so each of the two pows of the ratio differs by at most 3 ulp (3 * 2^-52 relative) and
# each side's division adds 2^-53: 14 * 2^-53 < 2^-49 in float64, then at most half a float32 ulp (2^-24); 2^-48 also
# covers the product of the two.
WEIGHT_REL = 2.0 ** -24 + 2.0 ** -48


def _filled_ring(cap, od, ad, seed, spread):
    import gym_uav_collision_avoidance_b200 as G

    rb = G.PrioritizedDeviceReplay(cap, od, ad, seed=seed)
    g = torch.Generator(device="cuda").manual_seed(seed)
    _push(rb, cap, g)
    td = torch.exp(torch.rand(cap, generator=g, device="cuda") * math.log(spread))  # priorities spanning `spread`
    rb.update_priorities(torch.arange(cap, device="cuda"), td)
    return rb


@gpu
@pytest.mark.parametrize("batch", [1, 256, 4096])
def test_draws_match_the_restatement(batch):
    cap = 700_001
    rb = _filled_ring(cap, 17, 3, seed=11, spread=1e4)
    g = torch.Generator(device="cuda").manual_seed(batch)
    for seed in (0, 11, 2 ** 63 - 25):
        rb._sample_seed = seed
        for k in range(3):
            if k == 2:
                _push(rb, 5000, g)  # the counter follows the appends, and new slots enter with the maximum
                rb._per_draws += 2 ** 32
            beta = (0.4, 1.0, 0.0)[k]
            draw, appends, size = rb._per_draws, int(rb.meta[3]), int(rb.meta[2])
            tree = rb.tree.cpu().numpy()
            s, a, r, n, m, idx, w = rb.sample_prioritized(batch, beta)
            want_idx, want_w = restated_draws(tree, seed, draw + appends, batch, beta, size)
            assert np.array_equal(idx.cpu().numpy(), want_idx), (seed, k)
            got_w = w.cpu().numpy().astype(np.float64)
            assert (np.abs(got_w - want_w) <= WEIGHT_REL * want_w).all(), (seed, k, np.abs(got_w - want_w).max())
            assert got_w.max() == 1.0 or np.abs(got_w.max() - 1.0) <= WEIGHT_REL
            t = torch.from_numpy(want_idx).cuda()
            assert torch.equal(s, rb.state[t]) and torch.equal(a, rb.action[t]) and torch.equal(n, rb.next_state[t])
            assert torch.equal(r, rb.reward[t]) and torch.equal(m, rb.mask[t])
            assert bool((rb.tree[rb.leaves + idx] > 0).all())


@gpu
def test_slot_frequencies_follow_the_priorities():
    """4,096 slots with fixed priorities spanning 1e3, 2^22 draws at a fixed seed: the slot counts pass a chi-square test
    against p_i / sum(p) (bins with an expected count below 5 merged).  Deterministic: seed and priorities are fixed."""
    from scipy import stats

    import gym_uav_collision_avoidance_b200 as G

    cap = 4096
    rb = G.PrioritizedDeviceReplay(cap, 2, 2, seed=123)
    z = torch.zeros(cap, device="cuda")
    rb.push(z[:, None].repeat(1, 2), z[:, None].repeat(1, 2), z, z[:, None].repeat(1, 2), torch.zeros(cap, dtype=torch.uint8, device="cuda"))
    p = np.random.default_rng(7).permutation(np.logspace(0, 3, cap))
    from gym_uav_collision_avoidance_b200 import ops

    ops.per_update(rb.tree, rb.per_meta, torch.arange(cap, device="cuda"), torch.from_numpy(p).cuda(), cap)
    counts = torch.zeros(cap, dtype=torch.int64, device="cuda")
    batch = 1 << 16
    out = None
    for _ in range((1 << 22) // batch):
        out = rb.sample_prioritized(batch, 0.5, out=out)
        counts += torch.bincount(out[5], minlength=cap)
    counts = counts.cpu().numpy()
    expected = p / p.sum() * (1 << 22)
    order = np.argsort(expected)
    obs_m, exp_m, acc_o, acc_e = [], [], 0, 0.0
    for i in order:  # merge the smallest bins until each holds at least 5 expected draws
        acc_o += counts[i]
        acc_e += expected[i]
        if acc_e >= 5:
            obs_m.append(acc_o)
            exp_m.append(acc_e)
            acc_o, acc_e = 0, 0.0
    if acc_e:
        obs_m[-1] += acc_o
        exp_m[-1] += acc_e
    res = stats.chisquare(np.array(obs_m, np.float64), np.array(exp_m))
    assert counts.sum() == 1 << 22 and res.pvalue > 1e-3, res


@gpu
def test_empty_ring_yields_slot_0_with_weight_0():
    import gym_uav_collision_avoidance_b200 as G

    rb = G.PrioritizedDeviceReplay(1000, 5, 2, seed=1)
    s, a, r, n, m, idx, w = rb.sample_prioritized(300, 0.4)
    assert bool((idx == 0).all()) and bool((w == 0).all()) and not bool(s.any()) and not bool(r.any())
    assert rb.tree.abs().sum().item() == 0.0  # the ticket in element 0 is back to 0


@gpu
@pytest.mark.parametrize("case", ["index_at_capacity", "negative_index", "negative_priority", "nan_priority", "inf_priority"])
def test_bad_updates_are_dropped_whole(case):
    import gym_uav_collision_avoidance_b200 as G
    from gym_uav_collision_avoidance_b200 import ops

    cap = 5000
    rb = G.PrioritizedDeviceReplay(cap, 3, 2, seed=1)
    model = Model(cap)
    _push(rb, 3000, torch.Generator(device="cuda").manual_seed(1))
    model.sync(rb.meta.tolist())
    idx = torch.arange(0, 2000, 2, device="cuda")
    pr = torch.linspace(0.5, 50.0, 1000, dtype=torch.float64, device="cuda")  # would raise the maximum
    k = 637
    if case == "index_at_capacity":
        idx[k] = cap
    elif case == "negative_index":
        idx[k] = -1
    else:
        pr[k] = {"negative_priority": -1e-300, "nan_priority": float("nan"), "inf_priority": float("inf")}[case]
    before = rb.tree.clone()
    ops.per_update(rb.tree, rb.per_meta, idx, pr, cap)
    model.update(idx.cpu().numpy(), pr.cpu().numpy())
    assert torch.equal(rb.tree, before) and rb.max_priority == 1.0 and rb.refused_updates == 1
    assert_matches(rb, model, case)
    rb.update_priorities(torch.tensor([1, 2], device="cuda"), torch.tensor([float("nan"), 1.0], device="cuda"))
    assert rb.refused_updates == 2


def test_capacity_beyond_2_26_is_refused_before_any_launch():
    import gym_uav_collision_avoidance_b200 as G

    with pytest.raises(ValueError, match="2\\^26"):
        G.PrioritizedDeviceReplay(2 ** 26 + 1, 10, 2)


@gpu
def test_captured_acting_and_learner_steps_replay_correctly():
    """An acting step (BatchedRollout on a prioritized ring, fused append + sync) and a learner step (sample_prioritized +
    update_priorities) each captured once: every replay keeps the tree equal to the restatement, and the learner's draws
    move on as the ring grows."""
    import gym_uav_collision_avoidance_b200 as G

    B, N = 512, 10
    env = G.BatchedMultiUAVWorld2D(B, num_agents=N, reset_mode=G.RESET_ON_DONE0, max_episode_steps=40, seed=2)
    rb = G.PrioritizedDeviceReplay(B * N * 5 + 3, 10, 2, seed=8, alpha=0.7, eps=1e-3)
    ro = G.BatchedRollout(env, None, rb, action_mode="polar", warmup_uniform=True)
    assert ro.fused_append
    model = Model(rb.capacity)
    ro.reset()
    batch, beta = 256, 0.5
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        ro.run(2)
        out = rb.sample_prioritized(batch, beta)
        rb.update_priorities(out[5], out[2] * 3.0 - 1.0)
    torch.cuda.current_stream().wait_stream(s)
    torch.cuda.synchronize()
    model.synced_appends(rb.meta.tolist(), B * N)
    model.update(out[5].cpu().numpy(), _priorities(rb, out[2] * 3.0 - 1.0))
    assert_matches(rb, model, "warm-up")

    act, learn = torch.cuda.CUDAGraph(), torch.cuda.CUDAGraph()
    with torch.cuda.graph(act):
        ro.run(2)
    draw = rb._per_draws
    with torch.cuda.graph(learn):
        rb.sample_prioritized(batch, beta, out=out)
        rb.update_priorities(out[5], out[2] * 3.0 - 1.0)
    torch.cuda.synchronize()
    assert_matches(rb, model, "capturing launches nothing")
    seen = []
    for rnd in range(4):
        before = rb.meta.tolist()
        act.replay()
        torch.cuda.synchronize()
        after = rb.meta.tolist()
        assert after[3] == before[3] + 2
        model.synced_appends(after, B * N)
        assert_matches(rb, model, f"acting replay {rnd}")
        tree = rb.tree.cpu().numpy()
        learn.replay()
        torch.cuda.synchronize()
        want_idx, want_w = restated_draws(tree, rb._sample_seed, draw + after[3], batch, beta, after[2])
        assert np.array_equal(out[5].cpu().numpy(), want_idx), rnd
        got_w = out[6].cpu().numpy().astype(np.float64)
        assert (np.abs(got_w - want_w) <= WEIGHT_REL * want_w).all(), rnd
        model.update(want_idx, _priorities(rb, out[2] * 3.0 - 1.0))
        assert_matches(rb, model, f"learner replay {rnd}")
        seen.append(want_idx)
    assert all(not np.array_equal(seen[i], seen[i + 1]) for i in range(len(seen) - 1))
    assert rb.missed_syncs == 0
