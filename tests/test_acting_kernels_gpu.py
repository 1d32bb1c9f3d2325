"""The two kernels of an acting step besides the env step — `policy_act_kernel` (csrc/uavca_policy.cu: tcgen05 MLP,
output heads, Philox / Box-Muller noise, tanh squash) and `replay_sample_kernel` (csrc/uavca_kernels.cu: device-drawn
replay slots) — against restatements kept in this file:

* Philox4x32-10 over numpy uint64 (pinned to the Random123 known answers) and every device counter layout;
* Box-Muller exactly as the kernel forms its uniforms, the rest in float64;
* the policy in float64 with fp16 rounding at exactly the kernel's quantisation points (the "emulation"), and the
  unquantised float64 policy;
* the replay slots, which are integer and IEEE float64 arithmetic and so are restated exactly.

Every tolerance is derived below from the documented error of each operation, not fitted to a run.  Tests without the
`gpu` marker need no device."""
import math

import numpy as np
import pytest
import torch

gpu = pytest.mark.gpu

M32 = np.uint64(0xFFFFFFFF)
U24 = 2.0 ** -24  # unit roundoff of float32 round-to-nearest
# CUDA C++ Programming Guide, single-precision intrinsics: __logf on [0.5, 2] and __sincosf on [-pi, pi] have an absolute
# error of at most 2^-21.41; __logf elsewhere at most 3 ulp; __expf(x) at most 2 + floor(|1.173 x|) ulp; __fdividef 2 ulp.
INTRINSIC_ABS = 2.0 ** -21.41
TWO_PI_F32 = float(np.float32(2 * math.pi))  # the constant the kernel multiplies u2 by, rounded to float32


# ---- Philox4x32-10 ------------------------------------------------------------------------------------------------------


def philox4x32_10(c0, c1, c2, c3, k0, k1):
    """Philox4x32-10 (Salmon et al., SC'11) on numpy uint64 arrays holding 32-bit words; broadcasts over the counters."""
    c0, c1, c2, c3 = np.broadcast_arrays(*(np.asarray(c, dtype=np.uint64) & M32 for c in (c0, c1, c2, c3)))
    k0, k1 = np.uint64(k0) & M32, np.uint64(k1) & M32
    for _ in range(10):
        p0 = np.uint64(0xD2511F53) * c0  # < 2^64: exact in uint64
        p1 = np.uint64(0xCD9E8D57) * c2
        c0, c1, c2, c3 = (p1 >> np.uint64(32)) ^ c1 ^ k0, p1 & M32, (p0 >> np.uint64(32)) ^ c3 ^ k1, p0 & M32
        k0 = (k0 + np.uint64(0x9E3779B9)) & M32
        k1 = (k1 + np.uint64(0xBB67AE85)) & M32
    return c0, c1, c2, c3


def test_philox_restatement_reproduces_the_random123_known_answers():
    kat = [((0, 0, 0, 0, 0, 0), (0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8)),
           ((M32,) * 6, (0x408F276D, 0x41C83B0E, 0xA20BC7C6, 0x6D5451FD)),
           ((0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344, 0xA4093822, 0x299F31D0),
            (0xD16CFE09, 0x94FDCCEB, 0x5001E420, 0x24126EA1))]
    for args, want in kat:
        assert tuple(int(w) for w in philox4x32_10(*args)) == want
    # vectorised evaluation equals the scalar one
    rows = np.arange(1000, dtype=np.uint64)
    v = philox4x32_10(rows, 7, 3, 0, 11, 12)
    for r in (0, 1, 999):
        assert tuple(int(w[r]) for w in v) == tuple(int(w) for w in philox4x32_10(r, 7, 3, 0, 11, 12))


# ---- device counter layouts ---------------------------------------------------------------------------------------------
# Every key is a seed the caller picks (env seed, rollout action seed, policy seed, replay seed), and users pick the same
# small seeds everywhere, so two streams are only independent if their COUNTERS can never coincide.  The layouts
# (uavca_device.cuh) and the domain each one documents:

TAG_POS, TAG_TGT, TAG_VEL, TAG_ACT, TAG_POLICY, TAG_SAMPLE = range(6)


def reset_counter(env, episode, stream, uav, attempt):
    """Auto-reset draws: (global env, episode, stream << 16 | uav, attempt); stream 0..2, uav < 2^16, 32-bit words."""
    return env, episode, (np.uint64(stream) << np.uint64(16)) | np.asarray(uav, np.uint64), attempt


def action_counter(env, uav, t):
    """The rollout's random actions at global step t: (env, t >> 1, 3 << 16 | uav, t >> 33), each cut to 32 bits;
    uav < 2^16."""
    t = np.asarray(t, np.uint64)
    return env, (t >> np.uint64(1)) & M32, np.uint64(TAG_ACT << 16) | np.asarray(uav, np.uint64), (t >> np.uint64(33)) & M32


def indexed_counter(tag, index, ctr):
    """Policy rows and replay samples: (index, ctr, tag << 16 | index >> 32, ctr >> 32); index < 2^48, ctr < 2^64."""
    index, ctr = np.asarray(index, np.uint64), np.asarray(ctr, np.uint64)
    return index & M32, ctr & M32, np.uint64(tag << 16) | (index >> np.uint64(32)), ctr >> np.uint64(32)


def policy_block(seed, rows, ctr):
    return philox4x32_10(*indexed_counter(TAG_POLICY, rows, ctr), seed & 0xFFFFFFFF, seed >> 32)


def sampler_block(seed, samples, ctr):
    return philox4x32_10(*indexed_counter(TAG_SAMPLE, samples, ctr), seed & 0xFFFFFFFF, seed >> 32)


def test_device_philox_streams_are_pairwise_disjoint():
    """No two device consumers can ever form the same Philox counter, whatever their seeds: over each layout's documented
    domain (extremes and random interior points) the upper half of counter word 2 is one constant per consumer, and the
    six constants differ.  (The policy and the sampler used to put their call counter in words 2 and 3 untagged: with equal
    seeds the sampler's slot for sample j was the policy's Box-Muller u1 of UAV row j, and the env's reset stream of env
    `row` could be drawn as policy noise.)"""
    rng = np.random.default_rng(0)
    n = 4096

    def words(bits, edges):  # the domain's edges and random interior points
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
    }
    tags = {}
    for name, ctr in layouts.items():
        ctr = np.broadcast_arrays(*(np.asarray(w, np.uint64) for w in ctr))
        assert all((w <= M32).all() for w in ctr), f"{name}: a counter word exceeds 32 bits"
        t = np.unique(ctr[2] >> np.uint64(16))
        assert t.size == 1, f"{name}: counter word 2 carries more than one stream tag over its domain: {t[:8]}"
        tags[name] = int(t[0])
    assert len(set(tags.values())) == len(tags), f"two streams share a tag: {tags}"


# ---- Box-Muller as the kernel forms it ----------------------------------------------------------------------------------


def box_muller(x, y):
    """The kernel's u1, u2 (float32: ((code + 0.5f) * 2^-24) of the top 24 bits, the + 0.5f rounding to even for codes
    >= 2^23) and the float64 (eps0, eps1) = sqrt(-2 ln u1) (cos, sin)(2 pi u2) from exactly those uniforms."""
    u1 = ((np.asarray(x) >> np.uint64(8)).astype(np.float32) + np.float32(0.5)) * np.float32(2.0 ** -24)
    u2 = ((np.asarray(y) >> np.uint64(8)).astype(np.float32) + np.float32(0.5)) * np.float32(2.0 ** -24)
    rad = np.sqrt(-2.0 * np.log(u1.astype(np.float64)))
    th = 2 * np.pi * u2.astype(np.float64)
    return u1, u2, np.stack([rad * np.cos(th), rad * np.sin(th)], axis=-1)


def noise_error_bound(u1, u2):
    """Per-row bound on |kernel eps - box_muller eps| (both components), from the documented intrinsic errors:
      L = __logf(u1): |dL| <= 2^-21.41 on [0.5, 1], else 3 ulp;  -2L is exact;  rad = sqrtf(-2L) rounds once, and
        |sqrt(a) - sqrt(b)| <= min(sqrt|a - b|, |a - b| / sqrt(b));
      theta = fl(float32(2 pi) * u2): the constant's rounding plus one product rounding;
      __sincosf(theta), theta in [0, 2 pi): outside [-pi, pi] the guide gives no number.  The intrinsic scales the
        argument by 1/(2 pi) in float32 (an error of at most theta * 2^-23 in the angle, ~3.7e-7 at pi, which is what the
        2^-21.41 on [-pi, pi] is made of) before the hardware sine of the fraction of a turn, so the bound is taken as
        2^-21.41 * (1 + theta / pi): the documented figure at pi doubled, three times it at 2 pi;
      eps = rad * cs rounds once."""
    u1 = np.asarray(u1, np.float64)
    u2 = np.asarray(u2, np.float64)
    L = np.log(u1)
    ulp_L = np.spacing(np.abs(L).astype(np.float32)).astype(np.float64)
    dL = np.where(u1 >= 0.5, INTRINSIC_ABS, 3 * ulp_L)
    rad = np.sqrt(-2 * L)
    da = 2 * dL
    with np.errstate(divide="ignore"):
        drad = np.minimum(np.sqrt(da), np.where(rad > 0, da / np.where(rad > 0, rad, 1), np.inf))
    drad = drad + U24 * (rad + drad)
    th = 2 * np.pi * u2
    dth = abs(TWO_PI_F32 - 2 * np.pi) * u2 + U24 * th
    dcs = dth + INTRINSIC_ABS * (1 + (th + dth) / np.pi)
    return drad + (rad + drad) * dcs + U24 * (rad + drad) * (1 + dcs)


def expf_rel(x):
    """Relative error bound of __expf(x): (2 + floor(|1.173 x|)) ulp, one ulp <= 2^-23 of the value."""
    return (2 + np.floor(np.abs(1.173 * x))) * 2.0 ** -23


def tanh_fast_error(x):
    """|tanh_fast(x) - tanh(x)| for the kernel's 1 - 2 / (__expf(2|x|) + 1): __expf relative error e_r enters
    2/(e+1) as e/(e+1) e_r; + 1 rounds (2^-24), __fdividef 2 ulp (<= 2^-22 relative), 1 - q rounds (2^-24)."""
    ax = np.abs(x)
    with np.errstate(over="ignore"):
        e = np.exp(2 * ax)
        q = 2 / (e + 1)
    rel_q = expf_rel(2 * ax) * np.where(np.isfinite(e), e / (e + 1), 1.0) + U24 + 2.0 ** -22
    return q * rel_q + U24


def action_error_bound(mean, log_std, eps, deps):
    """Per-row bound on |kernel action - tanh(mean + exp(log_std) eps)| with (mean, log_std) the kernel's own head values
    (the kernel samples from exactly those floats) and eps within deps of the kernel's draw:
    std = __expf(log_std); x = fmaf(std, eps, mean) rounds once; tanh_fast; tanh is 1-Lipschitz.  Doubled to cover
    the second-order products dropped in the terms above."""
    std = np.exp(log_std)
    dstd = std * expf_rel(log_std)
    x = mean + std * eps
    dx = dstd * (np.abs(eps) + deps) + std * deps
    dx = dx + U24 * (np.abs(x) + dx)
    return 2 * (dx + tanh_fast_error(x))


def test_box_muller_uniforms_round_like_the_kernel():
    top = np.uint64(2 ** 24 - 1) << np.uint64(8)
    codes = np.array([0, 1, 2 ** 23 - 1, 2 ** 23, 2 ** 24 - 4, 2 ** 24 - 3, 2 ** 24 - 2, 2 ** 24 - 1], np.uint64)
    u1, u2, eps = box_muller(codes << np.uint64(8), np.zeros_like(codes))
    assert u1[0] == np.float32(2.0 ** -25) and u1[1] == np.float32(1.5 * 2.0 ** -24)
    assert u1[2] == np.float32((2 ** 23 - 0.5) * 2.0 ** -24)  # below 2^23 the + 0.5 is exact
    # at and above 2^23 code + 0.5 is a tie that float32 rounds to even
    assert u1[3] == np.float32(2.0 ** -1)
    assert u1[4] == np.float32(1 - 2.0 ** -22) and u1[5] == np.float32(1 - 2.0 ** -23)
    assert u1[6] == np.float32(1 - 2.0 ** -23) and u1[7] == np.float32(1.0)
    assert eps[7, 0] == 0.0  # the top code: radius 0
    assert np.isfinite(eps).all() and np.abs(eps).max() <= math.sqrt(50 * math.log(2)) + 1e-12  # u1 >= 2^-25
    assert box_muller(np.array([0], np.uint64), np.array([top]))[1][0] == np.float32(1.0)  # u2 = 1: theta = 2 pi
    # the bound grows where sqrt amplifies the log error (u1 -> 1) and stays ~1e-6 elsewhere
    b = noise_error_bound(u1, np.full(u1.shape, 0.3, np.float32))
    assert b[7] > 1e-4 and b[3] < 5e-6


# Pairs (call counter, row) of the policy stream with seed 0 whose u1 code is one of the top four or bottom two, or whose
# u2 code sits at 0, 1/4, 1/2, 3/4 or 1 of the circle: found by evaluating philox4x32_10 over rows [0, 2^22) for the
# counters 0..23 (a few seconds of numpy; test_extreme_draw_table_holds_what_it_claims re-derives each entry).
EXTREME_DRAWS = [  # (counter, row, u1 code, u2 code)
    (8, 580460, 2 ** 24 - 1, 9599689), (13, 3083347, 2 ** 24 - 1, 10734064), (14, 4081194, 2 ** 24 - 1, 11661258),
    (13, 1903734, 2 ** 24 - 2, 14989319), (13, 3689163, 2 ** 24 - 2, 8330038),
    (0, 1675950, 2 ** 24 - 3, 11642301), (9, 93879, 2 ** 24 - 3, 10914211),
    (9, 688129, 2 ** 24 - 4, 5186024),
    (9, 3258637, 0, 1363630), (14, 630660, 0, 4936360),
    (0, 2867445, 1, 3030827), (0, 3569142, 1, 7201011),
    (9, 1140698, 2545847, 0), (9, 2823335, 3858134, 0),
    (14, 814306, 3851029, 2 ** 22), (14, 2386229, 16493175, 2 ** 22),
    (0, 1119596, 10075758, 2 ** 23), (0, 3062373, 7284533, 2 ** 23),
    (9, 196626, 10767053, 3 * 2 ** 22), (9, 3804179, 16537386, 3 * 2 ** 22),
    (0, 788480, 12234987, 2 ** 24 - 1),
]


def test_extreme_draw_table_holds_what_it_claims():
    for ctr, row, c1, c2 in EXTREME_DRAWS:
        x, y, _, _ = policy_block(0, row, ctr)
        assert (int(x) >> 8, int(y) >> 8) == (c1, c2), (ctr, row)
    c1s = {c1 for _, _, c1, _ in EXTREME_DRAWS}
    c2s = {c2 for _, _, _, c2 in EXTREME_DRAWS}
    assert {2 ** 24 - 1, 2 ** 24 - 2, 2 ** 24 - 3, 2 ** 24 - 4, 0, 1} <= c1s
    assert {0, 2 ** 22, 2 ** 23, 3 * 2 ** 22, 2 ** 24 - 1} <= c2s


# ---- replay slots -------------------------------------------------------------------------------------------------------


def restated_slots(seed, ctr, batch, head, size, cap, recency):
    """replay_sample_kernel's slots: x = word 0 of the sampler's block for (sample, ctr); uniform (x * size) >> 32;
    recency-weighted age = floor(sqrt((x + 0.5) / 2^32) * size) <= size - 1 from the oldest slot (IEEE float64: the
    kernel's sqrt and product round exactly as numpy's)."""
    if size == 0:
        return np.zeros(batch, np.int64)
    x = sampler_block(seed, np.arange(batch, dtype=np.uint64), ctr)[0]
    if recency:
        age = (np.sqrt((x.astype(np.float64) + 0.5) * 2.0 ** -32) * float(size)).astype(np.int64)
        age = np.minimum(age, size - 1)
        slot = (head if size == cap else 0) + age
        return np.where(slot >= cap, slot - cap, slot)
    return ((x * np.uint64(size)) >> np.uint64(32)).astype(np.int64)


def test_replay_slot_restatement_follows_both_laws():
    """Over 2^20 evenly spaced 32-bit draws the restated slots realise the laws exactly: uniform P = 1/size, recency
    P(age a) = (2a + 1) / size^2 (p_i ~ i + 1/2), both within one draw's share per slot."""
    x = (np.arange(2 ** 20, dtype=np.uint64) << np.uint64(12)) + np.uint64(2048)
    for size in (1, 3, 1000):
        uni = ((x * np.uint64(size)) >> np.uint64(32)).astype(np.int64)
        assert uni.min() >= 0 and uni.max() < size
        assert np.abs(np.bincount(uni, minlength=size) / x.size - 1 / size).max() <= 1.5 / x.size + 1e-12
        age = np.minimum((np.sqrt((x.astype(np.float64) + 0.5) * 2.0 ** -32) * size).astype(np.int64), size - 1)
        want = (2 * np.arange(size) + 1) / size ** 2
        assert np.abs(np.bincount(age, minlength=size) / x.size - want).max() <= 1.5 / x.size + 1e-12


# ======================================= GPU: the policy kernel ==========================================================


def _sms():
    return torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count


def _rows(spec):
    """Row counts relative to the SM count S (the kernel's grid is min(tiles, S), each CTA loops over its tiles)."""
    S = _sms()
    return {"1": 1, "127": 127, "128": 128, "129": 129, "128S-1": 128 * S - 1, "128S": 128 * S, "128S+1": 128 * S + 1,
            "2x128S+5": 2 * 128 * S + 5, "163840": 163840}[spec]


def _policy(seed=3, biases=0.3):
    import gym_uav_collision_avoidance_b200 as G

    torch.manual_seed(seed)
    p = G.GaussianPolicy(10, 2).cuda()
    with torch.no_grad():
        for lin in (p.linear1, p.linear2, p.mean_linear, p.log_std_linear):
            lin.bias.uniform_(-biases, biases)
    return p


def _params(p):
    """The module's parameters in float64, heads in the kernel's order (mean0, mean1, log_std0, log_std1)."""
    d = lambda t: t.detach().double()
    if hasattr(p, "l1"):  # TD3-style actor: the log_std head pinned at its floor by FusedGaussianPolicy
        W3 = torch.cat([d(p.l3.weight), torch.zeros_like(d(p.l3.weight))])
        b3 = torch.cat([d(p.l3.bias), torch.full_like(d(p.l3.bias), -20.0)])
        l1, l2 = p.l1, p.l2
    else:
        W3 = torch.cat([d(p.mean_linear.weight), d(p.log_std_linear.weight)])
        b3 = torch.cat([d(p.mean_linear.bias), d(p.log_std_linear.bias)])
        l1, l2 = p.linear1, p.linear2
    return dict(W1=d(l1.weight), b1=d(l1.bias), W2=d(l2.weight), b2=d(l2.bias), W3=W3, b3=b3)


def f16(x):
    """Round float64 to the nearest fp16 value, ties to even, in float64 (exact; |x| < 65504)."""
    _, e = torch.frexp(x)  # |x| in [2^(e-1), 2^e): fp16 spacing 2^(e-11), at least 2^-24 (subnormals)
    q = ((torch.clamp(e.to(torch.int64) - 11, min=-24) + 1023) << 52).view(torch.float64)  # 2^k from its bits, exact
    return torch.round(x / q) * q  # torch.round: half to even


def test_fp16_rounding_restatement_is_numpys():
    """f16 against numpy's float64 -> float16 conversion (correctly rounded): random values over the whole fp16 range,
    subnormals, and exact ties between neighbouring fp16 values."""
    rng = np.random.default_rng(1)
    x = np.concatenate([rng.standard_normal(20000) * 10.0 ** rng.integers(-8, 4, 20000),
                        rng.uniform(-2.0 ** -14, 2.0 ** -14, 5000), [0.0, -0.0, 65504.0, 2.0 ** -24, 3 * 2.0 ** -25]])
    h = np.float16(rng.uniform(-1000, 1000, 5000)).astype(np.float64)  # midpoints between fp16 neighbours
    x = np.concatenate([x, (h + np.nextafter(h.astype(np.float16), np.float16(np.inf)).astype(np.float64)) / 2])
    x = x[np.abs(x) <= 65504]
    assert np.array_equal(f16(torch.from_numpy(x)).numpy(), x.astype(np.float16).astype(np.float64))


def _clamp_heads(pre):
    return torch.cat([pre[:, :2], pre[:, 2:].clamp(-20.0, 2.0)], 1)


TC_STEP = 2.0 ** -22  # tcgen05.mma, fp32 accumulate: error per K=16 step <= 2^-22 (|accumulator| + sum |products|)
FMA_DEPTH = 22        # heads_fma: 16 chained FMAs per lane, 2 shuffle adds, the 4 column groups + b3: 22 roundings


def emulate(P, obs):
    """The kernel's arithmetic in float64 with fp16 rounding where the kernel rounds, and a per-row bound on the kernel's
    remaining difference (fp32 accumulation order, fp16 rounding flips that follow from it):
      x = fp16(obs); W1, b1, W2, b2, W3, b3 = fp16 (the host packing);
      d1 = x W1^T + b1 (one MMA step: |err| <= B1 = TC_STEP * S1, S1 = |x| |W1|^T + |b1|, + the fp32 rounding of d1);
      h1 = fp16(relu(d1)): fp16 o relu is monotone, so the kernel's h1 lies in [fp16(relu(d1 - B1)), fp16(relu(d1 + B1))]
        and dh1 = the wider side of that interval around the emulated h1 (0 unless d1 sits within B1 of a rounding edge,
        then one fp16 ulp);
      x2 = h1 W2^T + b2 (16 MMA steps, b2 added in fp32): the kernel's x2 differs by W2 (h1' - h1) (the flips, linear) plus
        acc2 = 16 TC_STEP (h1 |W2|^T + |W2| dh1) + 2^-24 |x2|; |W2| dh1 + acc2 bounds the whole difference (dx2);
      h2 = relu(x2), unrounded.  Units with |x2| > dx2 keep their ReLU state: through those the flips reach the heads
        linearly, as sum_k G_jk (h1'_k - h1_k) with G = W3 diag(active) W2 (bounded by |G| dh1), and acc2 through |W3|;
        a unit that may change state contributes at most |W3| dx2;
      heads = h2 W3^T + b3 (fp32 FMAs): + FMA_DEPTH 2^-24 (h2 |W3|^T + |W3| dx2 + |b3|);
      then the clamp of log_std (1-Lipschitz).
    -> (heads [M, 4], bound [M, 4], heads before the clamp [M, 4])."""
    Q = {k: f16(v) for k, v in P.items()}
    x = f16(obs)
    S1 = x.abs() @ Q["W1"].abs().T + Q["b1"].abs()
    d1 = x @ Q["W1"].T + Q["b1"]
    B1 = TC_STEP * S1 + U24 * (d1.abs() + TC_STEP * S1)
    h1 = f16(torch.relu(d1))
    dh1 = torch.maximum(f16(torch.relu(d1 + B1)) - h1, h1 - f16(torch.relu(d1 - B1)))
    del S1, B1, d1
    aW2 = Q["W2"].abs()
    prop2 = dh1 @ aW2.T
    x2 = h1 @ Q["W2"].T + Q["b2"]
    acc2 = 16 * TC_STEP * (h1 @ aW2.T + prop2) + U24 * (x2.abs() + prop2)
    dx2 = prop2 + acc2
    h2 = torch.relu(x2)
    sure = x2.abs() > dx2
    active = (x2 > 0) & sure
    aW3 = Q["W3"].abs()
    bound = torch.empty((obs.shape[0], 4), dtype=obs.dtype, device=obs.device)
    for j in range(4):
        G = (Q["W3"][j] * active) @ Q["W2"]
        bound[:, j] = ((G.abs() * dh1).sum(1) + (acc2 * active) @ aW3[j] + (dx2 * ~sure) @ aW3[j]
                       + FMA_DEPTH * U24 * (h2 @ aW3[j] + dx2 @ aW3[j] + Q["b3"][j].abs()))
    pre = h2 @ Q["W3"].T + Q["b3"]
    return _clamp_heads(pre), bound, pre


def float64_policy(P, obs):
    """The unquantised policy in float64 and, per row and head, sigma of the head error that rounding every fp16
    operand causes: each rounding is a relative error of at most 2^-11 (RNE, 11 significant bits), modelled as uniform,
    variance 2^-22 / 3, independent between operands.  To first order the head error is sum_i (d head / d v_i) v_i delta_i
    over every rounded value v_i (obs, W1, b1, h1, W2, b2, W3, b3), so its variance is
    2^-22 / 3 * sum_i (d head / d v_i)^2 v_i^2, formed below without materialising the per-weight gradients."""
    W1, b1, W2, b2, W3, b3 = (P[k] for k in ("W1", "b1", "W2", "b2", "W3", "b3"))
    d1 = obs @ W1.T + b1
    h1 = torch.relu(d1)
    d2 = h1 @ W2.T + b2
    h2 = torch.relu(d2)
    pre = h2 @ W3.T + b3
    h1W2sq = (h1 * h1) @ (W2 * W2).T          # [M, 256]: sum_k W2_nk^2 h1_k^2
    obsW1sq = (obs * obs) @ (W1 * W1).T        # [M, 256]: sum_i W1_ki^2 obs_i^2
    var = torch.empty_like(pre)
    for j in range(4):
        g2 = W3[j] * (d2 > 0)                  # d head / d (d2 + b2)
        gh1 = g2 @ W2                          # d head / d h1
        g1 = gh1 * (d1 > 0)                    # d head / d d1
        var[:, j] = (b3[j] ** 2 + (h2 * h2) @ (W3[j] ** 2) + (g2 * g2) @ (b2 * b2) + ((g2 * g2) * h1W2sq).sum(1)
                     + ((gh1 * h1) ** 2).sum(1) + (g1 * g1) @ (b1 * b1) + ((g1 * g1) * obsW1sq).sum(1)
                     + (((g1 @ W1) * obs) ** 2).sum(1))
    return _clamp_heads(pre), torch.sqrt(var * 2.0 ** -22 / 3)


def _act(f, obs, noise=None):
    M = obs.shape[0]
    out = torch.full((M, 2), float("nan"), device=obs.device)
    head = torch.full((M, 4), float("nan"), device=obs.device)
    f.act(obs, out=out, noise=noise, head=head)
    torch.cuda.synchronize()
    return out, head


def _assert_within(got, want, bound, what):
    err = (got.double() - want).abs()
    bad = ~(err <= bound)  # NaN fails too
    if bad.any():
        i = int(torch.nonzero(bad.flatten())[0])
        raise AssertionError(f"{what}: {int(bad.sum())} values outside the bound; first at flat index {i}: got "
                             f"{got.flatten()[i].item()!r}, want {want.flatten()[i].item()!r}, bound {bound.flatten()[i].item():.3g}")


@gpu
@pytest.mark.parametrize("rows", ["1", "127", "128", "129", "128S-1", "128S", "128S+1", "2x128S+5", "163840"])
def test_policy_heads_match_the_fp16_emulation(rows):
    """Heads (mean, log_std) of every row within the emulation bound: one tile, ragged tiles, one tile per CTA, a CTA with
    a second tile, and configs[4]'s 163,840 rows."""
    import gym_uav_collision_avoidance_b200 as G

    M = _rows(rows)
    p = _policy()
    f = G.FusedGaussianPolicy(p, seed=9)
    g = torch.Generator(device="cuda").manual_seed(M)
    obs = torch.rand((M, 10), generator=g, device="cuda") * 2 - 1
    _, head = _act(f, obs)
    want, bound, _ = emulate(_params(p), obs.double())
    # the bound itself: ~5e-5 for a typical row (400x under the 2e-2 the fp32 comparison used to allow), < 4e-4 for every row
    assert float(bound.median()) < 1e-4 and float(bound.max()) < 4e-4, (float(bound.median()), float(bound.max()))
    _assert_within(head, want, bound, f"heads, {M} rows")


@gpu
def test_policy_heads_over_a_long_pipeline():
    """~2^22 rows (222 tiles per CTA on 148 SMs): every row at a tile edge, the first and last tiles of every CTA, and a
    random subset against the emulation; the rest must be finite."""
    import gym_uav_collision_avoidance_b200 as G

    S = _sms()
    M = (1 << 22) + 77
    p = _policy(seed=4)
    f = G.FusedGaussianPolicy(p, seed=1)
    g = torch.Generator(device="cuda").manual_seed(5)
    obs = torch.rand((M, 10), generator=g, device="cuda") * 4 - 2
    _, head = _act(f, obs)
    assert bool(torch.isfinite(head).all())
    tiles = (M + 127) // 128
    edges = torch.arange(tiles, device="cuda") * 128
    pick = [edges, edges + 127, edges + 63]
    for t in list(range(S)) + list(range(tiles - S, tiles)):  # first and last tile of every CTA: all their rows
        pick.append(torch.arange(t * 128, t * 128 + 128, device="cuda"))
    pick.append(torch.randint(0, M, (40000,), generator=g, device="cuda"))
    idx = torch.cat(pick).clamp_(max=M - 1).unique()
    want, bound, _ = emulate(_params(p), obs[idx].double())
    _assert_within(head[idx], want, bound, f"heads of {idx.numel()} sampled rows out of {M}")


@gpu
@pytest.mark.parametrize("M", [1, 100, 128, 1000, 163840])
def test_policy_heads_match_the_float64_policy(M):
    """The precision of the acting path against the unquantised float64 policy (the fp32 PyTorch policy is the same up
    to its own rounding): heads within 7 sigma of the fp16-operand rounding error (float64_policy) plus the emulation
    bound; the action with caller-supplied noise within what those head errors and the sampling add; |action| <= 1."""
    import gym_uav_collision_avoidance_b200 as G

    p = _policy()
    f = G.FusedGaussianPolicy(p, seed=9)
    g = torch.Generator(device="cuda").manual_seed(M + 1)
    obs = torch.rand((M, 10), generator=g, device="cuda") * 2 - 1
    noise = torch.randn((M, 2), generator=g, device="cuda")
    act, head = _act(f, obs, noise)
    P = _params(p)
    want, sigma = float64_policy(P, obs.double())
    _, emu_bound, _ = emulate(P, obs.double())
    bound = 7 * sigma + emu_bound
    _assert_within(head, want, bound, "heads against the float64 policy")
    m, l = want[:, :2], want[:, 2:]
    dl = bound[:, 2:]
    n = noise.double()
    x = m + l.exp() * n
    dx = bound[:, :2] + l.exp() * n.abs() * torch.expm1(dl)
    hb = action_error_bound(head[:, :2].double().cpu().numpy(), head[:, 2:].double().cpu().numpy(), n.cpu().numpy(), 0.0)
    _assert_within(act, torch.tanh(x), dx + torch.from_numpy(hb).cuda(), "action with caller noise")
    assert float(act.abs().max()) <= 1.0


def _regime_policy(regime):
    import torch.nn as nn
    import gym_uav_collision_avoidance_b200 as G

    if regime == "td3":
        class Actor(nn.Module):  # pytorch_td3_temp/td3.py:14-27
            def __init__(self):
                super().__init__()
                self.l1, self.l2, self.l3 = nn.Linear(10, 256), nn.Linear(256, 256), nn.Linear(256, 2)

        torch.manual_seed(5)
        return Actor().cuda()
    p = _policy(seed=6)
    with torch.no_grad():
        if regime == "scaled":  # heads of O(10..100): hidden activations far from 1
            for lin in (p.linear1, p.linear2, p.mean_linear, p.log_std_linear):
                lin.weight.mul_(2.5)
                lin.bias.mul_(2.5)
        elif regime == "log_std_clamp":  # log_std head 0 at ~+6 before the clamp, head 1 at ~-30
            p.log_std_linear.bias.copy_(torch.tensor([6.0, -30.0]))
        elif regime == "big_means":  # |mean| far beyond 10 with a small std: tanh saturates to exactly +-1
            p.mean_linear.bias.copy_(torch.tensor([14.0, -14.0]))
            p.log_std_linear.weight.zero_()
            p.log_std_linear.bias.fill_(-2.0)
    return p


@gpu
@pytest.mark.parametrize("regime", ["scaled", "log_std_clamp", "big_means", "td3"])
def test_policy_weight_regimes(regime):
    """Beyond default initialisation: scaled-up weights, log_std pushed through both clamp limits, means beyond +-10,
    and the TD3-style deterministic actor — heads at the emulation bound, Philox actions at the sampling bound."""
    import gym_uav_collision_avoidance_b200 as G

    p = _regime_policy(regime)
    seed, M = 21, 128 * _sms() + 50
    f = G.FusedGaussianPolicy(p, seed=seed)
    g = torch.Generator(device="cuda").manual_seed(7)
    obs = torch.rand((M, 10), generator=g, device="cuda") * 2 - 1
    act, head = _act(f, obs)
    P = _params(p)
    want, bound, pre = emulate(P, obs.double())
    _assert_within(head, want, bound, f"{regime}: heads")
    assert bool(torch.isfinite(act).all()) and float(act.abs().max()) <= 1.0
    u1, u2, eps = box_muller(*policy_block(seed, np.arange(M, dtype=np.uint64), 0)[:2])
    deps = noise_error_bound(u1, u2)[:, None]
    h = head.double().cpu().numpy()
    ref = np.tanh(h[:, :2] + np.exp(h[:, 2:]) * eps)
    ab = action_error_bound(h[:, :2], h[:, 2:], eps, deps)
    _assert_within(act, torch.from_numpy(ref).cuda(), torch.from_numpy(ab).cuda(), f"{regime}: actions")
    if regime == "log_std_clamp":
        hi, lo = pre[:, 2:] > 2 + bound[:, 2:], pre[:, 2:] < -20 - bound[:, 2:]
        assert int(hi[:, 0].sum()) == M and int(lo[:, 1].sum()) == M, "the regime does not reach both clamp limits"
        assert bool((head[:, 2:][hi] == 2.0).all()) and bool((head[:, 2:][lo] == -20.0).all())
    if regime == "big_means":
        m = head[:, :2].double()
        assert float(m.abs().min()) > 10
        assert torch.equal(act, torch.sign(m).float()), "tanh of |x| > 9.1 is exactly +-1 in float32"
    if regime == "td3":
        assert bool((head[:, 2:] == -20.0).all())
        _assert_within(act, torch.tanh(head[:, :2].double()), torch.full_like(act, 1e-6, dtype=torch.float64),
                       "td3: action = tanh(mean)")


@gpu
@pytest.mark.parametrize("case", ["host_calls", "device_counter", "counter_above_2^32", "seed_above_2^32"])
def test_policy_samples_match_the_restated_noise(case):
    """Philox actions against tanh(mean + exp(log_std) eps) with the kernel's own heads and eps restated from
    (seed, row, calls + counter) in the policy's stream layout.  A block keyed to the wrong row or counter, or swapped
    sin and cos, moves the action by O(1)."""
    import gym_uav_collision_avoidance_b200 as G

    seed, calls, dev = {"host_calls": (9, 17, 0), "device_counter": (9, 0, 1234),
                        "counter_above_2^32": (9, 2 ** 32 + 3, 5), "seed_above_2^32": (2 ** 33 + 5, 1, 2)}[case]
    p = _policy()
    f = G.FusedGaussianPolicy(p, seed=seed)
    f.calls = calls
    f.counter.fill_(dev)
    M = 2 * 128 * _sms() + 5
    g = torch.Generator(device="cuda").manual_seed(11)
    obs = torch.rand((M, 10), generator=g, device="cuda") * 2 - 1
    act, head = _act(f, obs)
    assert int(f.counter) == dev + 1
    u1, u2, eps = box_muller(*policy_block(seed, np.arange(M, dtype=np.uint64), calls + dev)[:2])
    h = head.double().cpu().numpy()
    ref = np.tanh(h[:, :2] + np.exp(h[:, 2:]) * eps)
    ab = action_error_bound(h[:, :2], h[:, 2:], eps, noise_error_bound(u1, u2)[:, None])
    _assert_within(act, torch.from_numpy(ref).cuda(), torch.from_numpy(ab).cuda(), f"{case}: actions")


@gpu
def test_box_muller_extremes():
    """The kernel at the draws of EXTREME_DRAWS (mean 0, log_std 0: action = tanh(eps)): u1 codes at the top (u1 -> 1,
    where __logf of 1 - 2^-23 must not come out positive and feed sqrtf a negative number) and bottom (radius ~5.9), u2
    at the quadrant edges.  Every action finite, |a| <= 1, within the sampling bound; all 2^22 rows of each run finite."""
    import gym_uav_collision_avoidance_b200 as G

    p = _policy()
    with torch.no_grad():
        for prm in p.parameters():
            prm.zero_()
    f = G.FusedGaussianPolicy(p, seed=0)
    M = 1 << 22
    obs = torch.zeros((M, 10), device="cuda")
    for ctr in sorted({c for c, _, _, _ in EXTREME_DRAWS}):
        f.calls = ctr
        f.counter.zero_()
        act, head = _act(f, obs)
        assert bool((head == 0).all())
        rows = np.array([r for c, r, _, _ in EXTREME_DRAWS if c == ctr], np.uint64)
        u1, u2, eps = box_muller(*policy_block(0, rows, ctr)[:2])
        a = act[torch.from_numpy(rows.astype(np.int64)).cuda()]
        assert bool(torch.isfinite(a).all()), f"non-finite action at counter {ctr}, rows {rows}: {a.tolist()}"
        ab = action_error_bound(np.zeros_like(eps), np.zeros_like(eps), eps, noise_error_bound(u1, u2)[:, None])
        _assert_within(a, torch.from_numpy(np.tanh(eps)).cuda(), torch.from_numpy(ab).cuda(), f"counter {ctr}")
        bad = ~torch.isfinite(act).all(1)
        assert not bool(bad.any()), f"counter {ctr}: non-finite actions at rows {torch.nonzero(bad).flatten()[:8].tolist()}"
        assert float(act.abs().max()) <= 1.0


@gpu
def test_policy_rows_are_independent_bit_for_bit():
    """Rows do not interact: permuting the rows (and the caller's noise with them) permutes the outputs exactly; one
    observation at every position of every tile, on every CTA, gives identical bits; a NaN row changes no other row."""
    import gym_uav_collision_avoidance_b200 as G

    S = _sms()
    M = 2 * 128 * S + 5
    f = G.FusedGaussianPolicy(_policy(), seed=2)
    g = torch.Generator(device="cuda").manual_seed(13)
    obs = torch.rand((M, 10), generator=g, device="cuda") * 2 - 1
    noise = torch.randn((M, 2), generator=g, device="cuda")
    a0, h0 = _act(f, obs, noise)
    perm = torch.randperm(M, generator=g, device="cuda")
    a1, h1 = _act(f, obs[perm].contiguous(), noise[perm].contiguous())
    assert torch.equal(a1, a0[perm]) and torch.equal(h1, h0[perm])
    k = 1234
    a2, h2 = _act(f, obs[k].expand(M, 10).contiguous(), noise[k].expand(M, 2).contiguous())
    assert torch.equal(h2, h0[k].expand(M, 4)) and torch.equal(a2, a0[k].expand(M, 2))
    _, h3 = _act(f, obs[k].expand(M, 10).contiguous())  # Philox noise: the heads still agree bit for bit
    assert torch.equal(h3, h2)
    bad = torch.tensor([0, 127, 128 * S - 1, 128 * S, M - 1], device="cuda")
    obs_nan = obs.clone()
    obs_nan[bad, 3] = float("nan")
    a4, h4 = _act(f, obs_nan, noise)
    keep = torch.ones(M, dtype=torch.bool, device="cuda")
    keep[bad] = False
    assert torch.equal(a4[keep], a0[keep]) and torch.equal(h4[keep], h0[keep])


@gpu
def test_refresh_rewrites_the_weights_a_captured_graph_reads():
    """An acting step captured in a CUDA graph, then a learner update in place and `refresh()`: the replay acts with the
    new weights (refresh writes into the tensors the graph captured instead of allocating new ones)."""
    import gym_uav_collision_avoidance_b200 as G

    p = _policy()
    f = G.FusedGaussianPolicy(p, seed=5)
    M = 3000
    g = torch.Generator(device="cuda").manual_seed(17)
    obs = torch.rand((M, 10), generator=g, device="cuda") * 2 - 1
    noise = torch.randn((M, 2), generator=g, device="cuda")
    out, head = torch.empty((M, 2), device="cuda"), torch.empty((M, 4), device="cuda")
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        f.act(obs, out=out, noise=noise, head=head)
    torch.cuda.current_stream().wait_stream(s)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        f.act(obs, out=out, noise=noise, head=head)
    old = emulate(_params(p), obs.double())[0]
    ptrs = {k: getattr(f, k).data_ptr() for k in ("w1", "w2", "w2b", "w3", "w3b")}
    with torch.no_grad():  # an optimiser step: parameters change in place
        for prm in p.parameters():
            prm.mul_(-0.8).add_(0.02)
    f.refresh()
    assert {k: getattr(f, k).data_ptr() for k in ptrs} == ptrs
    graph.replay()
    torch.cuda.synchronize()
    want, bound, _ = emulate(_params(p), obs.double())
    assert float((want - old).abs().max()) > 0.1  # the update is visible in the heads
    _assert_within(head, want, bound, "heads after refresh() under graph replay")


_BAD_INPUTS = {
    "state_float64": lambda M: dict(state=torch.zeros((M, 10), dtype=torch.float64, device="cuda")),
    "state_on_cpu": lambda M: dict(state=torch.zeros((M, 10))),
    "state_numel": lambda M: dict(state=torch.zeros((M, 11), device="cuda")),
    "out_shape": lambda M: dict(out=torch.zeros((M + 1, 2), device="cuda")),
    "out_dtype": lambda M: dict(out=torch.zeros((M, 2), dtype=torch.float64, device="cuda")),
    "out_device": lambda M: dict(out=torch.zeros((M, 2))),
    "noise_shape": lambda M: dict(noise=torch.zeros((M, 1), device="cuda")),
    "noise_dtype": lambda M: dict(noise=torch.zeros((M, 2), dtype=torch.float16, device="cuda")),
    "noise_device": lambda M: dict(noise=torch.zeros((M, 2))),
    "head_shape": lambda M: dict(head=torch.zeros((M, 2), device="cuda")),
    "head_dtype": lambda M: dict(head=torch.zeros((M, 4), dtype=torch.float64, device="cuda")),
    "head_device": lambda M: dict(head=torch.zeros((M, 4))),
}


@gpu
@pytest.mark.parametrize("case", sorted(_BAD_INPUTS))
def test_act_rejects_mismatched_tensors_before_launch(case):
    import gym_uav_collision_avoidance_b200 as G

    M = 64
    f = G.FusedGaussianPolicy(_policy(), seed=1)
    kw = dict(state=torch.zeros((M, 10), device="cuda"), out=torch.full((M, 2), 7.0, device="cuda"))
    kw.update(_BAD_INPUTS[case](M))
    sentinel = kw["out"].clone()
    with pytest.raises(ValueError):
        f.act(kw.pop("state"), **kw)
    torch.cuda.synchronize()
    assert int(f.counter) == 0 and torch.equal(kw["out"], sentinel)


@gpu
def test_policy_noise_and_replay_slots_are_independent_draws():
    """BatchedRollout keys the policy's noise on the ring's append counter and examples build the ring with seed 0, the
    policy's seed: the slots sample_fused draws must not be a function of the UAVs' Box-Muller radii.  (With a shared
    counter layout slot j was u1 of row j: correlation 1.)"""
    import gym_uav_collision_avoidance_b200 as G

    p = _policy()
    with torch.no_grad():
        for prm in p.parameters():
            prm.zero_()  # action = tanh(eps)
    C, M = 1 << 20, 8192
    rb = G.DeviceReplay(C, 1, 1, seed=0)
    f = G.FusedGaussianPolicy(p, seed=0)
    f.counter, f.own_counter = rb.meta[3:4], False  # as BatchedRollout wires them
    z = torch.zeros(C, device="cuda")
    rb.push(z[:, None], z[:, None], z, z[:, None], torch.zeros(C, dtype=torch.uint8, device="cuda"))
    a = f.act(torch.zeros((M, 10), device="cuda"))
    idx = rb.sample_fused(M, want_index=True)[5]
    eps = torch.atanh(a.double())
    u1_policy = torch.exp(-0.5 * (eps * eps).sum(1))
    u1_slots = (idx.double() + 0.5) / C
    corr = float(torch.corrcoef(torch.stack([u1_policy, u1_slots]))[0, 1])
    assert abs(corr) < 0.06, corr


# ======================================= GPU: the replay sampler =========================================================

_RING_CASES = {  # capacity, obs_dim, act_dim, transitions per push, batch
    "partial_od17": (1000, 17, 3, [300, 123], 8193),
    "wrapped_head400_od33": (1000, 33, 3, [700, 700], 7),
    "full_head0": (512, 10, 2, [256, 256], 8193),
    "size1_cap1": (1, 17, 3, [1], 8193),
    "size1_cap7": (7, 33, 3, [1], 7),
    "batch1_wrapped": (999, 17, 3, [600, 600, 600], 1),
}


@gpu
@pytest.mark.parametrize("case", sorted(_RING_CASES))
def test_replay_sample_matches_the_restatement(case):
    """Slots equal to restated_slots for both laws, keyed on draw + appends (meta[3]), gathered rows equal to the ring's
    rows; draws continue across appends and past 2^32."""
    import gym_uav_collision_avoidance_b200 as G

    cap, od, ad, pushes, batch = _RING_CASES[case]
    seed = 0x1234567 + cap
    rb = G.DeviceReplay(cap, od, ad, seed=seed)
    g = torch.Generator(device="cuda").manual_seed(cap + od)

    def push(m):
        rb.push(torch.rand((m, od), generator=g, device="cuda"), torch.rand((m, ad), generator=g, device="cuda"),
                torch.rand(m, generator=g, device="cuda"), torch.rand((m, od), generator=g, device="cuda"),
                (torch.rand(m, generator=g, device="cuda") < 0.2).to(torch.uint8))

    for m in pushes:
        push(m)
    for step in range(3):
        if step == 2:
            push(pushes[-1])
            rb._draws += 2 ** 32  # the draw counter's high word
        for recency in (False, True):
            head, _, size, appends = (int(v) for v in rb.meta.tolist())
            draw = rb._draws
            s, a, r, n, m, idx = rb.sample_fused(batch, recency_weighted=recency, want_index=True)
            want = restated_slots(rb._sample_seed, draw + appends, batch, head, size, cap, recency)
            assert np.array_equal(idx.cpu().numpy(), want), (case, step, recency)
            w = torch.from_numpy(want).cuda()
            assert torch.equal(s, rb.state[w]) and torch.equal(a, rb.action[w]) and torch.equal(n, rb.next_state[w])
            assert torch.equal(r, rb.reward[w]) and torch.equal(m, rb.mask[w])


@gpu
def test_replay_sample_on_an_empty_ring_returns_slot_0():
    import gym_uav_collision_avoidance_b200 as G

    rb = G.DeviceReplay(100, 17, 3, seed=1)
    for recency in (False, True):
        s, a, r, n, m, idx = rb.sample_fused(1000, recency_weighted=recency, want_index=True)
        assert bool((idx == 0).all()) and not bool(s.any()) and not bool(a.any()) and not bool(n.any())
        assert not bool(r.any()) and not bool(m.any())
