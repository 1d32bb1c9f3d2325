"""Batched acting path around the env step ("next" rows of SURVEY.md §8f): one policy forward over all B*N UAVs,
the polar action map fused into the step kernel, transitions appended to the device replay ring — nothing leaves
the GPU between `obs` and the next `obs`.

The reference acts one UAV at a time: `SAC.select_action` copies a (10,) observation to the GPU, samples, copies the
action back (pytorch_sac_temp/sac.py:38-44), N times per env step (test_sac_multi.py:69-80), then maps the action
to cartesian on the host (:77-80) and pushes N tuples into a Python list (:101-103).  All UAVs share one policy
(:90-91), so the batched equivalent is a single [B*N, 10] forward.  The networks are stock PyTorch (cuBLAS): dense
MLPs are the learner's side of the boundary, not part of the hot path this package accelerates.
"""
from __future__ import annotations

import math
from typing import Optional

import torch
import torch.nn as nn
import torch.nn.functional as F

from .replay import DeviceReplay

LOG_SIG_MAX, LOG_SIG_MIN, EPS = 2, -20, 1e-6  # pytorch_sac_temp/model.py:6-8


class GaussianPolicy(nn.Module):
    """Same architecture and sampling semantics as the reference policy (pytorch_sac_temp/model.py:64-101):
    10 -> 256 -> 256 -> (mean, log_std), tanh-squashed Gaussian.  Random-init here (the reference ships no weights);
    `load_state_dict` accepts a reference checkpoint's `policy_state_dict` (same parameter names)."""

    def __init__(self, num_inputs=10, num_actions=2, hidden=256):
        super().__init__()
        self.linear1 = nn.Linear(num_inputs, hidden)
        self.linear2 = nn.Linear(hidden, hidden)
        self.mean_linear = nn.Linear(hidden, num_actions)
        self.log_std_linear = nn.Linear(hidden, num_actions)
        for m in self.modules():  # weights_init_ (model.py:11-14)
            if isinstance(m, nn.Linear):
                nn.init.xavier_uniform_(m.weight, gain=1)
                nn.init.constant_(m.bias, 0)

    def forward(self, state):
        x = F.relu(self.linear1(state))
        x = F.relu(self.linear2(x))
        return self.mean_linear(x), torch.clamp(self.log_std_linear(x), min=LOG_SIG_MIN, max=LOG_SIG_MAX)

    def sample(self, state):
        """-> (action, log_prob, eval_action) as model.py:86-101.  Note the reference's third output is
        tanh(normal.sample()), not tanh(mean) (kept as is)."""
        mean, log_std = self.forward(state)
        std = log_std.exp()
        x_t = mean + std * torch.randn_like(mean)
        y_t = torch.tanh(x_t)
        log_prob = -((x_t - mean) ** 2) / (2 * std * std) - log_std - 0.5 * math.log(2 * math.pi)
        log_prob = (log_prob - torch.log(1 - y_t.pow(2) + EPS)).sum(1, keepdim=True)
        return y_t, log_prob, torch.tanh(mean + std * torch.randn_like(mean))

    @torch.no_grad()
    def act(self, state, evaluate=False):
        """Acting only (SAC.select_action, pytorch_sac_temp/sac.py:38-44): tanh(mean + std * eps) — in the reference both
        the training action and the `evaluate=True` action are samples (model.py:90,101), so one code path serves both;
        the log-probability is not needed to act and is not computed."""
        mean, log_std = self.forward(state)
        return torch.tanh(torch.addcmul(mean, log_std.exp(), torch.randn_like(mean)))


class FusedGaussianPolicy:
    """The acting path of a `GaussianPolicy` (10 -> 256 -> 256 -> 2+2) as ONE tcgen05 kernel (`uavca_policy_act`,
    csrc/uavca_policy.cu): both hidden layers on the tensor cores with the activations kept in shared memory / TMEM,
    output heads, tanh-Gaussian sampling (Philox noise) fused.  Operands are fp16 with fp32 accumulation.  Weights are
    packed once from the module; call `refresh()` after the learner updated it (test_sac_multi.py:85-91).  A TD3-style
    deterministic actor (attributes l1, l2, l3: pytorch_td3_temp/td3.py:14-27) is accepted too: action = tanh(l3(...))."""

    def __init__(self, policy: nn.Module, seed: int = 0):
        self.policy = policy
        self.seed = int(seed)
        self.calls = 0  # host-side offset of the Philox counter (set it to replay a draw)
        self.refresh()
        # device-side call counter: advanced by a one-element kernel after every act(), so a CUDA-graph replay of the
        # acting step draws fresh noise each time
        self.counter = torch.zeros(1, dtype=torch.int64, device=self.w2.device)
        self.own_counter = True  # False: somebody else advances `counter` once per step (the replay ring's append counter)

    @torch.no_grad()
    def refresh(self):
        """Re-pack the weights after the learner updated the policy.  The packed operands are rewritten in place, so an
        acting step captured in a CUDA graph before the update acts with the new weights when replayed."""
        packed = self._pack()
        if not hasattr(self, "w1"):
            for name, t in packed.items():
                setattr(self, name, t)
            return
        for name, t in packed.items():
            dst = getattr(self, name)
            if dst.device != t.device:
                raise ValueError("the policy moved to another device: build a new FusedGaussianPolicy")
            dst.copy_(t)

    def _pack(self) -> dict:
        p = self.policy
        if hasattr(p, "l1") and hasattr(p, "l3"):
            # deterministic TD3-style actor (pytorch_td3_temp/td3.py:14-27: l1, l2, l3, tanh): the same kernel with the
            # log_std head pinned at its floor (std = e^-20, the sampled term vanishes below fp32 resolution)
            lin1, lin2, mean_w, mean_b = p.l1, p.l2, p.l3.weight, p.l3.bias
            std_w, std_b = torch.zeros_like(mean_w), torch.full_like(mean_b, -20.0)
        else:
            lin1, lin2, mean_w, mean_b = p.linear1, p.linear2, p.mean_linear.weight, p.mean_linear.bias
            std_w, std_b = p.log_std_linear.weight, p.log_std_linear.bias
        w1, w2 = lin1.weight, lin2.weight
        if tuple(w1.shape) != (256, 10) or tuple(w2.shape) != (256, 256) or mean_w.shape[0] != 2:
            raise ValueError("the fused acting kernel is built for the reference architecture 10 -> 256 -> 256 -> 2")
        if not w1.is_cuda:
            raise ValueError("the policy must live on a CUDA device")
        dev, h = w1.device, torch.float16
        # fp16 K-major operands; every bias rides in an extra input column (include/uavca.h)
        w1p = torch.zeros((256, 16), dtype=h, device=dev)
        w1p[:, :10] = w1.to(h)
        w1p[:, 10] = lin1.bias.to(h)
        w2b = torch.zeros((256, 16), dtype=h, device=dev)
        w2b[:, 0] = lin2.bias.to(h)
        w3 = torch.zeros((16, 256), dtype=h, device=dev)
        w3[0:2] = mean_w.to(h)
        w3[2:4] = std_w.to(h)
        w3b = torch.zeros((16, 16), dtype=h, device=dev)
        w3b[0:2, 0] = mean_b.to(h)
        w3b[2:4, 0] = std_b.to(h)
        return dict(w1=w1p, w2=w2.to(h).contiguous(), w2b=w2b, w3=w3, w3b=w3b)

    def act(self, state: torch.Tensor, evaluate: bool = False, out: Optional[torch.Tensor] = None,
            noise: Optional[torch.Tensor] = None, head: Optional[torch.Tensor] = None) -> torch.Tensor:
        """state [M, 10] float32 CUDA -> action [M, 2] in (-1, 1).  `noise` [M, 2] overrides the Philox draws (tests);
        `head` [M, 4] receives (mean, log_std).  Every tensor must be float32 on the policy's device; anything else
        raises ValueError before the kernel is launched (the kernel reads and writes raw float32 rows)."""
        from . import ops

        dev = self.w2.device
        if state.dtype != torch.float32 or state.device != dev:
            raise ValueError(f"state must be float32 on {dev}, got {state.dtype} on {state.device}")
        if state.numel() % 10:
            raise ValueError(f"state holds {state.numel()} values, not a whole number of 10-feature observations")
        state = state.contiguous()
        M = state.numel() // 10
        for name, t, width in (("out", out, 2), ("noise", noise, 2), ("head", head, 4)):
            if t is None:
                continue
            if t.dtype != torch.float32 or t.device != dev or tuple(t.shape) != (M, width) or not t.is_contiguous():
                raise ValueError(f"{name} must be a contiguous float32 [{M}, {width}] tensor on {dev}, "
                                 f"got {t.dtype} {tuple(t.shape)} on {t.device}")
        if out is None:
            out = torch.empty((M, 2), dtype=torch.float32, device=state.device)
        ops.policy_act(state, self.w1, self.w2, self.w2b, self.w3, self.w3b, noise, self.seed, self.calls, self.counter,
                       out, head)
        if self.own_counter:
            self.counter += 1
        return out


class BatchedRollout:
    """obs -> policy -> step(action_mode) -> replay, all on the device; optionally replayed from a CUDA graph (capture an
    EVEN number of steps: the env alternates between two observation buffers, so that the observation an action was taken
    on survives the step without a copy)."""

    def __init__(self, env, policy: Optional[nn.Module] = None, replay: Optional[DeviceReplay] = None,
                 action_mode="polar", evaluate=False, warmup_uniform=False, precision="fp32", fused_append=True):
        """precision of the policy forward: "fp32" (the reference's arithmetic: PyTorch default, TF32 off), "tf32"
        (tensor-core GEMMs on fp32 storage), "bf16" (autocast) or "fused" (the one-kernel tcgen05 acting path,
        `FusedGaussianPolicy`).  The env step itself is unaffected."""
        if precision not in ("fp32", "tf32", "bf16", "fused"):
            raise ValueError("precision must be fp32, tf32, bf16 or fused")
        self.precision = precision
        self.fused = FusedGaussianPolicy(policy) if precision == "fused" else None
        self.env, self.policy, self.replay = env, policy, replay
        self.action_mode, self.evaluate, self.warmup_uniform = action_mode, evaluate, warmup_uniform
        B, N, D = env.num_envs, env.num_agents, env.obs_dim
        # the observation the action was taken on: env.obs of the previous step.  The env ping-pongs between two
        # observation buffers (`set_obs_buffer`), so nothing is copied.
        self.state = env.obs
        self._spare = torch.zeros((B, N, D), dtype=torch.float32, device=env.device)
        self.action = torch.zeros((B, N, 2), dtype=torch.float32, device=env.device)
        # step + replay append as ONE launch where the env has it (multi world on the warp kernels): no separate pass over
        # the transitions, no final_obs buffer
        self.fused_append = bool(replay is not None and fused_append and replay.capacity * 10 < 2 ** 31 and
                                 getattr(env, "supports_step_replay", lambda: False)())
        if replay is not None:
            if not self.fused_append:
                env.enable_final_obs()
            if self.fused is not None:
                # the ring's append counter advances once per acting step on the device: the policy's Philox noise is
                # keyed on it, so no separate counter kernel runs (and CUDA-graph replays still draw fresh noise)
                self.fused.counter = replay.meta[3:4]
                self.fused.own_counter = False
        self._graph = None
        self.steps = 0

    def reset(self):
        self.env.reset()
        return self.env.obs

    def _act(self):
        env = self.env
        self.state = env.obs  # acted on now, overwritten only by the step after next
        if self.policy is None or self.warmup_uniform:  # test_sac_multi.py:72-73: uniform actions during warm-up
            self.action.uniform_(-1.0, 1.0)
        else:
            x = self.state.view(-1, env.obs_dim)
            if self.precision == "fused":
                self.fused.act(x, evaluate=self.evaluate, out=self.action.view(-1, 2))
                return
            if self.precision == "bf16":
                with torch.autocast("cuda", dtype=torch.bfloat16):
                    a = self.policy.act(x, evaluate=self.evaluate)
            elif self.precision == "tf32":
                prev = torch.backends.cuda.matmul.allow_tf32
                torch.backends.cuda.matmul.allow_tf32 = True
                try:
                    a = self.policy.act(x, evaluate=self.evaluate)
                finally:
                    torch.backends.cuda.matmul.allow_tf32 = prev
            else:
                a = self.policy.act(x, evaluate=self.evaluate)
            self.action.copy_(a.view_as(self.action))

    def _env_step(self):
        env = self.env
        nxt, self._spare = self._spare, env.obs  # the step writes its observation into the other buffer
        env.set_obs_buffer(nxt)
        if self.fused_append:
            # next_state = the step's own observation (before any auto-reset), mask = float(not done): test_sac_multi.py:101-103
            env.step_replay(self.action, self.state, self.replay, evaluate=self.evaluate, action_mode=self.action_mode)
        elif env.num_agents == 1 and env.obs_dim == 4:
            env.step(self.action, action_mode=self.action_mode)
        else:
            env.step(self.action, evaluate=self.evaluate, action_mode=self.action_mode)

    def step(self):
        self._act()
        self._env_step()
        if self.replay is not None and not self.fused_append:
            # next_state = the step's own observation (before any auto-reset), mask = float(not done): test_sac_multi.py:101-103
            self.replay.push(self.state, self.action, self.env.reward, self.env.final_obs, self.env.done)
        self.steps += 1

    def run(self, steps: int):
        for _ in range(steps):
            self.step()

    def success_collision_rates(self):
        """SR / CR over the finished episodes (test_sac_multi.py:164-179): counts / (N * episodes)."""
        s = self.env.stats()
        denom = max(1, s["episodes"]) * self.env.num_agents
        return s["reach"] / denom, s["collisions"] / denom, s["episodes"]

    def evaluation_summary(self) -> dict:
        """The numbers the reference's evaluation block prints (test_sac_multi.py:164-176) over the finished episodes:
        SR = reach / (N * episodes), CR = collisions / (N * episodes), Avg_Score = sum_i rewards[i] * (1 - dones[i])
        / (N * episodes), plus the mean per-episode `score` (sum of rewards[0], :105).  The scores need an env built
        with track_scores=True."""
        s = self.env.stats()
        eps = max(1, s["episodes"])
        denom = eps * self.env.num_agents
        return dict(episodes=s["episodes"], SR=s["reach"] / denom, CR=s["collisions"] / denom,
                    Avg_Score=s["score_live_sum"] / denom, mean_episode_score=s["score0_sum"] / eps,
                    nonfinite=s["nonfinite"])
