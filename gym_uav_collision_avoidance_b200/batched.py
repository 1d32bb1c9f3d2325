"""Batched, device-resident versions of the reference worlds.

`BatchedMultiUAVWorld2D` / `BatchedUAVWorld2D` keep the reference's reset()/step() contract
(multi_uav_world_2d.py:116,177; uav_world_2d.py:119,137) over B independent environments held in one
structure-of-arrays state blob in HBM.  All inputs and outputs are CUDA tensors; the step is one kernel launch.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional

import numpy as np
import torch

from . import _capi, ops
from .replay import PrioritizedDeviceReplay
from ._capi import (ACTION_CARTESIAN, ACTION_POLAR, ACTION_SCALED, KIND_MULTI, KIND_SINGLE, RESET_ON_ALL_DONE,  # noqa: F401
                    RESET_ON_ANY_DONE, RESET_ON_DONE0, SOURCE_PHILOX, SOURCE_POOL)

_ACTION_MODES = {"cartesian": ACTION_CARTESIAN, "polar": ACTION_POLAR, "scaled": ACTION_SCALED,
                 ACTION_CARTESIAN: ACTION_CARTESIAN, ACTION_POLAR: ACTION_POLAR, ACTION_SCALED: ACTION_SCALED}

_FIELD_DTYPES = dict(pos=(torch.float32, 2), vel=(torch.float64, 2), tgt=(torch.float32, 2), init=(torch.float32, 0),
                     prev=(torch.float32, 0), flags=(torch.uint8, 0))
_ENV_FIELDS = dict(steps=torch.int32, reach=torch.int32, coll=torch.int32, episode=torch.int32)


class Box:
    """Record standing in for gym.spaces.Box (low/high/shape/dtype/sample), so callers that read
    `env.action_space.high` or `observation_space.shape[0]` (test_sac_multi.py:39-40,77) keep working without gym."""

    def __init__(self, low, high, shape, dtype=np.float32):
        self.dtype = np.dtype(dtype)
        self.shape = tuple(shape)
        self.low = np.broadcast_to(np.asarray(low, dtype=self.dtype), self.shape).copy()
        self.high = np.broadcast_to(np.asarray(high, dtype=self.dtype), self.shape).copy()

    def sample(self):
        return np.random.uniform(self.low, self.high, size=self.shape).astype(self.dtype)

    def __repr__(self):
        return f"Box({self.low}, {self.high}, {self.shape}, {self.dtype})"


class StateBlob:
    """One SoA state blob (uint8 CUDA tensor) with typed tensor views of its fields (zero-copy)."""

    def __init__(self, layout: _capi.Layout, num_envs: int, num_agents: int, device: torch.device):
        self.B, self.N = num_envs, num_agents
        self.layout = layout
        self.blob = torch.zeros(layout.total_bytes, dtype=torch.uint8, device=device)
        M = num_envs * num_agents
        for name, (dt, inner) in _FIELD_DTYPES.items():
            nbytes = M * max(inner, 1) * torch.empty((), dtype=dt).element_size()
            off = getattr(layout, name)
            shape = (num_envs, num_agents, inner) if inner else (num_envs, num_agents)
            setattr(self, name, self.blob[off:off + nbytes].view(dt).view(shape))
        for name, dt in _ENV_FIELDS.items():
            off = getattr(layout, name)
            setattr(self, name, self.blob[off:off + num_envs * 4].view(dt))
        self.stats = self.blob[layout.stats:layout.stats + 64].view(torch.int64)
        self.stats_f64 = self.blob[layout.stats:layout.stats + 64].view(torch.float64)  # slots 4, 5: score sums
        self.score = self.blob[layout.score:layout.score + num_envs * 16].view(torch.float64).view(num_envs, 2)
        self.float64_world = layout.tgt64 != layout.pos64  # config.circular: float64 locations, as the reference keeps them
        if self.float64_world:
            f64 = lambda off, inner: self.blob[off:off + M * max(inner, 1) * 8].view(torch.float64).view(  # noqa: E731
                (num_envs, num_agents, inner) if inner else (num_envs, num_agents))
            self.pos64, self.tgt64 = f64(layout.pos64, 2), f64(layout.tgt64, 2)
            self.init64, self.prev64 = f64(layout.init64, 0), f64(layout.prev64, 0)
            self.init64.fill_(1.0)
            self.prev64.fill_(1.0)
        self.init.fill_(1.0)
        self.prev.fill_(1.0)

    FIELDS = ("pos", "vel", "tgt", "init", "prev", "flags", "steps", "reach", "coll", "episode", "score")

    def load_arrays(self, **arrays) -> None:
        """Overwrite fields from host arrays / tensors of the matching shape (parity runs, checkpoints)."""
        for k, v in arrays.items():
            dst = getattr(self, k)
            src = torch.as_tensor(np.ascontiguousarray(v) if isinstance(v, np.ndarray) else v)
            if k == "episode" and src.dtype != torch.int32:
                src = src.to(torch.int64).to(torch.int32)
            dst.copy_(src.to(dst.dtype).reshape(dst.shape), non_blocking=False)

    def to_host(self) -> dict:
        out = {k: getattr(self, k).cpu().numpy() for k in self.FIELDS}
        if self.float64_world:
            out.update({k: getattr(self, k).cpu().numpy() for k in ("pos64", "tgt64", "init64", "prev64")})
        out["stats"] = self.stats.cpu().numpy()
        return out


class _BatchedBase:
    kind: int = KIND_MULTI
    # step() reaches the C-ABI either through the registered PyTorch custom ops (`ops.py`: what torch.compile traces,
    # ~27 us of Python dispatch per call) or, in plain eager code, by calling the same entry point directly
    # (~8 us per call).  Set to True to force the custom-op route everywhere.
    use_custom_ops: bool = False

    def __init__(self, num_envs: int, num_agents: int, cfg: _capi.Config, device=None):
        if not torch.cuda.is_available():
            raise _capi.UavcaError("gym_uav_collision_avoidance_b200 needs a CUDA device (B200, sm_100a); "
                                   "there is no CPU fallback")
        self.device = torch.device(device if device is not None else f"cuda:{torch.cuda.current_device()}")
        if self.device.type != "cuda":
            raise _capi.UavcaError("device must be a CUDA device")
        self._lib = _capi.load()
        self.cfg = cfg
        self.num_envs, self.num_agents = num_envs, num_agents
        self.obs_dim = _capi.OBS_DIM[cfg.kind]
        h = C.c_void_p()
        _capi.check(self._lib.uavca_create(C.byref(cfg), self.device.index or 0, C.byref(h)), "uavca_create")
        self._h = h.value
        lay = _capi.Layout()
        _capi.check(self._lib.uavca_state_layout(self._h, C.byref(lay)), "uavca_state_layout")
        self.state = StateBlob(lay, num_envs, num_agents, self.device)
        self._pool: Optional[StateBlob] = None
        B, N, D = num_envs, num_agents, self.obs_dim
        self.obs = torch.zeros((B, N, D), dtype=torch.float32, device=self.device)
        self.reward = torch.zeros((B, N), dtype=torch.float32, device=self.device)
        self.done = torch.zeros((B, N), dtype=torch.uint8, device=self.device)
        self.final_obs: Optional[torch.Tensor] = None
        self.reset_mask = torch.zeros(B, dtype=torch.uint8, device=self.device)
        self._stats = torch.zeros(8, dtype=torch.int64, device=self.device)
        self._ptrs = (self.state.blob.data_ptr(), self.obs.data_ptr(), self.reward.data_ptr(), self.done.data_ptr(),
                      self.reset_mask.data_ptr())

    def _direct(self) -> bool:
        return not (self.use_custom_ops or torch.compiler.is_compiling())

    def _stream(self) -> int:
        return torch.cuda.current_stream(self.device).cuda_stream

    # -- lifetime -----------------------------------------------------------------------------------------------
    def close(self):
        if getattr(self, "_h", None):
            self._lib.uavca_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # -- checkpointing ---------------------------------------------------------------------------------------------
    def state_dict(self) -> dict:
        """Everything needed to resume bit-identically: the SoA state blob (positions, velocities, targets, latches,
        counters, Philox episode counters, running totals) and the constructor configuration.  The reference never
        checkpoints its environments (SURVEY.md 5); with counter-based RNG the blob IS the whole state."""
        cfg = {name: getattr(self.cfg, name) for name, _ in self.cfg._fields_}
        return {"config": cfg, "blob": self.state.blob.cpu().clone(), "obs": self.obs.cpu().clone()}

    def load_state_dict(self, sd: dict) -> None:
        for k, v in sd["config"].items():
            if k != "env_index_base" and getattr(self.cfg, k) != v:
                raise ValueError(f"checkpoint was taken with {k}={v}, this env has {getattr(self.cfg, k)}")
        if sd["blob"].numel() != self.state.blob.numel():
            raise ValueError("checkpoint holds a different number of environments / agents")
        self.state.blob.copy_(sd["blob"])
        self.obs.copy_(sd["obs"])

    # -- reset pool (host-supplied reset states) -----------------------------------------------------------------
    def make_pool(self, pool_envs: int) -> StateBlob:
        lay = _capi.Layout()
        _capi.check(self._lib.uavca_pool_layout(self._h, pool_envs, C.byref(lay)), "uavca_pool_layout")
        pool = StateBlob(lay, pool_envs, self.num_agents, self.device)
        self._pool = pool
        _capi.check(self._lib.uavca_set_reset_pool(self._h, pool.blob.data_ptr(), pool_envs), "uavca_set_reset_pool")
        return pool

    # -- gym-shaped API --------------------------------------------------------------------------------------------
    def set_obs_buffer(self, obs: torch.Tensor) -> None:
        """Make `obs` ([B, N, D] float32 CUDA, contiguous) the tensor the next step / reset writes its observation into
        (`env.obs` afterwards).  Lets a caller ping-pong two buffers instead of copying the observation it acted on."""
        if obs.shape != self.obs.shape or obs.dtype != torch.float32 or obs.device != self.device or not obs.is_contiguous():
            raise ValueError("set_obs_buffer needs a contiguous float32 CUDA tensor shaped like env.obs")
        self.obs = obs
        self._ptrs = (self.state.blob.data_ptr(), self.obs.data_ptr(), self.reward.data_ptr(), self.done.data_ptr(),
                      self.reset_mask.data_ptr())

    def enable_final_obs(self, on: bool = True):
        """Also emit the step's own next-observation before any auto-reset (what a replay buffer stores)."""
        self.final_obs = torch.zeros_like(self.obs) if on else None

    def reset(self, mask: Optional[torch.Tensor] = None) -> torch.Tensor:
        if mask is not None:
            mask = mask.to(device=self.device, dtype=torch.uint8).contiguous()
        ops.reset(self._h, self.state.blob, mask, self.obs)
        return self.obs

    def observe(self) -> torch.Tensor:
        ops.observe(self._h, self.state.blob, self.obs)
        return self.obs

    def map_action(self, action: torch.Tensor, action_mode="polar") -> torch.Tensor:
        out = torch.empty_like(action)
        ops.map_action(self._h, action.contiguous(), _ACTION_MODES[action_mode], out)
        return out

    def stats(self) -> dict:
        """Totals over finished episodes plus the counters of the episodes in flight."""
        ops.stats(self._h, self.state.blob, self._stats)
        v = self._stats.cpu().tolist()
        sf = self.state.stats_f64[4:6].cpu().tolist()
        return dict(episodes=v[0], reach=v[1], collisions=v[2], steps=v[3], live_reach=v[4], live_collisions=v[5],
                    live_steps=v[6], num_envs=v[7],
                    # over finished episodes, with track_scores=True: sum of rewards[0] (test_sac_multi.py:105) and of
                    # rewards[i] * (1 - dones[i]) over all UAVs (:152-156); UAV-steps whose reward / position was not finite
                    score0_sum=sf[0], score_live_sum=sf[1], nonfinite=int(self.state.stats[6].item()))

    # the counters the reference keeps on the env object (multi_uav_world_2d.py:166-168), one value per env
    @property
    def steps(self) -> torch.Tensor:
        return self.state.steps

    @property
    def target_reach_count(self) -> torch.Tensor:
        return self.state.reach

    @property
    def collision_count(self) -> torch.Tensor:
        return self.state.coll

    @property
    def score(self) -> torch.Tensor:
        """[B, 2] float64, the episode in flight (needs track_scores=True): column 0 the running `score += rewards[0]`
        of the training loops (test_sac_multi.py:105, test_sac_multi_score.py:54), column 1 the running
        `total_score += rewards[i] * (1 - dones[i])` of the evaluation loop (test_sac_multi.py:152-156)."""
        return self.state.score

    def export_trajectory(self, env_slice, steps: int, actions=None, policy=None, action_mode="cartesian",
                          evaluate: bool = False) -> dict:
        """Host-side trajectory of a slice of the envs — what the reference draws with pygame (`render()`,
        multi_uav_world_2d.py:243-331) or collects by hand for plotting (test_sac_multi_plot_trajectory.py:46-68:
        every UAV's `location` per step, the targets, and the step at which it was done).

        Steps ALL envs `steps` times (actions: a [steps, B, N, 2] tensor, a callable `policy(obs) -> action`, or None
        for the Philox random stream) and returns NumPy arrays for `env_slice` (an int, slice or index tensor):
        pos [steps+1, E, N, 2] (row 0 = before the first step), target [steps+1, E, N, 2], velocity [steps+1, E, N, 2],
        done / reward [steps, E, N], reset [steps, E] (an auto-reset happened: the trajectory jumps), parked / collided
        [steps+1, E, N] and `done_step` [E, N] (first step each UAV reported done, -1 if never)."""
        import numpy as np

        idx = torch.arange(self.num_envs, device=self.device)[env_slice].reshape(-1)
        st = self.state
        rec = dict(pos=[st.pos[idx].cpu()], target=[st.tgt[idx].cpu()], velocity=[st.vel[idx].cpu()], flags=[st.flags[idx].cpu()],
                   done=[], reward=[], reset=[])
        for k in range(int(steps)):
            if actions is not None:
                a = actions[k]
            elif policy is not None:
                a = policy(self.obs)
            else:
                a = self.sample_actions(k)
                if action_mode == "cartesian":
                    a = a * float(self.max_speed[0])
            if self.kind == KIND_SINGLE:
                _, r, d, info = self.step(a, action_mode=action_mode)
            else:
                _, r, d, info = self.step(a, evaluate=evaluate, action_mode=action_mode)
            rec["pos"].append(st.pos[idx].cpu()); rec["target"].append(st.tgt[idx].cpu())
            rec["velocity"].append(st.vel[idx].cpu()); rec["flags"].append(st.flags[idx].cpu())
            rec["done"].append(d[idx].cpu()); rec["reward"].append(r[idx].cpu()); rec["reset"].append(info["reset_mask"][idx].cpu())
        out = {k: torch.stack(v).numpy() for k, v in rec.items()}
        flags = out.pop("flags")
        out["parked"], out["collided"] = (flags & 1).astype(bool), (flags & 2).astype(bool)
        done = out["done"].astype(bool)
        out["done"] = done
        out["reset"] = out["reset"].astype(bool)
        first = np.where(done.any(axis=0), done.argmax(axis=0), -1)
        out["done_step"] = first
        out["env_index"] = idx.cpu().numpy()
        return out

    @property
    def launch_count(self) -> int:
        return int(self._lib.uavca_launch_count(self._h))

    def _check_action(self, action: torch.Tensor) -> torch.Tensor:
        B, N = self.num_envs, self.num_agents
        if action.device != self.device or action.dtype != torch.float32:
            action = action.to(device=self.device, dtype=torch.float32)
        if action.numel() != B * N * 2:
            raise ValueError(f"action must hold {B}x{N}x2 values, got shape {tuple(action.shape)}")
        action = action.contiguous()
        if action.data_ptr() % 16:  # a view into a larger buffer: the kernels read float2 / 16-byte units
            action = action.clone()
        return action

    def step_f64(self, action: torch.Tensor, evaluate: bool = False):
        """`step()` fed FLOAT64 cartesian actions ([B,N,2] float64 CUDA; [B,2] / [B,1,2] for the single world) — what the
        reference's own loops build on the host (test_sac_multi.py:77-80) and `UAVAgent.step` consumes in float64
        (uav_agent.py:26).  Bit-exact for actions float32 cannot hold; same kernels as `step()` (`compat.py` uses it for
        python floats / float64 arrays)."""
        B, N = self.num_envs, self.num_agents
        action = action.to(device=self.device, dtype=torch.float64).contiguous()
        if action.numel() != B * N * 2:
            raise ValueError(f"action must hold {B}x{N}x2 values, got shape {tuple(action.shape)}")
        if action.data_ptr() % 16:
            action = action.clone()
        dist = getattr(self, "distance", None)
        _capi.check(self._lib.uavca_step_f64(self._h, self.state.blob.data_ptr(), action.data_ptr(), int(bool(evaluate)),
                                             self.obs.data_ptr(), self.reward.data_ptr(), self.done.data_ptr(),
                                             None if dist is None else dist.data_ptr(),
                                             None if self.final_obs is None else self.final_obs.data_ptr(),
                                             self.reset_mask.data_ptr(), self._stream()), "uavca_step_f64")
        info = {"distance": dist if dist is not None else 0, "reset_mask": self.reset_mask}
        if self.final_obs is not None:
            info["final_obs"] = self.final_obs
        return self.obs, self.reward, self.done, info

    def step_host(self, action: torch.Tensor, obs: torch.Tensor, reward: torch.Tensor, done: torch.Tensor,
                  action_mode="cartesian", evaluate: bool = False):
        """End-to-end step with HOST tensors (pinned for speed): H2D actions, step, D2H obs/reward/done."""
        for t in (action, obs, reward, done):
            if t.is_cuda or not t.is_contiguous():
                raise ValueError("step_host takes contiguous CPU tensors")
        _capi.check(self._lib.uavca_step_host(self._h, self.state.blob.data_ptr(), action.data_ptr(),
                                              _ACTION_MODES[action_mode], int(evaluate), obs.data_ptr(),
                                              reward.data_ptr(), done.data_ptr(), self._stream()), "uavca_step_host")
        return obs, reward, done

    # -- K steps per launch ------------------------------------------------------------------------------------------
    def sample_actions(self, step: int, action_seed: int = 0, out: Optional[torch.Tensor] = None) -> torch.Tensor:
        """The policy-space actions in [-1, 1)^2 that `rollout(actions=None)` draws at global step `step`
        (`env.action_space.sample()` for every UAV, as a counter-based Philox stream)."""
        if out is None:
            out = torch.empty((self.num_envs, self.num_agents, 2), dtype=torch.float32, device=self.device)
        ops.sample_actions(self._h, int(action_seed), int(step), out)
        return out

    def rollout(self, steps: int, actions: Optional[torch.Tensor] = None, action_mode="cartesian", evaluate: bool = False,
                action_seed: int = 0, step0: int = 0, out: Optional[dict] = None, want_actions: bool = False,
                want_final_obs: bool = False, want_reset_mask: bool = False, sync_last: bool = True) -> dict:
        """`steps` consecutive env steps in ONE kernel launch — the reference's random-action driver loops
        (run.py:10-16, run_multi.py:10-16: `env.step(env.action_space.sample())`, reset on done) or an open-loop
        action block.  The env state stays in registers between the steps; only the per-step outputs stream out.

        actions: [K, B, N, 2] float32 CUDA tensor in `action_mode`, or None: every UAV then draws uniform actions from
        the Philox stream keyed by (action_seed, global env index, UAV, step0 + k); `action_mode="cartesian"` then spans
        the whole action box (a * max_speed).  Returns a dict of [K, ...] tensors: obs, reward, done (+ actions,
        final_obs, reset_mask, distance on request).  Pass the dict back as `out=` to reuse the buffers (CUDA graphs).
        `self.obs` / `self.reward` / `self.done` receive the last step (`sync_last`).  Bit-identical to `steps` calls of
        `step()` fed the same actions."""
        K, B, N, D = int(steps), self.num_envs, self.num_agents, self.obs_dim
        if K < 1:
            raise ValueError("rollout needs steps >= 1")
        if actions is not None:
            if actions.device != self.device or actions.dtype != torch.float32:
                actions = actions.to(device=self.device, dtype=torch.float32)
            if actions.numel() != K * B * N * 2:
                raise ValueError(f"actions must hold {K}x{B}x{N}x2 values, got shape {tuple(actions.shape)}")
            actions = actions.contiguous()
        if out is None:
            kw = dict(device=self.device)
            out = dict(obs=torch.empty((K, B, N, D), dtype=torch.float32, **kw),
                       reward=torch.empty((K, B, N), dtype=torch.float32, **kw),
                       done=torch.empty((K, B, N), dtype=torch.uint8, **kw))
            if want_actions and actions is None:
                out["actions"] = torch.empty((K, B, N, 2), dtype=torch.float32, **kw)
            if want_final_obs:
                out["final_obs"] = torch.empty((K, B, N, D), dtype=torch.float32, **kw)
            if want_reset_mask:
                out["reset_mask"] = torch.empty((K, B), dtype=torch.uint8, **kw)
            if self.kind == KIND_SINGLE:
                out["distance"] = torch.empty((K, B), dtype=torch.float32, **kw)
        if out["obs"].shape[0] != K:
            raise ValueError("the `out` buffers were made for a different number of steps")
        act_out = out.get("actions") if actions is None else None
        if self._direct():  # plain eager code: the C-ABI entry point itself (the custom op below costs ~20 us more per call)
            p = lambda t: None if t is None else t.data_ptr()  # noqa: E731
            rc = self._lib.uavca_rollout(self._h, self.state.blob.data_ptr(), K, p(actions), _ACTION_MODES[action_mode],
                                         int(bool(evaluate)), int(action_seed), int(step0), out["obs"].data_ptr(),
                                         out["reward"].data_ptr(), out["done"].data_ptr(), p(act_out), p(out.get("final_obs")),
                                         p(out.get("reset_mask")), p(out.get("distance")), self._stream())
            if rc:
                _capi.check(rc, "uavca_rollout")
        else:
            ops.rollout(self._h, self.state.blob, K, actions, _ACTION_MODES[action_mode], bool(evaluate), int(action_seed),
                        int(step0), out["obs"], out["reward"], out["done"], act_out, out.get("final_obs"),
                        out.get("reset_mask"), out.get("distance"))
        if sync_last:  # keep the env object coherent: env.obs is what a policy acts on next
            self.obs.copy_(out["obs"][-1])
            self.reward.copy_(out["reward"][-1])
            self.done.copy_(out["done"][-1])
        return out


class BatchedMultiUAVWorld2D(_BatchedBase):
    """B x MultiUAVWorld2D (multi_uav_world_2d.py:10).  Constructor kwargs follow the reference (:13)."""

    kind = KIND_MULTI

    def __init__(self, num_envs: int, x_size=50.0, y_size=50.0, max_speed=10.0, max_acceleration=5.0, num_agents=4,
                 collider_radius=1.0, d_sense=15, *, device=None, seed=0, reset_mode=0, max_episode_steps=0,
                 reset_source=SOURCE_PHILOX, circular=False, env_index_base=0, hard_collision_radius=0.5,
                 track_scores=False):
        cfg = _capi.default_config(KIND_MULTI)
        cfg.track_scores = int(bool(track_scores))
        cfg.num_envs, cfg.num_agents = num_envs, num_agents
        cfg.x_size, cfg.y_size, cfg.max_speed, cfg.max_acceleration = x_size, y_size, max_speed, max_acceleration
        cfg.collider_radius, cfg.d_sense, cfg.hard_collision_radius = collider_radius, d_sense, hard_collision_radius
        cfg.seed, cfg.reset_mode, cfg.max_episode_steps = seed, reset_mode, max_episode_steps
        cfg.reset_source, cfg.circular, cfg.env_index_base = reset_source, int(circular), env_index_base
        # np.linalg.norm(env.action_space.high) with a float32 `high` (test_sac_multi.py:77)
        cfg.polar_scale = float(np.linalg.norm(np.full(2, max_speed, dtype=np.float32)))
        super().__init__(num_envs, num_agents, cfg, device)
        # attributes the reference exposes (multi_uav_world_2d.py:14-47; `max_acceleratoin` sic)
        self.x_size, self.y_size = x_size, y_size
        self.map_diagonal_size = np.linalg.norm([x_size, y_size])
        self.min_location = np.array([-x_size / 2.0, -y_size / 2.0])
        self.max_location = np.array([x_size / 2.0, y_size / 2.0])
        self.max_speed = np.array([max_speed, max_speed])
        self.min_speed = -self.max_speed
        self.max_acceleratoin = np.array([max_acceleration, max_acceleration])
        self.min_acceleratoin = -self.max_acceleratoin
        self.tau, self.collider_radius, self.d_sense = 0.02, collider_radius, d_sense
        self.observation_space = Box(np.array([0, -1, 0, -1, 0, -1, -1, 0, -1, 1]), np.ones(10), (10,))  # :44-45 (sic)
        self.action_space = Box(-max_speed, max_speed, (2,))  # :47

    def step(self, action: torch.Tensor, evaluate: bool = False, action_mode="cartesian"):
        """action [B,N,2] float32 CUDA -> (obs [B,N,10], reward [B,N], done [B,N] uint8, info)."""
        action = self._check_action(action)
        if self._direct():
            sp, op, rp, dp, mp = self._ptrs
            fp = None if self.final_obs is None else self.final_obs.data_ptr()
            rc = self._lib.uavca_step_multi(self._h, sp, action.data_ptr(), _ACTION_MODES[action_mode], int(bool(evaluate)),
                                            op, rp, dp, fp, mp, self._stream())
            if rc:
                _capi.check(rc, "uavca_step_multi")
        else:
            ops.step_multi(self._h, self.state.blob, action, _ACTION_MODES[action_mode], bool(evaluate), self.obs,
                           self.reward, self.done, self.final_obs, self.reset_mask)
        info = {"distance": 0, "reset_mask": self.reset_mask}  # multi_uav_world_2d.py:111-114
        if self.final_obs is not None:
            info["final_obs"] = self.final_obs
        return self.obs, self.reward, self.done, info


    def supports_step_replay(self) -> bool:
        """`step_replay` runs on the warp kernels: up to 32 UAVs per env, float32 world."""
        return self.num_agents <= 32 and not self.cfg.circular

    def step_replay(self, action: torch.Tensor, prev_obs: torch.Tensor, replay, evaluate: bool = False,
                    action_mode="cartesian"):
        """`step(action)` that also appends every UAV's transition (prev_obs, action, reward, next observation before any
        auto-reset, 1 - done) to `replay` (a `DeviceReplay`) in the SAME launch — env.step followed by the N
        `memory.push` calls of a training step (test_sac_multi.py:99-103).  `prev_obs` is the observation the action was
        taken on; it must not be the tensor this step writes (`env.obs`): ping-pong two buffers with `set_obs_buffer`.
        A `PrioritizedDeviceReplay` is synced after the launch (one more launch): the new slots take its largest priority."""
        action = self._check_action(action)
        if prev_obs.data_ptr() == self.obs.data_ptr():
            raise ValueError("prev_obs is the buffer this step writes its observation into (use set_obs_buffer)")
        if prev_obs.shape != self.obs.shape or prev_obs.dtype != torch.float32 or not prev_obs.is_contiguous():
            raise ValueError("prev_obs must be a contiguous float32 tensor shaped like env.obs")
        if replay.obs_dim != self.obs_dim or replay.act_dim != 2 or replay.state.device != self.obs.device:
            raise ValueError("the replay ring does not match this env (obs_dim / act_dim / device)")
        if self._direct():
            sp, op, rp, dp, mp = self._ptrs
            fp = None if self.final_obs is None else self.final_obs.data_ptr()
            rc = self._lib.uavca_step_multi_replay(self._h, sp, action.data_ptr(), _ACTION_MODES[action_mode],
                                                   int(bool(evaluate)), prev_obs.data_ptr(), op, rp, dp, fp, mp,
                                                   replay.state.data_ptr(), replay.action.data_ptr(), replay.reward.data_ptr(),
                                                   replay.next_state.data_ptr(), replay.mask.data_ptr(), replay.capacity,
                                                   replay.meta.data_ptr(), self._stream())
            if rc:
                _capi.check(rc, "uavca_step_multi_replay")
        else:
            ops.step_multi_replay(self._h, self.state.blob, action, _ACTION_MODES[action_mode], bool(evaluate), prev_obs,
                                  self.obs, self.reward, self.done, self.final_obs, self.reset_mask, replay.state,
                                  replay.action, replay.reward, replay.next_state, replay.mask, replay.meta)
        if isinstance(replay, PrioritizedDeviceReplay):
            replay.sync()
        info = {"distance": 0, "reset_mask": self.reset_mask}
        if self.final_obs is not None:
            info["final_obs"] = self.final_obs
        return self.obs, self.reward, self.done, info


class BatchedUAVWorld2D(_BatchedBase):
    """B x UAVWorld2D (uav_world_2d.py:11).  Constructor kwargs follow the reference (:14)."""

    kind = KIND_SINGLE

    def __init__(self, num_envs: int, x_size=100.0, y_size=100.0, agent_num=4, max_speed=12.0, max_acceleration=5.0, *,
                 device=None, seed=0, reset_mode=0, max_episode_steps=0, reset_source=SOURCE_PHILOX, env_index_base=0,
                 float32_first_step=False, track_scores=False):
        cfg = _capi.default_config(KIND_SINGLE)
        cfg.track_scores = int(bool(track_scores))
        cfg.num_envs, cfg.num_agents = num_envs, 1
        cfg.x_size, cfg.y_size, cfg.max_speed, cfg.max_acceleration = x_size, y_size, max_speed, max_acceleration
        cfg.seed, cfg.reset_mode, cfg.max_episode_steps = seed, reset_mode, max_episode_steps
        cfg.reset_source, cfg.env_index_base = reset_source, env_index_base
        cfg.single_f32_first_step = int(float32_first_step)
        cfg.polar_scale = float(np.float32(max_speed))  # env.action_space.high[0] (test_sac.py:77)
        super().__init__(num_envs, 1, cfg, device)
        self.x_size, self.y_size = x_size, y_size
        self.map_diagonal_size = np.linalg.norm([x_size, y_size])
        self.min_location = np.array([-x_size / 2.0, -y_size / 2.0])
        self.max_location = np.array([x_size / 2.0, y_size / 2.0])
        self.max_speed = np.array([max_speed, max_speed])
        self.min_speed = -self.max_speed
        self.max_acceleratoin = np.array([max_acceleration, max_acceleration])
        self.min_acceleratoin = -self.max_acceleratoin
        self.tau = 0.02
        self.observation_space = Box(np.array([0., -1., 0., -1.]), np.ones(4), (4,))  # uav_world_2d.py:55
        self.action_space = Box(-max_speed, max_speed, (2,))  # :64
        self.distance = torch.zeros(num_envs, dtype=torch.float32, device=self.device)

    def step(self, action: torch.Tensor, action_mode="cartesian"):
        """action [B,2] float32 CUDA -> (obs [B,1,4], reward [B,1], done [B,1] uint8, info)."""
        action = self._check_action(action)
        if self._direct():
            sp, op, rp, dp, mp = self._ptrs
            fp = None if self.final_obs is None else self.final_obs.data_ptr()
            rc = self._lib.uavca_step_single(self._h, sp, action.data_ptr(), _ACTION_MODES[action_mode], op, rp, dp,
                                             self.distance.data_ptr(), fp, mp, self._stream())
            if rc:
                _capi.check(rc, "uavca_step_single")
        else:
            ops.step_single(self._h, self.state.blob, action, _ACTION_MODES[action_mode], self.obs, self.reward, self.done,
                            self.distance, self.final_obs, self.reset_mask)
        info = {"distance": self.distance, "reset_mask": self.reset_mask}  # uav_world_2d.py:114-117
        if self.final_obs is not None:
            info["final_obs"] = self.final_obs
        return self.obs, self.reward, self.done, info


# ---- NVTX ranges (SURVEY.md 5: tracing).  Off by default and free when off: with UAVCA_NVTX=1 in the environment the entry
# points of the batched classes are wrapped once, at import, in `torch.cuda.nvtx` ranges named after the reference call
# they replace, so a timeline (nsys / ncu --nvtx) shows env.step / env.reset / rollout as named spans around the kernels.
def _nvtx_wrap(cls, name, label):
    import functools

    fn = getattr(cls, name)

    @functools.wraps(fn)
    def wrapped(self, *args, **kw):
        torch.cuda.nvtx.range_push(label)
        try:
            return fn(self, *args, **kw)
        finally:
            torch.cuda.nvtx.range_pop()

    setattr(cls, name, wrapped)


if os.environ.get("UAVCA_NVTX", "0") not in ("", "0"):
    for _cls, _tag in ((BatchedMultiUAVWorld2D, "MultiUAVWorld2D"), (BatchedUAVWorld2D, "UAVWorld2D")):
        for _name in ("step", "step_f64", "step_host", "reset", "observe", "rollout", "stats"):
            _nvtx_wrap(_cls, _name, f"uavca:{_tag}.{_name}")
    _nvtx_wrap(BatchedMultiUAVWorld2D, "step_replay", "uavca:MultiUAVWorld2D.step+memory.push")
