"""The loop of the reference's test_sac_multi.py (data collection + evaluation, :62-183) on the batched device env.

Reference, per env step (one env, N agents):            Here, per env step (B envs x N agents):
  for i in range(N): agents[i].select_action(states[i])    one policy kernel over [B*N, 10]            (FusedGaussianPolicy)
  v, theta -> [v cos, v sin] on the host (:77-80)          polar map fused into the step kernel         (action_mode="polar")
  env.step(converted_actions)            (:99)             env.step(action)                             (one launch)
  memory.push(...) for i in range(N)     (:101-103)        appended by the step kernel itself           (same launch)
  reset when dones[0] or 1500 steps      (:111-119)        auto-reset inside the step (RESET_ON_DONE0, max_episode_steps)
  every 10 episodes: 10 evaluation episodes, SR / CR       evaluation batch with RESET_ON_ALL_DONE, evaluate=True

The learner (SAC.update_parameters, pytorch_sac_temp/sac.py:46-98) is stock PyTorch and out of scope; `replay.sample(256)`
/ `replay.sample_fused(256)` (one launch, slots drawn on the device) return exactly the five tensors it consumes;
`replay.sample_nstep(256, n, gamma, stride)` returns n-step returns for the same learner.

    python examples/rollout_sac_multi.py [--envs 16384] [--agents 10] [--steps 2000]
"""
import argparse
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

import gym_uav_collision_avoidance_b200 as G


def main(argv=None):
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=16384)
    ap.add_argument("--agents", type=int, default=10)     # NUM_AGENTS (test_sac_multi.py:24)
    ap.add_argument("--steps", type=int, default=2000)
    ap.add_argument("--warmup-steps", type=int, default=100)  # uniform random actions first (:72-73)
    ap.add_argument("--eval-envs", type=int, default=4096)
    args = ap.parse_args(argv)
    dev = torch.device("cuda:0")
    torch.manual_seed(0)

    env = G.BatchedMultiUAVWorld2D(args.envs, num_agents=args.agents, reset_mode=G.RESET_ON_DONE0,
                                   max_episode_steps=1500, seed=1)          # MAX_EPISOED_STEPS (:17)
    policy = G.GaussianPolicy(env.observation_space.shape[0], env.action_space.shape[0]).to(dev)
    replay = G.DeviceReplay(1_000_000, 10, 2, device=dev, seed=0)             # replay_size (:21)
    ro = G.BatchedRollout(env, policy, replay, action_mode="polar", precision="fused", warmup_uniform=True)
    ro.reset()
    ro.run(args.warmup_steps)
    ro.warmup_uniform = False
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    ro.run(args.steps)
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    batch = replay.sample_fused(256)                                          # what SAC.update_parameters consumes (:48)
    print(f"collected {args.steps * args.envs * args.agents:,} transitions in {dt:.2f} s "
          f"({args.steps * args.envs / dt:,.0f} env-steps/s, eager launches); replay holds {len(replay):,}; "
          f"sampled batch shapes {[tuple(t.shape) for t in batch]}")
    # 3-step returns for the same learner: successors are envs * agents slots apart
    nstep = replay.sample_nstep(256, n=3, gamma=0.99, stride=args.envs * args.agents)
    print(f"3-step batch shapes {[tuple(t.shape) for t in nstep]} (state, action, reward_3, next_state_3, discount); "
          f"mean discount {nstep[4].mean().item():.3f}")

    # evaluation protocol (:136-179): evaluate=True (out-of-bounds does not end the episode), stop at all(dones)
    ev = G.BatchedMultiUAVWorld2D(args.eval_envs, num_agents=args.agents, reset_mode=G.RESET_ON_ALL_DONE,
                                  max_episode_steps=1500, seed=2)
    ero = G.BatchedRollout(ev, policy, None, action_mode="polar", precision="fused", evaluate=True)
    ero.reset()
    ero.run(1500)
    sr, cr, episodes = ero.success_collision_rates()
    print(f"evaluation over {episodes:,} finished episodes: SR = {sr:.3f}, CR = {cr:.3f} (random-init policy)")
    return sr, cr, episodes


if __name__ == "__main__":
    main()
