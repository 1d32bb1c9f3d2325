"""Device time per env step of K-steps-per-launch rollouts (uavca_rollout), one stream, CUDA events.
    python tools/rollout_time.py KIND N B K [philox|block] [reps] [plain|general]      (KIND = multi | single)
general: the launch also asks for final_obs, reset_mask and (Philox) the actions taken, as a training-style rollout does;
the multi-UAV world then runs its general kernel instance instead of the plain one."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import gym_uav_collision_avoidance_b200 as G

kind = sys.argv[1] if len(sys.argv) > 1 else "multi"
N = int(sys.argv[2]) if len(sys.argv) > 2 else 8
B = int(sys.argv[3]) if len(sys.argv) > 3 else 65536
K = int(sys.argv[4]) if len(sys.argv) > 4 else 32
mode = sys.argv[5] if len(sys.argv) > 5 else "philox"
reps = int(sys.argv[6]) if len(sys.argv) > 6 else 20
launch = sys.argv[7] if len(sys.argv) > 7 else "plain"
want = dict(want_final_obs=True, want_reset_mask=True, want_actions=True) if launch == "general" else {}
dev = torch.device("cuda:0")
if kind == "single":
    env = G.BatchedUAVWorld2D(B, reset_mode=G.RESET_ON_ANY_DONE, max_episode_steps=1500, seed=0x5EED)
    N, amax, alg = 1, 12.0, 89.0
else:
    env = G.BatchedMultiUAVWorld2D(B, num_agents=N, reset_mode=G.RESET_ON_DONE0, max_episode_steps=1500, seed=0x5EED)
    amax, alg = 10.0, 107.0 + 24.0 / N
env.reset()
acts = None
if mode == "block":
    acts = (torch.rand((K, B, N, 2), device=dev) * 2 - 1) * amax
out = env.rollout(K, acts, action_seed=1, step0=0, sync_last=False, **want)
torch.cuda.synchronize()
best = 1e30
for r in range(3):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(reps):
        env.rollout(K, acts, action_seed=1, step0=(r * reps + i + 1) * K, out=out, sync_last=False)
    e1.record()
    torch.cuda.synchronize()
    best = min(best, e0.elapsed_time(e1) * 1e3 / (reps * K))
out_bytes = (4 if kind == "single" else 10) * 4 + 4 + 1 + (8 if mode == "block" else 0)
print(f"{os.environ.get('UAVCA_LIB', 'default').split('/')[-1]:24s} rollout {kind} N={N} B={B} K={K} {mode:6s} {launch:7s} {best:9.3f} us/step "
      f"{B * N / best / 1e3:7.2f} G UAV-steps/s  frac(alg {alg:.1f} B) {B * N * alg / best / 1e3 / 6515.7:.3f}  "
      f"frac(moved {out_bytes} B) {B * N * out_bytes / best / 1e3 / 6515.7:.3f}", flush=True)
