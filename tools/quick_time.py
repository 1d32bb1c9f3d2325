"""Device time per step of one workload (CUDA-graph replay over a ring of batches larger than L2), no CPU legs.
    python tools/quick_time.py [N] [B] [steps]      (UAVCA_LIB selects the library variant)"""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import gym_uav_collision_avoidance_b200 as G

N = int(sys.argv[1]) if len(sys.argv) > 1 else 8
B = int(sys.argv[2]) if len(sys.argv) > 2 else 65536
steps = int(sys.argv[3]) if len(sys.argv) > 3 else 2000
dev = torch.device("cuda:0")
per = B * N * 102
ring = max(1, min(64, int(-(-3.2 * 126e6 // per))))
envs = [G.BatchedMultiUAVWorld2D(B, num_agents=N, reset_mode=1, max_episode_steps=1500, seed=0x5EED, env_index_base=r * B) for r in range(ring)]
gen = torch.Generator(device=dev).manual_seed(1234)
acts = [(torch.rand((B, N, 2), generator=gen, device=dev) * 20 - 10) for _ in range(max(ring, 4))]
for e in envs:
    e.reset()
G_STEPS = min(steps, 200)
for k in range(2 * ring):
    envs[k % ring].step(acts[k % len(acts)])
torch.cuda.synchronize()
st = torch.cuda.Stream()
S = int(os.environ.get("STREAMS", "1"))  # independent batches of the ring pipelined over S streams
side = [torch.cuda.Stream() for _ in range(S - 1)]
g = torch.cuda.CUDAGraph()
with torch.cuda.graph(g, stream=st):
    fork = torch.cuda.Event()
    fork.record(st)
    for s_ in side:
        s_.wait_event(fork)
    for k in range(G_STEPS):
        lane = (k % ring) % S  # a batch always runs on the same stream: its own steps stay ordered
        with torch.cuda.stream(st if lane == 0 else side[lane - 1]):
            envs[k % ring].step(acts[(k + k // ring) % len(acts)])
    for s_ in side:
        j = torch.cuda.Event()
        j.record(s_)
        st.wait_event(j)
g.replay()
torch.cuda.synchronize()
reps = max(1, steps // G_STEPS)
best = 1e30
for _ in range(3):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with torch.cuda.stream(st):
        e0.record(st)
        for _ in range(reps):
            g.replay()
        e1.record(st)
    st.synchronize()
    best = min(best, e0.elapsed_time(e1) * 1e3 / (reps * G_STEPS))
alg = 107 + 24 / N
print(f"{os.environ.get('UAVCA_LIB', 'default').split('/')[-1]:28s} streams={S} N={N} B={B} ring={ring} "
      f"{best:9.2f} us/step  {B * N / best / 1e3:7.2f} G UAV-steps/s  frac {B * N * alg / best / 1e3 / 6515.7:.3f}", flush=True)
