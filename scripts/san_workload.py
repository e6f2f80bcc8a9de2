import sys, os
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
from basilisk_env_b200.vec_env import LeoPowerAttVecEnv
from basilisk_env_b200.opnav_env import OpNavVecEnv
env = LeoPowerAttVecEnv(200, device=0, auto_reset=True, step_duration=20.0, max_length=2)
env.reset(seed=1)
for t in range(4):
    env.step(torch.full((200,), t % 3, dtype=torch.int32, device="cuda"))
env.step_host(np.zeros(200, np.int32))
print("leo", env.episode_stats()); env.close()
on = OpNavVecEnv(100, device=0, auto_reset=True, step_duration_min=2.0, max_length=2, camera_reenable=1, sample_orbit=1)
on.reset(seed=2)
for t in range(4):
    on.step(torch.full((100,), t % 2, dtype=torch.int32, device="cuda"))
on.step_host(np.zeros(100, np.int32))
print("opnav", on.episode_stats()); on.close()
# SURVEY 8(f)-4 paths: ephemeris tables (global-memory look-ups) and the planet-fixed degree-2 variant (larger bus)
from basilisk_env_b200 import ephemeris as eph
env = LeoPowerAttVecEnv(200, device=0, auto_reset=True, step_duration=20.0, max_length=2, rw_set=1)
env.set_gravity_degree2(True)
env.set_ephemeris("sun", eph.ChebTable.fit(eph.analytic_sun, 0.0, 40.0, 3, 6))
env.set_ephemeris("orientation", eph.ChebTable.fit(eph.iau_earth_angles, 0.0, 100.0, 1, 4))
env.reset(seed=3)
for t in range(4):
    env.step(torch.full((200,), (t + 1) % 3, dtype=torch.int32, device="cuda"))
print("leo degree2+tables", env.episode_stats()); env.close()
on = OpNavVecEnv(100, device=0, auto_reset=True, step_duration_min=2.0, max_length=2, camera_reenable=1)
on.set_ephemeris(eph.ChebTable.fit(lambda t: np.array([2.0e11, 5.0e10, 1.0e10]) + 2.0e4 * t * np.array([-0.2, 1.0, 0.4]), 0.0, 200.0, 2, 3))
on.reset(seed=4)
for t in range(3):
    on.step(torch.full((100,), t % 2, dtype=torch.int32, device="cuda"))
print("opnav table", on.episode_stats()); on.close()
# chunked work items through the queue (more groups than resident warps): 60000 envs, 6 s intervals = 6 chunks of 10 ticks
env = LeoPowerAttVecEnv(60000, device=0, auto_reset=True, step_duration=6.0, max_length=3, seed=5)
env.reset()
for t in range(3):
    env.step(torch.full((60000,), t % 3, dtype=torch.int32, device="cuda"))
# ... and with mixed actions: the envs are bucketed by action (bucket_count_kernel + bucket_fill_kernel), the step kernel gathers through the permutation
gq = torch.Generator(device="cuda"); gq.manual_seed(1)
for t in range(2):
    env.step(torch.randint(0, 4, (60000,), dtype=torch.int32, device="cuda", generator=gq))
print("leo queue+chunks", env.episode_stats()); env.close()
# round 2: zero-copy host buffers (the kernel reads / writes page-locked host memory), per-env episode record, async / wait,
# the stable-baselines adapter; batches of 200 envs run the small-batch organisation (MINB = 1), 60000 the throughput one
env = LeoPowerAttVecEnv(200, device=0, auto_reset=True, step_duration=20.0, max_length=2, seed=6)
env.reset()
act, out = env.host_buffers(episode=True)
for t in range(4):
    act[:] = t % 3
    env.step_host_async(act, out); env.step_host_wait()
env.step(torch.zeros(200, dtype=torch.int32, device="cuda"))
env.step_host(np.ones(200, np.int32))          # pageable buffers: staging path
print("leo zero-copy", env.episode_stats(), float(out[4].sum()), int(out[5].sum())); env.close()
from basilisk_env_b200.sb_vec_env import LeoPowerAttSBVecEnv
sb = LeoPowerAttSBVecEnv(96, device=0, seed=7, step_duration=20.0, max_length=2)
sb.reset()
for t in range(4):
    sb.step(np.full(96, t % 3))
print("sb adapter ok"); sb.close()
# round 2: the split (two warps per env group) organisation: named barriers + shared-memory mailbox; one group per
# block (several groups per block need more than 148 groups: tests/test_gpu_split.py), both configurations, mode 2 (desat chain crosses the FSW barrier), fresh and running envs in one warp
for n, kw in ((64, {}), (64 * 6, {}), (64, dict(use_j2=1, rw_set=1))):
    env = LeoPowerAttVecEnv(n, device=0, auto_reset=True, step_duration=20.0, max_length=2, seed=8, organisation="split", **kw)
    env.reset()
    for t in range(4):
        env.step(torch.randint(0, 3, (n,), dtype=torch.int32, device="cuda"))
    print("leo split", n, env.kernel_name(), env.episode_stats()["episodes"]); env.close()
# round 2: the opNav decision interval as two kernels with the work queues of both (more groups than one resident set of the
# three-block builds: 60000 envs), measurement hand-over buffer, auto-reset in the second kernel; 0.5 min intervals = 30 ticks
on = OpNavVecEnv(60000, device=0, auto_reset=True, step_duration_min=0.5, max_length=2, camera_reenable=1, sample_orbit=1, noise_seed=9)
on.reset(seed=9)
for t in range(3):
    on.step(torch.randint(0, 2, (60000,), dtype=torch.int32, device="cuda"))
print("opnav two kernels + queues", on.episode_stats()["episodes"]); on.close()

# opNav three-kernel interval (opt-in): noise kernel -> slot-major buffer -> dynamics kernel fed through cp.async -> filter
os.environ["BSKENV_OPNAV_NOISE_SPLIT"] = "1"
on = OpNavVecEnv(333, device=0, auto_reset=True, step_duration_min=2.0, max_length=2, camera_reenable=1, sample_orbit=1)
on.reset(seed=8)
for t in range(4):
    on.step(torch.randint(0, 2, (333,), dtype=torch.int32, device="cuda"))
assert on.launch_count() == 12
print("opnav three-kernel", on.episode_stats()); on.close()
os.environ["BSKENV_OPNAV_NOISE_SPLIT"] = "0"
