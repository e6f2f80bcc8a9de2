"""ms per decision step with an initial-condition pool (bskenv_set_ic_pool) against the same handle without one, auto_reset on.

    python scripts/ic_pool_bench.py [--steps 10] [--reps 5] [--out FILE]

With a pool the step path is the unchanged step kernel(s) plus one launch of the reset kernel over the envs that finished;
without one the reset happens inside the step kernel.  Cases: LEO at 131072 envs (one thread per env, work queue) and 4096
envs (split organisation), each at the default max_length and at max_length = 4 (a quarter of the envs reset every step),
and opNav at its bench.py size.  Both handles of a case live in one process and are timed alternately (reps x steps
intervals each, device events, after a warm-up), on the same seeded actions.  `reset_ms` is the reset kernel alone over a
25 % mask (device events around repeated masked resets of a third handle).  Prints one JSON object with the GPU name, power
limit and max SM clock next to the numbers."""
import argparse
import json
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--opnav-envs", type=int, default=113664)
    ap.add_argument("--out")
    args = ap.parse_args()
    import torch
    from penv_bench import gpu_info
    from basilisk_env_b200.vec_env import LeoPowerAttVecEnv
    from basilisk_env_b200.opnav_env import OpNavVecEnv
    from tests.test_ic_pool_gpu import leo_pool, opnav_pool

    if not torch.cuda.is_available():
        raise SystemExit("ic_pool_bench.py: no CUDA device")
    cases = [("leo", 131072, "thread", None), ("leo", 131072, "thread", 4), ("leo", 4096, "split", None), ("leo", 4096, "split", 4),
             ("opnav", args.opnav_envs, None, None)]
    res = {**gpu_info(), "steps_per_rep": args.steps, "reps": args.reps, "cases": []}
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for kind, n, org, max_len in cases:
        hi = 3 if kind == "leo" else 2
        pool = leo_pool(64, 4) if kind == "leo" else opnav_pool(64, 4)
        g = torch.Generator("cuda").manual_seed(n)
        acts = torch.randint(0, hi, (args.steps, n), dtype=torch.int32, device="cuda", generator=g)
        kw = {} if max_len is None else {"max_length": max_len}

        def make(with_pool):
            env = (LeoPowerAttVecEnv(n, device=0, seed=1, auto_reset=True, organisation=org, **kw) if kind == "leo"
                   else OpNavVecEnv(n, device=0, seed=1, auto_reset=True, **kw))
            if with_pool:
                env.set_ic_pool(pool, assign="per_episode")
            env.reset()
            return env
        envs = {"no_pool": make(False), "pool": make(True)}
        for env in envs.values():
            for t in range(args.warmup):
                env.step(acts[t % args.steps])
        torch.cuda.synchronize()
        times = {k: [] for k in envs}
        for _ in range(args.reps):
            for k, env in envs.items():
                ev0.record()
                for t in range(args.steps):
                    env.step(acts[t])
                ev1.record()
                ev1.synchronize()
                times[k].append(ev0.elapsed_time(ev1) / args.steps)
        resetter = make(True)
        mask = (torch.rand(n, generator=g, device="cuda") < 0.25).to(torch.uint8)
        resetter.reset(mask=mask)
        torch.cuda.synchronize()
        ev0.record()
        for _ in range(20):
            resetter.reset(mask=mask)
        ev1.record()
        ev1.synchronize()
        entry = {"workload": kind, "envs": n, "organisation": org, "max_length": max_len or "default",
                 "kernel": envs["pool"].kernel_name() if kind == "leo" else "opnav",
                 "reset_ms": ev0.elapsed_time(ev1) / 20}
        for k, v in times.items():
            entry[k] = {"ms_per_step_median": float(np.median(v)), "ms_per_step_min": float(np.min(v)), "ms_per_step_max": float(np.max(v))}
        entry["overhead_pct"] = 100.0 * (entry["pool"]["ms_per_step_median"] / entry["no_pool"]["ms_per_step_median"] - 1.0)
        res["cases"].append(entry)
        for env in list(envs.values()) + [resetter]:
            env.close()
        print(json.dumps(entry), flush=True)
    print(json.dumps(res))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
