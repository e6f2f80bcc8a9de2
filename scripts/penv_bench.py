"""ms per decision step of the batch-global step kernel against the per-env parameter kernel (bskenv_set_param_pool).

    python scripts/penv_bench.py [--envs 131072 4096] [--steps 10] [--reps 5] [--out FILE]

Both handles live in one process and are timed alternately (reps x steps intervals each, device events, after a warm-up of
every shape), on the same seeded initial conditions and actions; the per-env handle carries a pool of 64 dispersed rows
assigned per episode.  With BSKENV_LIB pointing at a build with -DLEO_PENV_GLOBAL the per-env kernel reads its stage-rate
parameters from global memory instead of the shared-memory bus (DESIGN.md section 12).  Prints one JSON object with the GPU
name and power limit next to the numbers."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, clock = [x.strip() for x in q.split(",")]
        return {"gpu": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as exc:           # the numbers stay meaningful only with the card named: say it is missing
        return {"gpu": "unknown", "error": str(exc)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, nargs="+", default=[131072, 4096])
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out")
    args = ap.parse_args()
    import torch
    from basilisk_env_b200.vec_env import LeoPowerAttVecEnv
    from basilisk_env_b200 import build
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests"))
    from oracle_params import dispersed_pool

    if not torch.cuda.is_available():
        raise SystemExit("penv_bench.py: no CUDA device")
    res = {"lib": os.path.basename(build.LIB), **gpu_info(), "steps_per_rep": args.steps, "reps": args.reps, "sizes": {}}
    for n in args.envs:
        g = torch.Generator("cuda").manual_seed(n)
        acts = torch.randint(0, 3, (args.steps, n), dtype=torch.int32, device="cuda", generator=g)
        envs = {}
        for kind in ("batch", "penv"):
            env = LeoPowerAttVecEnv(n, device=0, seed=1, auto_reset=True)
            if kind == "penv":
                env.set_param_pool(dispersed_pool(64, seed=4), assign="per_episode")
            env.reset()
            for t in range(args.warmup):
                env.step(acts[t % args.steps])
            envs[kind] = env
        torch.cuda.synchronize()
        times = {k: [] for k in envs}
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        for _ in range(args.reps):
            for kind, env in envs.items():
                ev0.record()
                for t in range(args.steps):
                    env.step(acts[t])
                ev1.record()
                ev1.synchronize()
                times[kind].append(ev0.elapsed_time(ev1) / args.steps)
        entry = {k: {"kernel": envs[k].kernel_name(), "ms_per_step_median": float(np.median(v)),
                     "ms_per_step_min": float(np.min(v)), "ms_per_step_max": float(np.max(v))} for k, v in times.items()}
        entry["penv_over_batch"] = entry["penv"]["ms_per_step_median"] / entry["batch"]["ms_per_step_median"]
        res["sizes"][str(n)] = entry
        for env in envs.values():
            env.close()
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
