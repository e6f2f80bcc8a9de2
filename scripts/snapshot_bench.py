"""Cost of per-env state snapshots (bskenv_snapshot / bskenv_restore and the opNav pair) next to get_state / set_state.

    python scripts/snapshot_bench.py [--reps 20] [--warmup 3] [--out profiles/snapshot_bench.json]

Cases: the LEO batch at 131072 envs without and with a parameter pool (with one the parameter block is read from the state
allocation; without one it is the configuration's block, a kernel argument), and the opNav batch at 113664 envs (bench.py's
sizes).  Each case times, with device events around `reps` back-to-back calls after `warmup` untimed ones: snapshot and
restore of every env (indices NULL) and of a random 10 % subset (indices in random order), and get_state / set_state of the
whole batch.  A restore checks its records on the device and waits for the stream before it scatters, so its time includes
the check kernel, one 16-byte read-back and the synchronisation.  `bytes` = every record word read once and written once
(2 x m x W x 8; get_state / set_state: 2 x n x fields x 8), `gbps` = bytes / time, `of_peak` = gbps over the 7.7 TB/s of the
B200 data sheet.  The full LEO records (180 MB) exceed the 126 MB L2; the opNav ones (104 MB) do not, so part of their traffic
may be served from L2.  Prints and writes one JSON object with the GPU name, power limit and max SM clock."""
import argparse
import ctypes as C
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

PEAK_GBPS = 7700.0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--leo-envs", type=int, default=131072)
    ap.add_argument("--opnav-envs", type=int, default=113664)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "snapshot_bench.json"))
    args = ap.parse_args()
    import numpy as np
    import torch
    from penv_bench import gpu_info
    from basilisk_env_b200.vec_env import LeoPowerAttVecEnv
    from basilisk_env_b200.opnav_env import OpNavVecEnv

    if not torch.cuda.is_available():
        raise SystemExit("snapshot_bench.py: no CUDA device")
    res = {**gpu_info(), "reps": args.reps, "warmup": args.warmup, "peak_gbps": PEAK_GBPS, "cases": []}
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def timed(fn, bytes_):
        for _ in range(args.warmup):
            fn()
        torch.cuda.synchronize()
        ev0.record()
        for _ in range(args.reps):
            fn()
        ev1.record()
        ev1.synchronize()
        ms = ev0.elapsed_time(ev1) / args.reps
        gbps = bytes_ / (ms * 1e-3) / 1e9
        return {"ms": round(ms, 5), "bytes": int(bytes_), "gbps": round(gbps, 1), "of_peak": round(gbps / PEAK_GBPS, 4)}

    def rng_pool(k):
        r = np.random.RandomState(7)
        return {"mass": r.uniform(250.0, 420.0, k), "panelArea": r.uniform(0.5, 1.5, k)}

    for kind, n, pool in (("leo", args.leo_envs, False), ("leo", args.leo_envs, True), ("opnav", args.opnav_envs, False)):
        env = LeoPowerAttVecEnv(n, device=0, seed=1) if kind == "leo" else OpNavVecEnv(n, device=0, seed=1)
        if pool:
            env.set_param_pool(rng_pool(64))
        env.reset()
        f, h = env._f, env._h
        st = env._stream()
        W = int(f.snapshot_width(h))
        fields = env.n_double_fields + env.n_int_fields
        m = n // 10
        sub = torch.randperm(n, device="cuda", generator=torch.Generator("cuda").manual_seed(3))[:m].contiguous()
        rec_all = torch.empty((n, W), dtype=torch.float64, device="cuda")
        rec_sub = torch.empty((m, W), dtype=torch.float64, device="cuda")
        d = torch.empty((env.n_double_fields, n), dtype=torch.float64, device="cuda")
        i = torch.empty((env.n_int_fields, n), dtype=torch.int64, device="cuda")
        ra, rs, sp = C.c_void_p(rec_all.data_ptr()), C.c_void_p(rec_sub.data_ptr()), C.c_void_p(sub.data_ptr())
        dp, ip, op = C.c_void_p(d.data_ptr()), C.c_void_p(i.data_ptr()), C.c_void_p(env.obs.data_ptr())

        def call(rc):
            assert rc == 0, f.last_error(h).decode()
        call(f.snapshot(h, n, None, ra, st))
        call(f.snapshot(h, m, sp, rs, st))
        case = {"kind": kind, "envs": n, "param_pool": pool, "W": W, "subset": m}
        case["snapshot_all"] = timed(lambda: call(f.snapshot(h, n, None, ra, st)), 2 * n * W * 8)
        case["restore_all"] = timed(lambda: call(f.restore(h, n, None, ra, op, st)), 2 * n * W * 8)
        case["snapshot_10pct"] = timed(lambda: call(f.snapshot(h, m, sp, rs, st)), 2 * m * W * 8)
        case["restore_10pct"] = timed(lambda: call(f.restore(h, m, sp, rs, op, st)), 2 * m * W * 8)
        case["get_state"] = timed(lambda: call(f.get_state(h, dp, ip, st)), 2 * n * fields * 8)
        case["set_state"] = timed(lambda: call(f.set_state(h, dp, ip, st)), 2 * n * fields * 8)
        res["cases"].append(case)
        env.close()
    text = json.dumps(res, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(text + "\n")


if __name__ == "__main__":
    main()
