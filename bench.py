#!/usr/bin/env python
"""Headline benchmark: env decision-steps/s of the LEO power/attitude environment step.

    python bench.py --gpus N --steps K --warmup W            (N>1: launched under torch.distributed.run)
    python bench.py --impl reference ...                      (CPU arm: the oracle port on the host cores)

One "step" = one decision interval (180 s of simulated time = 1800 RK4 ticks + 1800 environment
ticks + 180 flight-software ticks) of EVERY env of the batch = one launch of leo_step_kernel.
Workload: BASELINE.json configs[2] -- 2^20 envs sharded over 8 GPUs, i.e. 131072 envs per GPU with
weak scaling (per-GPU work fixed), random initial orbits, i.i.d. uniform actions, auto-reset so the
batch stays in steady state.  Side measurements in the same line: "batch4096" (configs[1]: the split organisation of the
kernel, with the one-thread organisation beside it), "stress" (configs[4]: J2 + four wheels + dumping, FP64 and mixed precision) and "opnav" (configs[3]).
`e2e` goes through bskenv_step_host with host buffers (zero-copy page-locked memory).  Prints ONE JSON line (rank 0).
`--dump-outputs DIR` also writes what the last timed step of the headline returned, so that two builds can be compared on the
same seeded inputs."""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True     # the benchmark writes nothing into the tree (it may run from a read-only checkout)

METRIC = "env decision-steps/sec"
UNIT = "env-steps/s"
ENVS_PER_GPU = 131072          # 2^20 envs over 8 GPUs (BASELINE.json configs[2])
H2D_BYTES_PER_ENV = 4          # int32 action
D2H_BYTES_PER_ENV = 5 * 8 + 8 + 1 + 1   # obs[5] f64, reward f64, done u8, done_reason u8
# ALGORITHMIC bytes per env-step: persistent state read + written once, plus the step I/O (DESIGN.md)
STATE_BYTES_PER_ENV = (89 + 22) * 8
# the ncu capture of the shipped build whose executed-flop count the roofline numerator is checked against
FLOP_CAPTURE = "profiles/ncu_leo_r02f.md: 1.9484e6 per env-step"     # the ncu capture of the shipped build the flop model is checked against


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--envs-per-gpu", type=int, default=ENVS_PER_GPU)
    ap.add_argument("--cpu-seconds", type=float, default=12.0, help="bounded CPU-baseline sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip the 4096-env and opNav side measurements")
    ap.add_argument("--workload", default="leo", choices=["leo", "opnav"],
                    help="leo: the headline line (default); opnav: the same JSON line for BASELINE configs[3] (N=1 only)")
    ap.add_argument("--opnav-envs", type=int, default=113664,
                    help="opNav batch: two resident sets of the step kernel's three-block organisation (148 SMs x 3 blocks x 128 "
                         "threads = 56832 envs each) = three sets of its two-block organisation")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last timed step of the headline returned (obs, reward, done and "
                         "the info arrays) as DIR/<name>.npy, float64, at most 64 MB (a fixed sample of envs beyond that; "
                         "env_index.npy names them); rank 0's envs under --gpus N > 1")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if args.dump_outputs and (args.impl != "native" or args.workload != "leo"):
        ap.error("--dump-outputs applies to the headline (--impl native --workload leo)")
    return args


class ClockSampler:
    """nvidia-smi clocks + throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows, self.proc, self.thread = [], None, None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), line.strip()))

    def mark(self):
        return time.perf_counter()

    def stop(self, t0, t1):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        self.proc.wait()              # reap it: no defunct nvidia-smi left behind
        self.thread.join()
        sm, mx, pw, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        rows = [r for t, r in self.rows if t0 - 0.05 <= t <= t1 + 0.15] or [r for _, r in self.rows]
        for r in rows:
            f = [x.strip() for x in r.split(",")]
            try:
                sm.append(float(f[0])); mx.append(float(f[1])); pw.append(float(f[2]))
            except (ValueError, IndexError):
                continue
            for nm, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "samples": len(sm), "reasons": sorted(reasons)}


def host_threads():
    """All host threads this process may use.  torchrun exports OMP_NUM_THREADS=1 to its workers; the CPU arm asks
    OpenMP for an explicit thread count instead, so that it is the same under `python` and under `torchrun`."""
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        return max(1, os.cpu_count() or 1)


CPU_BUILDS = {"parity": "-O2 -ffp-contract=off (the build every parity test runs against)",
              "fast": "-O3 -march=native (contraction allowed; compiled on this box)"}


def cpu_arm(envs_per_core_step, seconds, min_steps, warmup, threads=None, fixed_steps=None, build="fast"):
    """Times the oracle port (oracle/bsk_oracle.c, OpenMP over envs) on the host cores: the same
    workload definition (random initial orbits, i.i.d. uniform actions), bounded sample."""
    from oracle import oracle as orc
    from tests import parity
    threads = threads or host_threads()
    L = orc.fast_lib() if build == "fast" else orc.lib()
    n = envs_per_core_step * threads
    rows = parity.sample_rows(orc, n, seed=7)
    batch = orc.LeoEnvBatch(rows, L=L)
    rng = np.random.RandomState(3)
    for _ in range(warmup):
        batch.step(rng.randint(0, 3, n), nthreads=threads)
    steps, t0 = 0, time.perf_counter()
    while True:
        batch.step(rng.randint(0, 3, n), nthreads=threads)
        steps += 1
        el = time.perf_counter() - t0
        if fixed_steps is not None:
            if steps >= fixed_steps:
                break
        elif el >= seconds and steps >= min_steps:
            break
    return {"value": n * steps / el, "unit": UNIT, "cores": threads, "kind": "port", "build": build, "build_flags": CPU_BUILDS[build],
            "sample": f"{n} envs x {steps} decision steps (oracle/bsk_oracle.c, gcc {CPU_BUILDS[build].split(' (')[0]}, OpenMP over envs, "
                      f"{threads} thread{'s' if threads > 1 else ''}, {el:.1f} s)",
            "ms_per_step": el / steps * 1e3, "envs": n, "steps": steps}


def cpu_baseline_block(seconds):
    """BASELINE.md section 3: the restated CPU path with 1 thread and with all host threads, as the parity build and as an
    optimised build.  The block's own value is the strongest of the four (optimised build, all threads)."""
    per = max(seconds / 4.0, 1.0)
    variants = [cpu_arm(8, per, 1, 1, threads=1, build="parity"), cpu_arm(8, per, 1, 1, threads=1, build="fast"),
                cpu_arm(4, per, 2, 1, build="parity"), cpu_arm(4, per, 2, 1, build="fast")]
    best = max(variants[2:], key=lambda v: v["value"])
    keys = ("value", "unit", "cores", "kind", "sample", "build_flags")
    out = {k: best[k] for k in keys}
    out["variants"] = [{k: v[k] for k in ("value", "cores", "build_flags", "sample")} for v in variants]
    out["note"] = ("in-repo FP64 restatement of the Basilisk 1.x algorithms (Basilisk itself cannot be built here); scalar code, one env "
                   "per thread")
    return out


def run_reference(args, rank):
    if rank != 0:
        return
    res = cpu_arm(envs_per_core_step=32, seconds=0.0, min_steps=1, warmup=args.warmup, fixed_steps=args.steps, build="fast")
    line = {"metric": METRIC, "value": res["value"], "unit": UNIT, "impl": "reference", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": res["ms_per_step"], "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": workload_name(args.envs_per_gpu), "note":
                       "CPU arm = in-repo FP64 restatement of the Basilisk 1.x algorithms (Basilisk itself cannot be built "
                       "or installed in this image: no Eigen/SWIG/conan/CSPICE, no network), optimised host build "
                       f"({CPU_BUILDS['fast']}), all host threads; each step is a bounded sample of {res['envs']} envs of the same workload"},
            "cpu_baseline": {k: res[k] for k in ("value", "unit", "cores", "kind", "sample", "build_flags")},
            "e2e": {"value": res["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def workload_name(envs_per_gpu):
    return (f"LEO power/attitude env, {envs_per_gpu} envs per GPU (BASELINE configs[2]: 2^20 envs over 8 GPUs), random initial "
            "orbits, i.i.d. uniform actions {0,1,2}, auto-reset, FP64")


def time_device_steps(env, actions_dev, steps, warmup, torch, dist, world):
    """K launches on the current stream between CUDA events; per-launch events give the kernel duration.  Also returns what
    the last timed env.step returned (the env's own buffers: valid until its next step)."""
    for t in range(warmup):
        env.step(actions_dev[t % len(actions_dev)])
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
        torch.cuda.synchronize()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(steps + 1)]
    ev[0].record()
    for t in range(steps):
        last = env.step(actions_dev[(warmup + t) % len(actions_dev)])
        ev[t + 1].record()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    total_ms = ev[0].elapsed_time(ev[steps])
    per = [ev[t].elapsed_time(ev[t + 1]) for t in range(steps)]
    return total_ms, per, last


DUMP_LIMIT_BYTES = 64 << 20


def snapshot_outputs(obs, reward, done, info):
    """Device copies of what one LeoPowerAttVecEnv.step returned, as float64 arrays [N] or [N, 5].  terminal_obs is defined
    only for the envs that finished in that step (the library leaves the other rows as they were): those rows are zeroed."""
    fin = done.bool()
    return {"obs": obs.double().clone(), "reward": reward.double().clone(), "done": done.double(),
            "done_reason": info["done_reason"].double(), "terminal_obs": info["terminal_obs"].double() * fin[:, None],
            "episode_r": info["episode_r"].double().clone(), "episode_l": info["episode_l"].double()}


def dump_outputs(outdir, arrays):
    """Writes each array as outdir/<name>.npy.  Beyond DUMP_LIMIT_BYTES in all, a fixed seeded sample of envs (rows) is
    written; env_index.npy holds the env indices of the rows either way."""
    n = len(arrays["obs"])
    per_env = 8 * (1 + sum(int(np.prod(a.shape[1:])) for a in arrays.values()))
    m = min(n, DUMP_LIMIT_BYTES // per_env)
    idx = np.arange(n) if m == n else np.sort(np.random.RandomState(0).choice(n, m, replace=False))
    os.makedirs(outdir, exist_ok=True)
    np.save(os.path.join(outdir, "env_index.npy"), idx.astype(np.float64))
    for name, a in arrays.items():
        np.save(os.path.join(outdir, f"{name}.npy"), a.cpu().numpy()[idx])


def main():
    args = parse()
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        if args.workload == "opnav":
            if rank == 0:
                cb = opnav_cpu_arm(8, 0.0, fixed_steps=args.steps)
                print(json.dumps({"metric": METRIC, "value": cb["value"], "unit": UNIT, "impl": "reference", "n_gpus": args.gpus,
                                  "steps": args.steps, "warmup": args.warmup, "ms_per_step": cb["ms_per_step"],
                                  "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
                                  "data": "synthetic", "config": {"workload": opnav_workload_name(args.opnav_envs)},
                                  "cpu_baseline": {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample", "build_flags")},
                                  "e2e": {"value": cb["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                                  "gpu_launches": 0}), flush=True)
            return
        run_reference(args, rank)
        return
    if args.workload == "opnav":
        if rank == 0:
            run_opnav(args)
        return
    import torch
    import torch.distributed as dist
    from basilisk_env_b200.vec_env import LeoPowerAttVecEnv, fp64_peak_tflops, all_reduce_stats
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (the environment step has no CPU path)")
    torch.cuda.set_device(local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    E, K, W = args.envs_per_gpu, args.steps, args.warmup
    dev = torch.device("cuda", local_rank)
    env = LeoPowerAttVecEnv(E, device=local_rank, first_env_index=rank * E, seed=20211504, auto_reset=True)
    env.reset()
    g = torch.Generator(device=dev).manual_seed(1234 + rank)
    n_act = K + W
    actions_dev = torch.randint(0, 3, (n_act, E), dtype=torch.int32, device=dev, generator=g)
    actions_host = actions_dev.cpu().numpy()
    # host side of the plugin call: page-locked buffers the library hands out (env.host_buffers -> zero-copy); a caller
    # with ordinary numpy arrays gets the same result through staging + one memcpy per buffer
    act_pinned, outs = env.host_buffers()

    # FP64 roofline denominator: measured live (MEASURED_PEAKS.json carries HBM and bf16 only)
    peak_tf = fp64_peak_tflops(local_rank, 0.5) if rank == 0 else None

    sampler = ClockSampler(local_rank) if rank == 0 else None
    l0 = env.launch_count()
    t_mark0 = time.perf_counter()
    total_ms, per_ms, last = time_device_steps(env, actions_dev, K, W, torch, dist, world)
    dumped = snapshot_outputs(*last) if args.dump_outputs and rank == 0 else None   # before the steps below overwrite them
    # ---- end to end through the host-buffer C-ABI entry point (bskenv_step_host) ----
    for t in range(min(W, 3)):
        act_pinned[:] = actions_host[t]
        env.step_host(act_pinned, outs)
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    e0 = time.perf_counter()
    for t in range(K):
        act_pinned[:] = actions_host[W + t]           # the trainer's actions of this step (host memory)
        env.step_host(act_pinned, outs)               # actions in, results out and the sync: all inside the call
    torch.cuda.synchronize()
    e2e_ms = (time.perf_counter() - e0) * 1e3
    t_mark1 = time.perf_counter()
    # kernels per decision step (large batches: bucket count + bucket fill + step kernel) x the 2K steps of the timed regions
    launches = (env.launch_count() - l0) // (W + K + min(W, 3) + K) * 2 * K
    kernel_name = env.kernel_name()
    clocks = sampler.stop(t_mark0, t_mark1) if sampler else None
    checksum = float(outs[1].sum())

    t = torch.tensor([total_ms, e2e_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    total_ms, e2e_ms = float(t[0]), float(t[1])
    stats = env.episode_stats(all_reduce=world > 1)          # the one optional collective (8 scalars)

    if rank == 0:
        n_total = E * world
        value = n_total * K / (total_ms * 1e-3)
        e2e_value = n_total * K / (e2e_ms * 1e-3)
        kern_ms = float(np.mean(per_ms))
        flops = env.flops_per_step()
        achieved_tf = flops * E / (kern_ms * 1e-3) / 1e12
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except OSError:
            pass
        traffic = None
        try:
            traffic = json.load(open(os.path.join(ROOT, "profiles", "traffic.json"))).get("dram_bytes_per_launch")
        except (OSError, ValueError):
            pass
        hbm_peak = peaks.get("hbm_gbs", 6650.0)
        alg_bytes = (2 * STATE_BYTES_PER_ENV + H2D_BYTES_PER_ENV + D2H_BYTES_PER_ENV) * E
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": total_ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic",
            "config": {"workload": workload_name(E), "envs_per_gpu": E, "envs_total": n_total, "ticks_per_step": 1800,
                       "l2": f"inputs larger than L2: {(STATE_BYTES_PER_ENV + 19 * 8) * E / 2**20:.0f} MiB of per-env state per GPU "
                             "vs 126 MB L2 (and the kernel is FP64-pipe bound, not memory bound)",
                       "parallelism": f"env-sharded x{world}, no collective on the step path"},
            "roofline": {"bound": "fp64", "achieved": achieved_tf, "peak": peak_tf, "unit": "TFLOP/s",
                         "frac": achieved_tf / peak_tf if peak_tf else None, "traffic": traffic,
                         "traffic_note": "ncu capture at 131072 envs (profiles/traffic.json); above the algorithmic bytes by design: the "
                                         "interval runs as 6 chunks with a state round trip each, gathered through the action-bucket permutation "
                                         "(DESIGN.md section 5), < 2 % of HBM bandwidth",
                         "kernel": kernel_name, "kernel_ms": kern_ms, "flop_per_env_step": flops,
                         "flop_source": "operation list of the kernel as built (bskenv_flops_per_step), equal to the executed "
                                        f"2*DFMA+DMUL+DADD count of ncu ({FLOP_CAPTURE}); the un-fused "
                                        "Basilisk formulation of SURVEY 8(d) would be 4.29e6",
                         "peak_source": "DFMA-chain microbenchmark run in this process (bskenv_fp64_peak); MEASURED_PEAKS.json "
                                        "has no FP64 figure; nominal 148 SM x 64 FMA/clk x 1.965 GHz = 37.2 TFLOP/s",
                         "hbm": {"achieved": alg_bytes / (kern_ms * 1e-3) / 1e9, "peak": hbm_peak, "unit": "GB/s",
                                 "frac": alg_bytes / (kern_ms * 1e-3) / 1e9 / hbm_peak, "algorithmic_bytes_per_launch": alg_bytes,
                                 "peak_source": "MEASURED_PEAKS.json" if peaks else "fallback"}},
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": H2D_BYTES_PER_ENV * E, "d2h_bytes_per_step": D2H_BYTES_PER_ENV * E,
                    "ms_per_step": e2e_ms / K, "api": "bskenv_step_host with page-locked host buffers (env.host_buffers): the kernel reads the actions from and writes "
                           "obs / reward / done / reason to host memory in place, over PCIe, inside the launch"},
            "gpu_launches": int(launches), "clocks": clocks,
            "episode_stats": stats, "checksum": checksum,
        }
        if not args.no_extra:
            line["batch4096"] = side_batch(4096, torch, dev, peak_tf)
            if world == 1:
                line["stress"] = side_stress(65536, torch, dev, peak_tf)
                line["opnav"] = side_opnav(args.opnav_envs, torch, dev, peak_tf, steps=3, warmup=3,
                                           cpu_seconds=0.0 if args.no_cpu_baseline else 4.0)
        if world == 1 and not args.no_cpu_baseline:
            line["cpu_baseline"] = cpu_baseline_block(args.cpu_seconds)
        else:
            line["cpu_baseline"] = None
        print(json.dumps(line), flush=True)
        if dumped is not None:
            dump_outputs(args.dump_outputs, dumped)
    env.close()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def side_batch(n, torch, dev, peak_tf):
    """BASELINE configs[1]: 4096 envs on one GPU -- fewer env groups than SM sub-partitions.  The library picks the split
    organisation (two warps per group of 32 envs: csrc/leo_split.cuh, DESIGN.md section 5b); the one-thread organisation
    (bskenv_set_organisation) is timed beside it on the same actions, and the split one also end to end through
    bskenv_step_host with host buffers."""
    from basilisk_env_b200.vec_env import LeoPowerAttVecEnv
    acts = torch.randint(0, 3, (13, n), dtype=torch.int32, device=dev)
    acts_host = acts.cpu().numpy()
    out = {}
    for org in ("auto", "thread"):
        env = LeoPowerAttVecEnv(n, device=dev.index, seed=5, auto_reset=True, organisation=org)
        env.reset()
        total_ms, per, _ = time_device_steps(env, acts, 10, 3, torch, None, 1)
        flops, name = env.flops_per_step(), env.kernel_name()
        ms = total_ms / 10
        tf = flops * n / (ms * 1e-3) / 1e12
        res = {"envs": n, "value": n / (ms * 1e-3), "unit": UNIT, "ms_per_step": ms, "fp64_tflops": tf,
               "frac": tf / peak_tf if peak_tf else None, "kernel": name}
        if org == "auto":
            act_pinned, outs = env.host_buffers()
            for t in range(3):
                act_pinned[:] = acts_host[t]; env.step_host(act_pinned, outs)
            torch.cuda.synchronize()
            e0 = time.perf_counter()
            for t in range(10):
                act_pinned[:] = acts_host[3 + t]; env.step_host(act_pinned, outs)
            torch.cuda.synchronize()
            e_ms = (time.perf_counter() - e0) * 1e3 / 10
            res["e2e"] = {"value": n / (e_ms * 1e-3), "unit": UNIT, "ms_per_step": e_ms, "h2d_bytes_per_step": H2D_BYTES_PER_ENV * n,
                          "d2h_bytes_per_step": D2H_BYTES_PER_ENV * n, "api": "bskenv_step_host, page-locked host buffers"}
            out = res
        else:
            out["one_thread_per_env"] = {k: res[k] for k in ("value", "ms_per_step", "frac", "kernel")}
        env.close()
    return out


def side_stress(n, torch, dev, peak_tf, steps=5, warmup=3):
    """BASELINE configs[4]: J2 + drag + eclipse + four-wheel pyramid with momentum dumping, 65536 envs per GPU, FP64 and
    the mixed-precision build (precision = 1), with the deviation of the mixed trajectories from the FP64 ones after the
    timed steps (same initial conditions, same actions, no auto-reset so that the envs stay comparable)."""
    from basilisk_env_b200.vec_env import LeoPowerAttVecEnv
    from basilisk_env_b200 import _native
    F = lambda name: _native.state_field(name)[0]      # noqa: E731
    g = torch.Generator(device=dev).manual_seed(99)
    acts = torch.randint(0, 3, (steps + warmup, n), dtype=torch.int32, device=dev, generator=g)
    out, states = {"envs": n, "config": "use_j2=1, rw_set=1 (four-wheel pyramid), i.i.d. actions {0,1,2}"}, {}
    for prec, key in ((0, "fp64"), (1, "mixed")):
        env = LeoPowerAttVecEnv(n, device=dev.index, seed=17, use_j2=1, rw_set=1, precision=prec)
        env.reset()
        total_ms, per, _ = time_device_steps(env, acts, steps, warmup, torch, None, 1)
        ms = float(np.mean(per))
        flops = env.flops_per_step()
        tf = flops * n / (ms * 1e-3) / 1e12
        d, i = env.get_state()
        states[key] = (d.clone(), i.clone(), env.done.clone())
        out[key] = {"value": n * steps / (total_ms * 1e-3), "unit": UNIT, "ms_per_step": total_ms / steps, "kernel": env.kernel_name()}
        if prec == 0:
            out[key]["roofline"] = {"bound": "fp64", "achieved": tf, "peak": peak_tf, "unit": "TFLOP/s",
                                    "frac": tf / peak_tf if peak_tf else None, "kernel_ms": ms, "flop_per_env_step": flops}
        env.close()
    # steady state, as the headline measures it: auto-reset on, i.i.d. actions, a longer warm-up (the first intervals after a common
    # reset are slower: every env spins its wheels up at once); the no-reset runs above exist for the precision comparison
    env = LeoPowerAttVecEnv(n, device=dev.index, seed=17, use_j2=1, rw_set=1, auto_reset=True)
    env.reset()
    acts2 = torch.randint(0, 3, (13, n), dtype=torch.int32, device=dev, generator=g)
    total_ms, per, _ = time_device_steps(env, acts2, steps, 8, torch, None, 1)
    ms = float(np.mean(per))
    tf = env.flops_per_step() * n / (ms * 1e-3) / 1e12
    out["fp64_steady_state"] = {"value": n * steps / (total_ms * 1e-3), "unit": UNIT, "ms_per_step": total_ms / steps, "kernel": env.kernel_name(),
                                "warmup": 8, "auto_reset": True,
                                "roofline": {"bound": "fp64", "achieved": tf, "peak": peak_tf, "unit": "TFLOP/s", "frac": tf / peak_tf if peak_tf else None}}
    env.close()
    d0, i0, dn0 = states["fp64"]; d1, i1, dn1 = states["mixed"]

    def q(x):
        x = x.flatten().double().cpu().numpy()
        return {"median": float(np.median(x)), "p99": float(np.percentile(x, 99))}
    out["speedup_mixed_over_fp64"] = out["fp64"]["ms_per_step"] / out["mixed"]["ms_per_step"]
    out["deviation_after_steps"] = steps + warmup
    out["deviation"] = {"position_m": q((d0[F("r_BN_N"):F("r_BN_N") + 3] - d1[F("r_BN_N"):F("r_BN_N") + 3]).norm(dim=0)),
                        "sigma_BN": q((d0[F("sigma_BN"):F("sigma_BN") + 3] - d1[F("sigma_BN"):F("sigma_BN") + 3]).abs().max(dim=0).values),
                        "wheel_rad_s": q((d0[F("Omega"):F("Omega") + 4] - d1[F("Omega"):F("Omega") + 4]).abs().max(dim=0).values),
                        "done_flags_equal_frac": float((dn0 == dn1).double().mean()),
                        "fire_counters_equal_frac": float((i0[F("fireCounter"):F("fireCounter") + 8] == i1[F("fireCounter"):F("fireCounter") + 8]).all(dim=0).double().mean())}
    return out


# --------------------------------------------------------------------------------------------------
# opNav env (BASELINE configs[3]): dynamics + nav measurement model + relative-OD filter, batched
# --------------------------------------------------------------------------------------------------
OPNAV_STATE_BYTES_PER_ENV = (83 + 14) * 8
OPNAV_H2D_BYTES_PER_ENV = 4
OPNAV_D2H_BYTES_PER_ENV = 4 * 8 + 8 + 1 + 1 + 12 * 8


def opnav_workload_name(n):
    return (f"opNav env, {n} envs on one GPU (BASELINE configs[3]; {n / 56832:.2f} resident sets of 148 SMs x 3 blocks x 128 threads): Mars orbits from the reference's element ranges, filter "
            "initial error U(+-1e5 m, +-1e3 m/s), simple_nav noise on, one synthetic circle measurement per 60 s while imaging, "
            "i.i.d. uniform actions {0,1}, camera re-enabled by action 0, auto-reset, FP64; one step = 50 min = 3000 ticks")


def opnav_cpu_arm(envs_per_core, seconds, threads=None, fixed_steps=None, build="fast"):
    from oracle import opnav as on
    from tests import opnav_parity as par
    threads = threads or host_threads()
    n = envs_per_core * threads
    rows = par.sample_rows(on, n, seed=7)
    batch = on.OpNavEnvBatch(rows, on.default_cfg(seed=5, camera_reenable=1), L=on.lib(fast=(build == "fast")))
    rng = np.random.RandomState(3)
    batch.step(rng.randint(0, 2, n), nthreads=threads)
    steps, t0 = 0, time.perf_counter()
    while True:
        batch.step(rng.randint(0, 2, n), nthreads=threads)
        steps += 1
        el = time.perf_counter() - t0
        if (fixed_steps is not None and steps >= fixed_steps) or (fixed_steps is None and el >= seconds):
            break
    return {"value": n * steps / el, "unit": UNIT, "cores": threads, "kind": "port", "ms_per_step": el / steps * 1e3,
            "build_flags": CPU_BUILDS[build],
            "sample": f"{n} envs x {steps} decision steps (oracle/opnav_oracle.c, gcc {CPU_BUILDS[build].split(' (')[0]}, OpenMP over envs, "
                      f"{threads} threads, {el:.1f} s)"}


def opnav_traffic(n):
    """DRAM bytes per decision interval (both opNav kernels) from the latest `ncu --set full` captures (profiles/traffic_opnav.json,
    of a launch with the same env count); None for any other size."""
    try:
        j = json.load(open(os.path.join(ROOT, "profiles", "traffic_opnav.json")))
        return j.get("dram_bytes_per_launch") if (j.get("envs") or 32768) == n else None
    except (OSError, ValueError):
        return None


def side_opnav(n, torch, dev, peak_tf, steps=3, warmup=3, cpu_seconds=4.0):
    from basilisk_env_b200.opnav_env import OpNavVecEnv
    env = OpNavVecEnv(n, device=dev.index, seed=5, auto_reset=True, sample_orbit=1, camera_reenable=1)
    env.reset()
    acts = torch.randint(0, 2, (steps + warmup, n), dtype=torch.int32, device=dev)
    acts_host = acts.cpu().numpy()
    l0 = env.launch_count()
    total_ms, per, _ = time_device_steps(env, acts, steps, warmup, torch, None, 1)
    act_pinned, outs = env.host_buffers()             # page-locked, device-mapped: the kernels read / write them in place
    act_pinned[:] = acts_host[0]
    env.step_host(act_pinned, outs)
    torch.cuda.synchronize()
    e0 = time.perf_counter()
    for t in range(steps):
        act_pinned[:] = acts_host[warmup + t]         # the trainer's actions of this step (host memory)
        env.step_host(act_pinned, outs)
    e2e_ms = (time.perf_counter() - e0) * 1e3 / steps
    per_step = (env.launch_count() - l0) // (warmup + steps + 1 + steps)    # kernels per decision step (two passes: two launches)
    launches = per_step * 2 * steps                                          # device-timed + host-buffer steps of the timed regions
    stats = env.episode_stats()
    flops = env.flops_per_step()
    env.close()
    ms = float(np.mean(per))
    tf = flops * n / (ms * 1e-3) / 1e12
    # the decision interval is two kernels (noise + dynamics, then the filter): the interval's measurements (one per camera frame:
    # tick, obs[3], R[6]) and an 8-double header cross in a global buffer, written once and read once; the dynamics side of the
    # state is read by both (the second pass needs position / velocity / attitude for the observation)
    meas_bytes = (8 + 10 * (3000 // 60 + 1)) * 8
    alg_bytes = (2 * OPNAV_STATE_BYTES_PER_ENV + 2 * meas_bytes + OPNAV_H2D_BYTES_PER_ENV + OPNAV_D2H_BYTES_PER_ENV) * n
    out = {"workload": opnav_workload_name(n), "envs": n, "value": n * steps / (total_ms * 1e-3), "unit": UNIT,
           "ms_per_step": total_ms / steps, "steps": steps, "warmup": warmup, "ticks_per_step": 3000,
           "roofline": {"bound": "fp64", "achieved": tf, "peak": peak_tf, "unit": "TFLOP/s", "frac": tf / peak_tf if peak_tf else None,
                        "kernel": "opnav_pass1_kernel + opnav_pass2_kernel (one decision interval)", "kernel_ms": ms, "flop_per_env_step": flops,
                        "flop_source": "operation list of opnav_core.cuh (bskenv_opnav_flops_per_step; DESIGN.md), within 1 % of the executed "
                                       "2*DFMA+DMUL+DADD count of ncu (profiles/ncu_opnav_p1_r02c.md + ncu_opnav_p2_r02c.md: 17.71e6 per env-step)",
                        "algorithmic_bytes_per_launch": alg_bytes},
           "e2e": {"value": n / (e2e_ms * 1e-3), "unit": UNIT, "ms_per_step": e2e_ms, "h2d_bytes_per_step": OPNAV_H2D_BYTES_PER_ENV * n,
                   "d2h_bytes_per_step": OPNAV_D2H_BYTES_PER_ENV * n,
                   "api": "bskenv_opnav_step_host with page-locked host buffers (env.host_buffers)"},
           "gpu_launches": int(launches), "episode_stats": stats, "checksum": float(outs[0].sum())}
    # the opt-in three-kernel interval (noise walk in a kernel of its own, 120 B of device buffer per env-tick; DESIGN.md 6b (iv)):
    # same actions, same results bit for bit -- measured beside the default, not the headline
    prev = os.environ.get("BSKENV_OPNAV_NOISE_SPLIT")
    os.environ["BSKENV_OPNAV_NOISE_SPLIT"] = "1"
    try:
        env = OpNavVecEnv(n, device=dev.index, seed=5, auto_reset=True, sample_orbit=1, camera_reenable=1)
        env.reset()
        l0 = env.launch_count()
        t_ms, per3, _ = time_device_steps(env, acts, steps, warmup, torch, None, 1)
        k3 = (env.launch_count() - l0) // (warmup + steps)
        out["three_kernel_interval"] = {"value": n * steps / (t_ms * 1e-3), "unit": UNIT, "ms_per_step": t_ms / steps, "kernels_per_step": int(k3),
                                        "noise_buffer_bytes": 15 * 8 * 3001 * ((n + 31) // 32 * 32) if k3 == 3 else 0,
                                        "enabled_by": "BSKENV_OPNAV_NOISE_SPLIT=1 (falls back to two kernels when the buffer does not fit)"}
        env.close()
    finally:
        if prev is None:
            del os.environ["BSKENV_OPNAV_NOISE_SPLIT"]
        else:
            os.environ["BSKENV_OPNAV_NOISE_SPLIT"] = prev
    if cpu_seconds > 0:
        cb = opnav_cpu_arm(2, cpu_seconds)
        out["cpu_baseline"] = {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample", "build_flags")}
    return out


def run_opnav(args):
    """The full JSON line for the opNav workload (N = 1)."""
    import torch
    from basilisk_env_b200.vec_env import fp64_peak_tflops
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (the environment step has no CPU path)")
    torch.cuda.set_device(0)
    dev = torch.device("cuda", 0)
    peak_tf = fp64_peak_tflops(0, 0.5)
    sampler = ClockSampler(0)
    t0 = time.perf_counter()
    r = side_opnav(args.opnav_envs, torch, dev, peak_tf, steps=args.steps, warmup=max(args.warmup, 3),
                   cpu_seconds=0.0 if args.no_cpu_baseline else args.cpu_seconds)
    clocks = sampler.stop(t0, time.perf_counter())
    n = args.opnav_envs
    line = {"metric": METRIC, "value": r["value"], "unit": UNIT, "n_gpus": 1, "steps": r["steps"], "warmup": r["warmup"],
            "ms_per_step": r["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
            "data": "synthetic",
            "config": {"workload": r["workload"], "envs_per_gpu": n, "ticks_per_step": 3000,
                       "l2": f"{(OPNAV_STATE_BYTES_PER_ENV + 12 * 8) * n / 2**20:.0f} MiB of per-env state, touched once per launch; "
                             "the kernel is FP64-pipe / latency bound, not memory bound"},
            "roofline": dict(r["roofline"], traffic=opnav_traffic(n)), "e2e": r["e2e"], "gpu_launches": r["gpu_launches"], "clocks": clocks,
            "episode_stats": r["episode_stats"], "checksum": r["checksum"], "cpu_baseline": r.get("cpu_baseline")}
    print(json.dumps(line), flush=True)


if __name__ == "__main__":
    main()
