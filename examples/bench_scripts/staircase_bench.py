"""Scheduled staircase (robustness map) throughput against the plain fused rollout of the same number of steps.

    python examples/bench_scripts/staircase_bench.py [--reps 5]

Cases (env-steps/s = envs x K x L / time, CUDA events, after a warm-up launch of every shape):
  wt  2^20 envs, Modular-256 actor, staircase 3, 6, 9, 4, 2 x 500 steps
  ph  2^23 envs, Modular-128 actor, staircase 10, 6, 3, 8, 5 x 50 steps
For each case: scenarios.staircase_metrics on a ready env (the scheduled launch; metrics only), the deterministic
vec.rollout of the same K L steps without replay rows (the ceiling: same kernel without the segment logic), alternated
rep by rep, and scenarios.robust_map end to end (env construction, reset, parameters, launch).
Prints the GPU name and power limit of the run first.
"""
import argparse
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
import pime_b200.scenarios as SC   # noqa: E402
import pime_b200.vec as V          # noqa: E402


def modular_pack(S, H, seed=0):
    rng = np.random.default_rng(seed)
    sd = {}
    for name, o, i in [("other_net.0", H, S - 1), ("other_net.2", H // 2, H), ("integrator_net.0", H, 1),
                       ("integrator_net.2", H // 2, H), ("net.0", H, H), ("net.2", 1, H)]:
        b = 1.0 / np.sqrt(i)
        sd[name + ".weight"] = rng.uniform(-b, b, (o, i)).astype(np.float32)
        sd[name + ".bias"] = rng.uniform(-b, b, o).astype(np.float32)
    return V.ActorPack("modular", S, H, 1).update(sd)


def timed(fn):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) * 1e-3


def case(name, plant, n, H, steps, setpoints, K, params, reps):
    pack = modular_pack(4 if plant == "wt" else 3, H)
    env = V.WaterTankVec(n) if plant == "wt" else V.PHVec(n)
    env.reset()
    T = len(setpoints) * steps
    priorK = -np.asarray(K, np.float64)[:env.state_dim]
    sched = lambda: SC.staircase_metrics(env, K, actor=pack, setpoints=setpoints, steps=steps)   # noqa: E731
    plain = lambda: env.rollout(T, priorK, actor=pack, deterministic=True)                      # noqa: E731
    rmap = lambda: SC.robust_map(K, params, actor=pack, plant=plant, steps=steps, setpoints=setpoints)  # noqa: E731
    for f in (sched, plain, rmap):   # warm-up
        f()
    torch.cuda.synchronize()
    ts, tp, tm = [], [], []
    for _ in range(reps):
        ts.append(timed(sched))
        tp.append(timed(plain))
    for _ in range(max(1, reps // 2)):
        tm.append(timed(rmap))
    env.check_status()
    steps_total = n * T
    s, p, m = np.median(ts), np.median(tp), np.median(tm)
    print(f"{name}: n={n} H={H} K={len(setpoints)} L={steps}")
    print(f"  scheduled launch (staircase_metrics) {s * 1e3:9.2f} ms  {steps_total / s:.3e} env-steps/s  "
          f"(min {min(ts) * 1e3:.2f}, max {max(ts) * 1e3:.2f} ms)")
    print(f"  plain deterministic rollout          {p * 1e3:9.2f} ms  {steps_total / p:.3e} env-steps/s  "
          f"(min {min(tp) * 1e3:.2f}, max {max(tp) * 1e3:.2f} ms)")
    print(f"  scheduled / plain time               {s / p:9.4f}")
    print(f"  robust_map end to end                {m * 1e3:9.2f} ms  {steps_total / m:.3e} env-steps/s", flush=True)
    del env
    torch.cuda.empty_cache()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "needs a CUDA device"
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    print("GPU:", q.stdout.strip().splitlines()[0] if q.returncode == 0 else torch.cuda.get_device_name(0), flush=True)
    rng = np.random.default_rng(1)
    n = 1 << 20
    wt_params = np.stack([rng.uniform(0.0015, 0.0024, n), rng.uniform(0.0015, 0.0024, n), rng.uniform(0.07, 0.17, n)], 1)
    case("wt robust map", "wt", n, 256, 500, SC.WT_INTEGRATOR_SETPOINTS, [0.0, 0.4, -0.4, 0.0], wt_params, args.reps)
    n = 1 << 23
    ph_params = np.stack([rng.uniform(0.005, 0.015, n), rng.uniform(0.0015, 0.0025, n)], 1)
    case("ph robust map", "ph", n, 128, 50, SC.PH_SETPOINTS, [-0.02, 0.02, 0.035], ph_params, args.reps)


if __name__ == "__main__":
    main()
