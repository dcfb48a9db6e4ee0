"""Scheduled staircase (robustness map) throughput against the plain fused rollout of the same number of steps.

    python examples/bench_scripts/staircase_bench.py [--reps 5] [--arm all|response|gains]

Cases (env-steps/s = envs x K x L / time, CUDA events, after a warm-up launch of every shape):
  wt  2^20 envs, Modular-256 actor, staircase 3, 6, 9, 4, 2 x 500 steps
  ph  2^23 envs, Modular-128 actor, staircase 10, 6, 3, 8, 5 x 50 steps
For each case: scenarios.staircase_metrics on a ready env (the scheduled launch; metrics only), the same launch with a
[K, n] per-env set-point matrix (every column the shared staircase, so the two launches do the same work and differ by
the set-point load alone), and the deterministic vec.rollout of the same K L steps without replay rows (the ceiling: same
kernel without the segment logic), alternated rep by rep, and scenarios.robust_map end to end (env construction, reset,
parameters, launch).
Then the clipped linear baseline (policy='linear'), metrics only: the fused map of the water tank in f32 at 2^23 envs and
in f64 at 2^20 envs (5 x 500 steps), against the per-step loop of scenarios.staircase(policy='linear') (prior kernel +
step kernel per step, trajectories kept) at 2^18 envs.  The f32 rate is set against the MUFU ceiling of the plant: 40
sqrt per env-step (20 Euler sub-steps x 2 tanks) at 16 MUFU ops / clk / SM, 148 SMs and 1.8 GHz = 1.07e11 env-steps/s.
Then the step response (--arm response runs this arm alone): the metrics-only launch with and without response=True
(settle, rise, effort, peak action per env and segment, the Tracked kernels), alternated rep by rep, for the agent on the
water tank (2^20 envs, Modular-256, 5 x 500 steps) and pH (2^23 envs, Modular-128, 5 x 50 steps) and for the linear
baseline in f32 on the water tank (2^23 envs, 5 x 500 steps).
Then per-env controller gains (--arm gains runs this arm alone): the step-response launch with one shared K against the
gain launch whose [S, n] K matrix has that K in every column (the same work), alternated rep by rep, median of the reps,
on the same three shapes; and one real gain x plant map, 64 x 64 (kp, ki) integrator gains x 2048 (a1, a2, Kp) rows =
2^23 envs, linear f32, 5 x 500 steps, with the step response.
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
    matrix = torch.tensor(setpoints, dtype=torch.float64, device="cuda")[:, None].expand(len(setpoints), n).contiguous()
    per_env = lambda: SC.staircase_metrics(env, K, actor=pack, setpoints=matrix, steps=steps)   # noqa: E731
    plain = lambda: env.rollout(T, priorK, actor=pack, deterministic=True)                      # noqa: E731
    rmap = lambda: SC.robust_map(K, params, actor=pack, plant=plant, steps=steps, setpoints=setpoints)  # noqa: E731
    for f in (sched, per_env, plain, rmap):   # warm-up
        f()
    torch.cuda.synchronize()
    ts, te, tp, tm = [], [], [], []
    for _ in range(reps):
        ts.append(timed(sched))
        te.append(timed(per_env))
        tp.append(timed(plain))
    for _ in range(max(1, reps // 2)):
        tm.append(timed(rmap))
    env.check_status()
    steps_total = n * T
    s, e, p, m = np.median(ts), np.median(te), np.median(tp), np.median(tm)
    print(f"{name}: n={n} H={H} K={len(setpoints)} L={steps}")
    print(f"  scheduled launch (staircase_metrics) {s * 1e3:9.2f} ms  {steps_total / s:.3e} env-steps/s  "
          f"(min {min(ts) * 1e3:.2f}, max {max(ts) * 1e3:.2f} ms)")
    print(f"  per-env set-points [K, n]            {e * 1e3:9.2f} ms  {steps_total / e:.3e} env-steps/s  "
          f"(min {min(te) * 1e3:.2f}, max {max(te) * 1e3:.2f} ms)")
    print(f"  per-env / shared time                {e / s:9.4f}")
    print(f"  plain deterministic rollout          {p * 1e3:9.2f} ms  {steps_total / p:.3e} env-steps/s  "
          f"(min {min(tp) * 1e3:.2f}, max {max(tp) * 1e3:.2f} ms)")
    print(f"  scheduled / plain time               {s / p:9.4f}")
    print(f"  robust_map end to end                {m * 1e3:9.2f} ms  {steps_total / m:.3e} env-steps/s", flush=True)
    del env
    torch.cuda.empty_cache()


MUFU_CEILING = 16 * 148 * 1.8e9 / 40   # env-steps/s of the f32 water tank: 40 sqrt per env-step


def linear_case(reps):
    K = [0.0, 0.4, -0.4, 0.0]
    setpoints, steps = SC.WT_INTEGRATOR_SETPOINTS, 500
    T = len(setpoints) * steps
    for dtype, n in ((torch.float32, 1 << 23), (torch.float64, 1 << 20)):
        env = V.WaterTankVec(n, dtype=dtype)
        env.reset()
        fused = lambda: SC.staircase_metrics(env, K, setpoints=setpoints, steps=steps, policy="linear")   # noqa: E731
        fused()
        t = [timed(fused) for _ in range(reps)]
        env.check_status()
        f = np.median(t)
        line = f"  fused linear map {str(dtype)[6:]:8s} n=2^{n.bit_length() - 1}  {f * 1e3:9.2f} ms  {n * T / f:.3e} env-steps/s"
        if dtype == torch.float32:
            line += f"  ({n * T / f / MUFU_CEILING:.1%} of the 1.07e11 MUFU ceiling)"
        print(line + f"  (min {min(t) * 1e3:.2f}, max {max(t) * 1e3:.2f} ms)", flush=True)
        del env
        torch.cuda.empty_cache()
    n = 1 << 18
    env = V.WaterTankVec(n)
    env.reset()
    loop = lambda: SC.staircase(env, "linear", K, setpoints=setpoints, steps=steps)   # noqa: E731
    loop()
    t = [timed(loop) for _ in range(max(1, reps // 2))]
    lp = np.median(t)
    print(f"  per-step linear loop float32 n=2^18  {lp * 1e3:9.2f} ms  {n * T / lp:.3e} env-steps/s", flush=True)


def response_arm(reps):
    """metrics only, with and without the step response, alternated rep by rep in the same env"""
    runs = (("wt agent  Modular-256 f32", "wt", 1 << 20, 256, 500, SC.WT_INTEGRATOR_SETPOINTS, [0.0, 0.4, -0.4, 0.0], "agent"),
            ("ph agent  Modular-128 f32", "ph", 1 << 23, 128, 50, SC.PH_SETPOINTS, [-0.02, 0.02, 0.035], "agent"),
            ("wt linear f32            ", "wt", 1 << 23, 0, 500, SC.WT_INTEGRATOR_SETPOINTS, [0.0, 0.4, -0.4, 0.0], "linear"))
    for name, plant, n, H, steps, setpoints, K, policy in runs:
        pack = modular_pack(4 if plant == "wt" else 3, H) if policy == "agent" else None
        env = V.WaterTankVec(n) if plant == "wt" else V.PHVec(n)
        env.reset()
        kw = dict(actor=pack, setpoints=setpoints, steps=steps, policy=policy)
        without = lambda: SC.staircase_metrics(env, K, **kw)                  # noqa: E731
        with_r = lambda: SC.staircase_metrics(env, K, response=True, **kw)    # noqa: E731
        without()
        with_r()
        torch.cuda.synchronize()
        t0, t1 = [], []
        for _ in range(reps):
            t0.append(timed(without))
            t1.append(timed(with_r))
        env.check_status()
        a, b = np.median(t0), np.median(t1)
        steps_total = n * len(setpoints) * steps
        print(f"  {name} n=2^{n.bit_length() - 1} K={len(setpoints)} L={steps}: metrics {a * 1e3:9.2f} ms "
              f"({steps_total / a:.3e} env-steps/s, min {min(t0) * 1e3:.2f}, max {max(t0) * 1e3:.2f}), with response "
              f"{b * 1e3:9.2f} ms ({steps_total / b:.3e}, min {min(t1) * 1e3:.2f}, max {max(t1) * 1e3:.2f}); "
              f"with / without {b / a:.4f}", flush=True)
        del env
        torch.cuda.empty_cache()


def gains_arm(reps):
    """metrics-only launches with the step response: shared K against a K matrix of equal columns, alternated rep by rep"""
    runs = (("wt agent  Modular-256 f32", "wt", 1 << 20, 256, 500, SC.WT_INTEGRATOR_SETPOINTS, [0.0, 0.4, -0.4, 0.0], "agent"),
            ("ph agent  Modular-128 f32", "ph", 1 << 23, 128, 50, SC.PH_SETPOINTS, [-0.02, 0.02, 0.035], "agent"),
            ("wt linear f32            ", "wt", 1 << 23, 0, 500, SC.WT_INTEGRATOR_SETPOINTS, [0.0, 0.4, -0.4, 0.0], "linear"))
    for name, plant, n, H, steps, setpoints, K, policy in runs:
        pack = modular_pack(4 if plant == "wt" else 3, H) if policy == "agent" else None
        env = V.WaterTankVec(n) if plant == "wt" else V.PHVec(n)
        env.reset()
        Kmat = torch.tensor(K, dtype=torch.float64, device="cuda")[:, None].expand(len(K), n).contiguous()
        kw = dict(actor=pack, setpoints=setpoints, steps=steps, policy=policy, response=True)
        shared = lambda: SC.staircase_metrics(env, K, **kw)        # noqa: E731
        per_env = lambda: SC.staircase_metrics(env, Kmat, **kw)    # noqa: E731
        shared()
        per_env()
        torch.cuda.synchronize()
        t0, t1 = [], []
        for _ in range(reps):
            t0.append(timed(shared))
            t1.append(timed(per_env))
        env.check_status()
        a, b = np.median(t0), np.median(t1)
        steps_total = n * len(setpoints) * steps
        print(f"  {name} n=2^{n.bit_length() - 1} K={len(setpoints)} L={steps}: shared K {a * 1e3:9.2f} ms "
              f"({steps_total / a:.3e} env-steps/s, min {min(t0) * 1e3:.2f}, max {max(t0) * 1e3:.2f}), per-env K "
              f"{b * 1e3:9.2f} ms ({steps_total / b:.3e}, min {min(t1) * 1e3:.2f}, max {max(t1) * 1e3:.2f}); "
              f"per-env / shared {b / a:.4f}", flush=True)
        del env, Kmat
        torch.cuda.empty_cache()
    # the map: u = kp (r - h2) + ki I, i.e. K = [0, kp, -kp, -ki], gain g on plant rows g m .. g m + m - 1
    rng = np.random.default_rng(2)
    m, steps, setpoints = 2048, 500, SC.WT_INTEGRATOR_SETPOINTS
    P = np.stack([rng.uniform(0.0015, 0.0024, m), rng.uniform(0.0015, 0.0024, m), rng.uniform(0.07, 0.17, m)], 1)
    kp, ki = np.meshgrid(np.linspace(0.05, 1.0, 64), np.linspace(0.0, 0.05, 64), indexing="ij")
    Kg = np.stack([0 * kp, kp, -kp, -ki]).reshape(4, -1)
    Kmap = torch.as_tensor(np.repeat(Kg, m, axis=1), device="cuda")
    params = np.tile(P, (Kg.shape[1], 1))
    n = params.shape[0]
    env = V.WaterTankVec(n, max_step=steps)
    env.reset()
    env.reset_changable_parameters(torch.as_tensor(params[:, 0]), torch.as_tensor(params[:, 1]), torch.as_tensor(params[:, 2]))
    run = lambda: SC.staircase_metrics(env, Kmap, setpoints=setpoints, steps=steps, policy="linear", response=True)  # noqa: E731
    res = run()
    t = [timed(run) for _ in range(reps)]
    env.check_status()
    f = np.median(t)
    settled = (res["settle"] < steps).double().mean().item()
    print(f"  gain map 64 x 64 (kp, ki) x {m} plants = 2^{n.bit_length() - 1} envs, linear f32, K=5 L={steps}: "
          f"{f * 1e3:9.2f} ms  {n * len(setpoints) * steps / f:.3e} env-steps/s (min {min(t) * 1e3:.2f}, "
          f"max {max(t) * 1e3:.2f} ms); {settled:.1%} of the segments settle inside 2 %", flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--arm", choices=("all", "response", "gains"), default="all")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "needs a CUDA device"
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    print("GPU:", q.stdout.strip().splitlines()[0] if q.returncode == 0 else torch.cuda.get_device_name(0), flush=True)
    if args.arm == "response":
        print("step response: metrics-only launch without / with response=True", flush=True)
        response_arm(args.reps)
        return
    if args.arm == "gains":
        print("per-env gains: step-response launch with a shared K / with a [S, n] K matrix of equal columns", flush=True)
        gains_arm(args.reps)
        return
    rng = np.random.default_rng(1)
    n = 1 << 20
    wt_params = np.stack([rng.uniform(0.0015, 0.0024, n), rng.uniform(0.0015, 0.0024, n), rng.uniform(0.07, 0.17, n)], 1)
    case("wt robust map", "wt", n, 256, 500, SC.WT_INTEGRATOR_SETPOINTS, [0.0, 0.4, -0.4, 0.0], wt_params, args.reps)
    n = 1 << 23
    ph_params = np.stack([rng.uniform(0.005, 0.015, n), rng.uniform(0.0015, 0.0025, n)], 1)
    case("ph robust map", "ph", n, 128, 50, SC.PH_SETPOINTS, [-0.02, 0.02, 0.035], ph_params, args.reps)
    del wt_params, ph_params
    print("wt linear baseline: K=5 L=500, metrics only", flush=True)
    linear_case(args.reps)
    print("step response: metrics-only launch without / with response=True", flush=True)
    response_arm(args.reps)
    print("per-env gains: step-response launch with a shared K / with a [S, n] K matrix of equal columns", flush=True)
    gains_arm(args.reps)


if __name__ == "__main__":
    main()
