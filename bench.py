#!/usr/bin/env python
"""bench.py -- fused env-steps/s (plant + P/PI prior + float32 obs + residual actor) on N B200s.

    python bench.py --gpus 1 --steps 5 --warmup 3                 # this repo's CUDA path (default)
    python bench.py --impl reference --gpus 1 --steps 3 --warmup 1  # the reference algorithm on the host CPU cores

One bench "step" = one fused-rollout launch: every env of the shard advances T=200 env steps (one full
episode of NonLinearWaterTankChangingParamUniformGoalIntegrator-SquareDistance-v2 with the Modular-256 residual
actor, Philox process + exploration noise, replay rows written to HBM, in-kernel auto-reset with ensemble
resampling).  Workload = BASELINE.json configs[2] ("1M-env water-tank ensemble rollout ... on 1 B200");
for N > 1 each rank owns its own 2^20 envs (weak scaling, envs sharded by global env id, no data-path
collective; one NCCL all-reduce of the 8-double episode statistics per step).

    python bench.py --workload ph    # configs[3]: pH plant, 2^23 envs over the ranks, T=50, Modular-128 (not the bench line)

Prints ONE JSON line (rank 0).  --dump-outputs DIR also writes, as .npy files, what the last timed rollout computed (a
seeded sample of envs): the inputs are seeded, so two builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

METRIC = "fused env-steps/sec (plant+PI+actor)"
UNIT = "env-steps/s"
WORKLOADS = {
    "wt": dict(name="1M-env water-tank ensemble rollout, fused step+PI+actor (configs[2])", S=4, T=200, H=256, envs=1 << 20,
               env="NonLinearWaterTankChangingParamUniformGoalIntegrator-SquareDistance-v2", K=[0.0, 0.4, -0.4, 0.0], sqrt=40),
    "ph": dict(name="pH ensemble sweep, 8M envs sharded by ensemble member (configs[3])", S=3, T=50, H=128, envs=1 << 23,
               env="PH1DChangingParamUniformGoalIntegrator-SqaureDistance-v35", K=[-0.02, 0.02, 0.035], sqrt=0),
    "wts10": dict(name="water-tank Stacking10 + ResidualPPO-256 (the network of run_watertank_changing.sh, configs[0]) at 2^19 envs", S=30, T=200,
                  H=256, envs=1 << 19, env="NonLinearWaterTankChangingParamUniformGoalStacking10-SquareDistance-v2",
                  K=[0.0] * 27 + [0.0, 0.4, -0.4], sqrt=40, kind="plain"),
    "train": dict(name="full PIME residual actor-critic training, GPU-resident replay, grad allreduce (configs[4])", S=4, T=200, H=256,
                  envs=1 << 16, env="NonLinearWaterTankChangingParamUniformGoalIntegrator-SquareDistance-v2",
                  K=[0.0, 0.4, -0.4, 0.0], sqrt=40),
}

FLOPS_PER_STEP = {("modular", 256, 4): 264704, ("modular", 128, 3): 66560, ("plain", 256, 30): 278016}  # 2 x weights, SURVEY 8a d4/d5
TANH_PER_STEP = {("modular", 256, 4): 1025, ("modular", 128, 3): 513, ("plain", 256, 30): 769}
# dram__bytes_read.sum + dram__bytes_write.sum of ONE launch (ncu --set full), keyed by (workload, envs, T); see profiles/
NCU_DRAM_BYTES_PER_LAUNCH = {("wt", 1 << 20, 200): 6.7555e9}   # profiles/r02_ncu_summary.md (algorithmic: 6.71e9 replay rows)
NCU_DRAM_BYTES_STEP = {"wt": 1.8658e9, "ph": 2.2754e9}   # wt_step_vec4_kernel / ph_step_kernel<float>, 2^25 envs (algorithmic 1.913e9 / 2.315e9), profiles/r02_ncu_summary.md
WT_STEP_BYTES_F32 = 57   # SURVEY 8d: 36 B read + 21 B written per env-step, SoA fp32
PH_STEP_BYTES_F32 = 69   # x, A, B are fp64 in the float flavour: read x8 r4 I4 A8 B8 C4 a4 t4 = 44, write x8 y4 I4 t4 rew4 done1 = 25


def parse():
    p = argparse.ArgumentParser()
    p.add_argument("--gpus", type=int, default=1)
    p.add_argument("--steps", type=int, default=5)
    p.add_argument("--warmup", type=int, default=3)
    p.add_argument("--impl", default="b200", choices=["b200", "reference"])
    p.add_argument("--workload", default="wt", choices=sorted(WORKLOADS))
    p.add_argument("--envs", type=int, default=0, help="envs per GPU (default: 2^20 for wt, 2^23 / world for ph)")
    p.add_argument("--T", type=int, default=0, help="env steps per launch (default: one episode)")
    p.add_argument("--net-dim", type=int, default=0)
    p.add_argument("--no-cpu-baseline", action="store_true")
    p.add_argument("--no-aux", action="store_true", help="skip the stand-alone step-kernel roofline measurements")
    p.add_argument("--no-extra", action="store_true", help="skip the configs[3] / configs[4] measurements that follow the headline")
    p.add_argument("--cpu-seconds", type=float, default=12.0)
    p.add_argument("--batch-size", type=int, default=1 << 17, help="train workload: PPO minibatch rows")
    p.add_argument("--repeat-times", type=int, default=2, help="train workload: PPO epochs over the buffer")
    p.add_argument("--tf32", action="store_true", help="train workload: TF32 cuBLAS GEMMs in the learner (default: fp32 like the reference)")
    p.add_argument("--dump-outputs", metavar="DIR", default=None,
                   help="after the timed steps, write what the last timed rollout returned (replay rows and final env state of a "
                        "fixed sample of envs, episode statistics) as DIR/<name>.npy")
    args = p.parse_args()
    if args.steps < 1:
        p.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl == "reference" or args.workload == "train"):
        p.error("--dump-outputs applies to the GPU rollout workloads (wt, ph, wts10)")
    return args


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        d = json.load(open(path))
        return dict(hbm=float(d["hbm_gbs"]), tf_burst=float(d["bf16_tflops"]), tf_sust=float(d.get("bf16_tflops_sustained", d["bf16_tflops"])),
                    sm_max=float(d.get("sm_max_mhz", 1965.0)), src="measured (MEASURED_PEAKS.json)")
    return dict(hbm=6650.0, tf_burst=1590.0, tf_sust=1400.0, sm_max=1965.0, src="fallback (B200_PROFILING.md)")


def actor_state_dict(H, S, seed=0, kind="modular"):
    """Modular actor at torch's default init scale; the last layer is N(0, 0.1^2) so that the MLP is not a numerical
    no-op (the reference zero-initialises it, which would make every product zero)."""
    rng = np.random.default_rng(seed)

    def lin(o, i):
        b = 1.0 / np.sqrt(i)
        return rng.uniform(-b, b, (o, i)).astype(np.float32), rng.uniform(-b, b, o).astype(np.float32)
    sd = {}
    if kind == "plain":
        for name, o, i in [("net.0", H, S), ("net.2", H, H), ("net.4", H, H), ("net.6", 1, H)]:
            sd[name + ".weight"], sd[name + ".bias"] = lin(o, i)
        sd["net.6.weight"] = rng.normal(0, 0.1, (1, H)).astype(np.float32)
    else:
        for name, o, i in [("other_net.0", H, S - 1), ("other_net.2", H // 2, H), ("integrator_net.0", H, 1),
                           ("integrator_net.2", H // 2, H), ("net.0", H, H), ("net.2", 1, H)]:
            sd[name + ".weight"], sd[name + ".bias"] = lin(o, i)
        sd["net.2.weight"] = rng.normal(0, 0.1, (1, H)).astype(np.float32)
    sd["a_std_log"] = np.array([[-0.5]], np.float32)
    return sd


# ------------------------------------------------------------------------------------------------ clocks sampler
class ClockSampler(threading.Thread):
    def __init__(self, index=0, period=0.05):
        super().__init__(daemon=True)
        self.index, self.period = index, period
        self.samples, self.reasons, self.power = [], set(), []
        self.sm_max = None
        self._stop_evt = threading.Event()
        self.ok = False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.sm_max = int(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self.ok = True
        except Exception:
            self.ok = False

    NAMES = {0x1: "gpu_idle", 0x2: "applications_clocks_setting", 0x4: "sw_power_cap", 0x8: "hw_slowdown", 0x10: "sync_boost",
             0x20: "sw_thermal_slowdown", 0x40: "hw_thermal_slowdown", 0x80: "hw_power_brake_slowdown", 0x100: "display_clock_setting"}

    def run(self):
        if not self.ok:
            return
        nv = self.nv
        while not self._stop_evt.is_set():
            try:
                self.samples.append(int(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
                self.power.append(nv.nvmlDeviceGetPowerUsage(self.h) / 1000.0)
                mask = int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h))
                for bit, name in self.NAMES.items():
                    if mask & bit and name != "gpu_idle":
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(self.period)

    def stop(self):
        self._stop_evt.set()
        self.join(timeout=2)
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.sm_max, "reasons": sorted(self.reasons), "samples": 0}
        return {"sm_mhz": float(np.median(self.samples)), "sm_max_mhz": self.sm_max, "reasons": sorted(self.reasons),
                "samples": len(self.samples), "power_w_max": max(self.power) if self.power else None}


# ------------------------------------------------------------------------------------------------ workload resolution
def resolve(args, world=1):
    w = dict(WORKLOADS[args.workload])
    w["H"] = args.net_dim or w["H"]
    w["T"] = args.T or w["T"]
    w["n"] = args.envs or (max(1, w["envs"] // world) if args.workload == "ph" else w["envs"])
    w.setdefault("kind", "modular")
    w["actor"] = ("ResidualIntegratorModularPPO-" if w["kind"] == "modular" else "ResidualPPO-") + str(w["H"])
    return w


def base_config(args, w):
    """The `config` object of the JSON line -- the same keys and values for the b200 arm and the reference arm."""
    n, T, S = w["n"], w["T"], w["S"]
    return {"workload": w["name"], "envs_per_gpu": n, "T": T, "actor": w["actor"], "env": w["env"],
            "noise_scale": 0.0 if args.workload == "ph" else 0.01,
            "policy": "stochastic (explore_env)", "replay": "GPU-resident, time-major [T,n,S]+[T,n,4] fp32",
            "l2": f"each step streams {n * T * (S + 4) * 4 / 1e9:.2f} GB of replay rows through L2 (>> 126 MB), "
                  "which flushes it between timed steps",
            "sharding": "contiguous env-id ranges per rank, Philox keyed by global env id"}


# ------------------------------------------------------------------------------------------------ CPU baseline
def cpu_baseline(w, seconds, sd):
    """The oracle (C restatement of the reference loop: fp64 plant + fp32 actor, oracle/pime_oracle.c) on all host
    cores: one thread per core, each running explore-style rollouts on its own slice of envs (ctypes releases the GIL)."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import pime_oracle as O
    O.build()
    cores = os.cpu_count() or 1
    H, S, T = w["H"], w["S"], w["T"]
    per = 16  # envs per thread per chunk
    acfg = O.ActorCfg(kind=1, state_dim=S, mid_dim=H, integrator_dim=1)
    params = O.pack_actor_params(sd, 1)
    priorK = -np.array(w["K"])
    is_wt = w["S"] == 4
    cfg = O.wt_cfg(reward_type="square_distance") if is_wt else O.ph_cfg()
    table = None if is_wt else O.ph_table()
    counts = [0] * cores
    deadline = [0.0]

    def work(tid):
        rng = np.random.default_rng(1000 + tid)
        while time.perf_counter() < deadline[0]:
            eps = rng.standard_normal((T, per)).astype(np.float32)
            I, t = np.zeros(per), np.zeros(per, np.int32)
            if is_wt:
                h1, h2, r = rng.uniform(0, 10, per), rng.uniform(0, 10, per), rng.uniform(0, 10, per)
                a1, a2, Kp = rng.uniform(0.0015, 0.0024, per), rng.uniform(0.0015, 0.0024, per), rng.uniform(0.07, 0.17, per)
                pn1, pn2 = rng.normal(0, 0.01, (T, per)), rng.normal(0, 0.01, (T, per))
                O.wt_rollout(cfg, acfg, params, -0.5, priorK, 1, 0, False, T, h1, h2, r, I, t, a1, a2, Kp, eps=eps, pn1=pn1, pn2=pn2)
            else:
                qww, qc = rng.uniform(0.005, 0.015, per), rng.uniform(0.0015, 0.0025, per)
                A, B, Cc = O.ph_update_system(qww, qc)
                x, r = rng.uniform(0, 50, per), rng.uniform(3, 11, per)
                y = table[np.rint(Cc * x * 1e5).astype(np.int64)]
                O.ph_rollout(cfg, table, acfg, params, -0.5, priorK, False, T, x, y, r, I, t, A, B, Cc, eps=eps)
            counts[tid] += per * T
    # warm-up (library load, page-in), then three samples of seconds / 3 (>= 4 s) each: the median is reported (SURVEY 8d)
    deadline[0] = time.perf_counter() + 0.5
    work(0)
    rates, totals, dts = [], [], []
    per_sample = max(seconds / 3.0, 4.0) if seconds >= 6.0 else seconds
    for _ in range(3 if seconds >= 6.0 else 1):
        for i in range(cores):
            counts[i] = 0
        t0 = time.perf_counter()
        deadline[0] = t0 + per_sample
        th = [threading.Thread(target=work, args=(i,)) for i in range(cores)]
        [x.start() for x in th]
        [x.join() for x in th]
        dts.append(time.perf_counter() - t0)
        totals.append(sum(counts))
        rates.append(totals[-1] / dts[-1])
    k = int(np.argsort(rates)[len(rates) // 2])
    total, dt = totals[k], dts[k]
    return {"value": rates[k], "unit": UNIT, "cores": cores, "kind": "port",
            "sample": f"median of {len(rates)} samples; this one: {total} env-steps ({total // T} episodes of T={T}, {'WT' if is_wt else 'pH'}-Integrator + "
                      f"Modular-{H} actor, fp64 plant / fp32 actor, C oracle, {cores} threads) in {dt:.1f} s"}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    w = resolve(args, int(os.environ.get("WORLD_SIZE", "1")))
    sd = actor_state_dict(w["H"], w["S"])
    vals = []
    for _ in range(max(1, args.warmup)):
        cpu_baseline(w, 1.0, sd)
    t0 = time.perf_counter()
    last = None
    for _ in range(max(1, args.steps)):
        last = cpu_baseline(w, max(2.0, min(args.cpu_seconds, 60.0 / max(1, args.steps))), sd)
        vals.append(last["value"])
    v = float(np.median(vals))
    last["value"] = v
    per_step_envsteps = v * (time.perf_counter() - t0) / max(1, args.steps)
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * (time.perf_counter() - t0) / max(1, args.steps),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64 plant / f32 actor",
            "data": "synthetic",
            "config": base_config(args, w),
            "note": "reference algorithm (C port of the numpy/torch loop) on all host cores; each step is a bounded "
                    f"sample (~{per_step_envsteps:.3g} env-steps) of the workload; value = median over the steps",
            "cpu_baseline": last,
            "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------ GPU arm

def time_e2e(step_fn, steps, world, units_per_step, barrier, dist):
    """Wall-clock of `steps` host-driven calls (each ends with a device->host read), max over ranks."""
    import torch
    step_fn()
    barrier()
    t0 = time.perf_counter()
    for _ in range(steps):
        step_fn()
    barrier()
    t = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return {"value": world * units_per_step * steps / float(t.item()), "unit": UNIT, "steps": steps}


def ph_e2e(env, actor, T, K, bs, bo, stats, steps, world, barrier, dist):
    """configs[3] end to end: PHVec.rollout_host -> pime_ph_rollout_host_f32 with pinned host state."""
    import torch
    n = env.n
    host = {k: getattr(env, k).detach().cpu().pin_memory() for k in env.HOST_FIELDS if k not in ("t",)}
    host["t"] = torch.zeros(n, dtype=torch.int32).pin_memory()
    ret_host = torch.empty(n, dtype=torch.float32).pin_memory()
    flat_host = actor.flat.detach().cpu().pin_memory()
    h2d = sum(v.numel() * v.element_size() for v in host.values()) + flat_host.numel() * 4
    d2h = n * 4 + n * (8 + 4 + 4 + 4) + 64

    def step():
        actor.flat.copy_(flat_host, non_blocking=True)
        actor.update_from_flat()
        out = env.rollout_host(host, T, -K, actor=actor, ep_return_host=ret_host, replay=(bs, bo), stats=stats)
        return float(out["stats"].cpu()[0])

    e = time_e2e(step, steps, world, n * T, barrier, dist)
    e.update({"h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
              "api": "PHVec.rollout_host -> pime_ph_rollout_host_f32 (pinned host state in, ep_return + final state out; copy-in / rollout / copy-out pipelined over env slices)"})
    return e


DUMP_BYTES = 48 << 20   # --dump-outputs writes well under 64 MB


def dump_outputs(path, env, bs, bo, stats):
    """What one rollout hands its caller: the replay rows [T, n, S] and [T, n, 4], the episode statistics and the float
    env state it leaves behind.  These are GBs at the default sizes, so a fixed, seeded sample of envs is written (every
    time step of each; the same envs for the same --envs)."""
    import torch
    T, n, S = bs.shape
    names = ["h1", "h2", "r", "I", "a1", "a2", "Kp"] if hasattr(env, "h1") else ["x", "y", "r", "I", "A", "B", "C", "qww_V", "qc_V"]
    state = {"env_" + k: getattr(env, k) for k in names + ["ep_return"]}      # [n] each
    if getattr(env, "frames", None) is not None:
        state["env_frames"] = env.frames                                       # [3 * num_stack, n]
    env_bytes = 4 * T * (S + 4) + sum(t.element_size() * t.numel() // n for t in state.values())
    m = min(n, max(1, DUMP_BYTES // env_bytes))
    idx = torch.as_tensor(np.sort(np.random.default_rng(0).choice(n, m, replace=False)), device=bs.device)
    out = {"buf_state": bs[:, idx], "buf_other": bo[:, idx], "stats": stats}
    out.update({k: t[..., idx] for k, t in state.items()})
    os.makedirs(path, exist_ok=True)
    for k, v in out.items():
        np.save(os.path.join(path, k + ".npy"), v.cpu().numpy())


def run_b200(args):
    import torch
    import torch.distributed as dist

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the pime_b200 hot path has no CPU fallback")
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    import pime_b200.vec as V

    pk = peaks()
    w = resolve(args, world)
    n, T, H, S = w["n"], w["T"], w["H"], w["S"]
    is_wt = args.workload == "wt"
    K = np.array(w["K"])
    kind = w["kind"]
    sd = actor_state_dict(H, S, kind=w["kind"])
    actor = V.ActorPack(w["kind"], S, H, 1).update(sd)
    if args.workload == "wts10":
        env = V.WaterTankVec(n, dtype=torch.float32, obs_mode="stacking", num_stack=10, reward_type="square_distance",
                             noise_scale=0.01, seed=0, env_offset=rank * n)
    elif is_wt:
        env = V.WaterTankVec(n, dtype=torch.float32, obs_mode="integrator", reward_type="square_distance", noise_scale=0.01,
                             seed=0, env_offset=rank * n)
    else:
        env = V.PHVec(n, dtype=torch.float32, seed=0, env_offset=rank * n)
    env.reset()
    # stand-alone step kernels (HBM rows of SURVEY 8d), each timed alone -- before the long rollout loop, i.e. in the same
    # burst state the HBM peak of MEASURED_PEAKS.json was measured in (the water-tank kernel is co-limited by its 40 MUFU.SQRT
    # per env-step, so its time follows the SM clock)
    aux = aux_step_rooflines(V, pk) if (rank == 0 and not args.no_aux and is_wt) else None
    bs = torch.empty((T, n, S), dtype=torch.float32, device="cuda")
    bo = torch.empty((T, n, 4), dtype=torch.float32, device="cuda")
    stats = torch.zeros(8, dtype=torch.float64, device="cuda")

    def step():
        stats.zero_()
        env.rollout(T, -K, actor=actor, auto_reset=True, replay=(bs, bo), stats=stats, gamma=0.99)
        if world > 1:
            dist.all_reduce(stats)  # episode-return statistics of the whole job (the path's only exchange)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    sampler = ClockSampler(local)   # NVML initialisation takes a rank-dependent 10-100 ms: keep it out of the timed region
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps + 1)]
    for _ in range(max(args.warmup, 0)):
        step()
    barrier()
    sampler.start()
    ev[0].record()
    for i in range(args.steps):
        step()
        ev[i + 1].record()
    barrier()
    clocks = sampler.stop()
    ms_total = ev[0].elapsed_time(ev[-1])
    kernel_ms = [ev[i].elapsed_time(ev[i + 1]) for i in range(args.steps)]
    tmax = torch.tensor([ms_total], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
    ms_total = float(tmax.item())
    value = world * n * T * args.steps / (ms_total * 1e-3)
    st = stats.cpu().numpy()
    env.check_status()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, env, bs, bo, stats)   # before the e2e calls below overwrite bs, bo, stats and the env

    # ---- e2e: the host-buffer API call (pinned host state in, ep_return out), H2D/D2H inside the timed region; timed over
    # args.steps calls directly after the device-timed loop (same clocks / thermal state, so the two numbers compare)
    e2e = None
    if is_wt:
        host = {k: getattr(env, k).detach().cpu().pin_memory() for k in ("h1", "h2", "r", "I", "a1", "a2", "Kp")}
        host["t"] = torch.zeros(n, dtype=torch.int32).pin_memory()
        host["episode"] = env.episode.detach().cpu().pin_memory()
        ret_host = torch.empty(n, dtype=torch.float32).pin_memory()
        flat_host = actor.flat.detach().cpu().pin_memory()
        h2d = sum(v.numel() * v.element_size() for v in host.values()) + flat_host.numel() * 4
        d2h = ret_host.numel() * 4 + 4 * n * 4 + 64

        def e2e_step():
            actor.flat.copy_(flat_host, non_blocking=True)           # actor weights from the (host-side) learner
            actor.update_from_flat()
            out = env.rollout_host(host, T, -K, actor=actor, ep_return_host=ret_host, replay=(bs, bo), stats=stats)
            return float(out["stats"].cpu()[0])                       # D2H of the step's metric (sum of episode returns)

        e2e = time_e2e(e2e_step, args.steps, world, n * T, barrier, dist)
        e2e.update({"h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                    "api": "WaterTankVec.rollout_host -> pime_wt_rollout_host_f32 (pinned host state in, ep_return + final state out; copy-in / rollout / copy-out pipelined over env slices)"})
    elif args.workload == "ph":
        e2e = ph_e2e(env, actor, T, K, bs, bo, stats, args.steps, world, barrier, dist)

    kname = f"rollout_kernel<{'PhGlue' if args.workload == 'ph' else 'WtGlue'}<float>, {kind}, {H}>"
    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_total / args.steps, "higher_is_better": True,
            "scaling": "strong" if (args.workload == "ph" and not args.envs) else "weak", "vs_baseline": None,
            "dtype": "f32 (plant, prior, obs, first and last actor layer; hidden layers: f16 tensor-core operands, f32 accumulate)",
            "data": "synthetic",
            "config": base_config(args, w),
            "clocks": clocks, "gpu_launches": args.steps,
            "episode_stats": {"mean_return": st[0] / max(st[2], 1), "episodes": st[2]}}
    if e2e:
        line["e2e"] = e2e

    extra = {}
    if is_wt and not args.no_extra and not (args.envs or args.T or args.net_dim):
        # configs[3] and configs[4] of BASELINE.json, measured in the same invocation (outside the timed region of the headline)
        # so that the driver's 1/2/4/8-GPU runs record them too
        del bs, bo
        if e2e is not None:
            del host, ret_host
        torch.cuda.empty_cache()
        extra["config4"] = extra_config4(V, world, rank, dist, barrier, pk)
        torch.cuda.empty_cache()
        extra["config5"] = extra_config5(world, rank, dist, barrier)
    if extra:
        line["extra"] = extra

    if rank == 0:
        flops = FLOPS_PER_STEP.get((kind, H, S))
        step_ms = float(np.mean(kernel_ms))
        if flops:
            ach = n * T * flops / (step_ms * 1e-3) / 1e12
            line["roofline"] = {"bound": "tensor", "achieved": ach, "peak": pk["tf_sust"], "unit": "TFLOP/s", "frac": ach / pk["tf_sust"],
                                "traffic": NCU_DRAM_BYTES_PER_LAUNCH.get((args.workload, n, T)), "kernel": kname,
                                "peak_source": pk["src"] + ", sustained bf16 (kernel runs for >50 ms)",
                                "note": "the binding unit is the MUFU pipe (one tanh per hidden activation), see sfu; HBM traffic is "
                                        "the replay rows only (traffic = dram bytes of one launch, ncu --set full, profiles/)"}
            sm_mhz = clocks.get("sm_mhz") or pk["sm_max"]
            mufu = n * T * (TANH_PER_STEP[(kind, H, S)] - 1 + w["sqrt"] + 6) / (step_ms * 1e-3)
            mufu_peak = 148 * 16 * sm_mhz * 1e6
            line["sfu"] = {"achieved_gops": mufu / 1e9, "peak_gops": mufu_peak / 1e9, "frac": mufu / mufu_peak,
                           "note": "MUFU ops/s (hidden tanh + plant sqrt + Box-Muller) vs 148 SM x 16/clk at the median SM clock "
                                   "under load (tanh.approx microbenchmark on this pool: 16.3 per clk per SM)"}
        if aux is not None:
            line["roofline_step"] = aux
        if not args.no_cpu_baseline and world == 1 and args.workload in ("wt", "ph"):
            line["cpu_baseline"] = cpu_baseline(w, args.cpu_seconds, sd)
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()



def extra_config4(V, world, rank, dist, barrier, pk, steps=5, warmup=2):
    """BASELINE configs[3]: pH ensemble sweep, 2^23 envs in total sharded contiguously over the ranks (strong scaling),
    T = 50, Modular-128, in-kernel auto-reset with ensemble resampling, replay rows written."""
    import torch
    w = dict(WORKLOADS["ph"])
    total = w["envs"]
    n, T, H, S = max(1, total // world), w["T"], w["H"], w["S"]
    K = np.array(w["K"])
    sd = actor_state_dict(H, S)
    actor = V.ActorPack("modular", S, H, 1).update(sd)
    env = V.PHVec(n, dtype=torch.float32, seed=0, env_offset=rank * n)
    env.reset()
    bs = torch.empty((T, n, S), dtype=torch.float32, device="cuda")
    bo = torch.empty((T, n, 4), dtype=torch.float32, device="cuda")
    stats = torch.zeros(8, dtype=torch.float64, device="cuda")

    def step():
        stats.zero_()
        env.rollout(T, -K, actor=actor, auto_reset=True, replay=(bs, bo), stats=stats, gamma=0.99)
        if world > 1:
            dist.all_reduce(stats)

    for _ in range(warmup):
        step()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        step()
    e1.record()
    barrier()
    t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item()) / steps
    env.check_status()
    out = {"metric": METRIC, "value": world * n * T / (ms * 1e-3), "unit": UNIT, "n_gpus": world, "ms_per_step": ms, "steps": steps,
           "scaling": "strong", "workload": w["name"], "envs_total": n * world, "envs_per_gpu": n, "T": T,
           "actor": "ResidualIntegratorModularPPO-" + str(H), "dtype": "x, A, B, table index: f64; rest f32; hidden layers f16 operands",
           "tensor_tflops": world * n * T * FLOPS_PER_STEP[("modular", H, S)] / (ms * 1e-3) / 1e12}
    out["e2e"] = ph_e2e(env, actor, T, K, bs, bo, stats, 3, world, barrier, dist)
    return out


LEARNER_FLOP_PER_ROW = 2 * 3 * (132352 + 133121)   # forward + data gradient + weight gradient of Modular-256 + CriticAdv-256, 2 FLOP per weight


def learner_roofline(buf_len, batch, repeat, update_ms):
    """Tensor-pipe view of the update: algorithmic FLOPs of the minibatch steps (x3 issued: hi/lo terms) over the update time
    (which also holds the value pass, GAE and the index draws) against the sustained bf16 peak of MEASURED_PEAKS.json."""
    pk = peaks()
    steps = int(repeat * buf_len / batch)
    alg = steps * batch * LEARNER_FLOP_PER_ROW / (update_ms * 1e-3) / 1e12
    return {"bound": "tensor", "achieved": alg, "issued": 3 * alg, "peak": pk["tf_sust"], "unit": "TFLOP/s", "frac": alg / pk["tf_sust"],
            "frac_issued": 3 * alg / pk["tf_sust"], "ms_per_minibatch": update_ms / max(steps, 1),
            "note": "algorithmic = 1.59 MFLOP per minibatch row; the step issues three fp16 MMAs per product; see DESIGN.md 4.3"}


def extra_config5(world, rank, dist, barrier, n=1 << 16, batch=1 << 17, repeat=2, iters=2):
    """BASELINE configs[4]: full residual PPO training -- explore (one fused launch into the GPU-resident replay), critic
    values + GAE kernels, repeat * T * n / batch minibatch steps with the gradient all-reduce when world > 1."""
    import torch
    import pime_b200.gym_api as G
    import pime_b200.rl as R
    w = WORKLOADS["train"]
    T, H = w["T"], w["H"]
    env = R.PreprocessEnv(G.make(w["env"], num_envs=n, dtype=torch.float32))
    env.env.vec.env_offset = rank * n
    torch.manual_seed(0)
    torch.backends.cuda.matmul.allow_tf32 = False
    agent = R.AgentResidualIntegratorModularPPO()
    agent.init(H, env.state_dim, env.action_dim, env.n_integrator)
    agent.init_residual({"init_K": env.K.reshape(-1, 1)})
    buf = R.ReplayBuffer(n * T, env.state_dim, 1, True, False, True, num_envs=n)
    t_roll = t_upd = 0.0

    def step():
        nonlocal t_roll, t_upd
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        steps = agent.explore_env(env, buf, n * T, 1.0, 0.99)
        torch.cuda.synchronize()
        t1 = time.perf_counter()
        agent.update_net(buf, steps, batch, repeat)
        torch.cuda.synchronize()
        t_roll += t1 - t0
        t_upd += time.perf_counter() - t1

    step()
    barrier()
    t_roll = t_upd = 0.0
    t0 = time.perf_counter()
    for _ in range(iters):
        step()
    barrier()
    dt = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(dt, op=dist.ReduceOp.MAX)
    return {"metric": "PPO training transitions/sec (explore + update)", "value": world * n * T * iters / float(dt.item()),
            "unit": "env-steps/s", "n_gpus": world, "scaling": "weak", "workload": w["name"], "envs_per_gpu": n, "T": T,
            "actor": "ResidualIntegratorModularPPO-" + str(H), "batch_size": batch, "repeat_times": repeat,
            "minibatches_per_iteration": int(repeat * n * T / batch), "iterations": iters,
            "learner": agent.learner_path, "dtype": "f32-grade learner (fp16 hi + lo operands, three MMAs per product, fp32 accumulation); rollout as the headline",
            "rollout_share": t_roll / max(t_roll + t_upd, 1e-9), "rollout_ms": 1e3 * t_roll / iters, "update_ms": 1e3 * t_upd / iters,
            "learner_roofline": learner_roofline(n * T, batch, repeat, 1e3 * t_upd / iters)}


def aux_step_rooflines(V, pk):
    """Stand-alone gym-API step kernels (state round-trips HBM every call): the HBM-bound rows of SURVEY 8d."""
    import torch
    out = {}
    n = 1 << 25  # 32 Mi envs: 1.2 GB of fp32 state per plant, far larger than L2
    for name in ("wt", "ph"):
        if name == "wt":
            env = V.WaterTankVec(n, dtype=torch.float32, obs_mode="integrator", noise_scale=0.0)
            nbytes = WT_STEP_BYTES_F32
        else:
            env = V.PHVec(n, dtype=torch.float32)
            nbytes = PH_STEP_BYTES_F32
        env.reset()
        act = torch.rand(n, device="cuda") * 2 - 1
        import ctypes as C
        import pime_b200._lib as L
        reward = torch.empty(n, dtype=torch.float32, device="cuda")
        done = torch.empty(n, dtype=torch.uint8, device="cuda")
        st = type(env._st).from_buffer_copy(env._st)
        st.ep_return = None   # the gym-API step of the reference keeps no running return: the 57 / 53 B of SURVEY 8d

        def launch():
            if name == "wt":
                L.check(L.lib().pime_wt_step_f32(C.byref(env.cfg), C.c_int64(n), C.byref(st), L.ptr(act), None, None,
                                                 C.c_uint64(0), C.c_uint64(0), C.c_uint32(0), None, L.ptr(reward), L.ptr(done),
                                                 L.stream_ptr()))
            else:
                L.check(L.lib().pime_ph_step_f32(C.byref(env.cfg), L.ptr(env.table), C.c_int64(n), C.byref(st), L.ptr(act),
                                                 None, L.ptr(reward), L.ptr(done), L.ptr(env.status), L.stream_ptr()))
        for _ in range(3):
            launch()
        torch.cuda.synchronize()
        reps = 10
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            launch()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / reps
        gbs = n * nbytes / (ms * 1e-3) / 1e9
        out[name] = {"bound": "hbm", "achieved": gbs, "peak": pk["hbm"], "unit": "GB/s", "frac": gbs / pk["hbm"],
                     "traffic": NCU_DRAM_BYTES_STEP.get(name),
                     "env_steps_per_s": n / (ms * 1e-3), "bytes_per_env_step": nbytes, "envs": n,
                     "kernel": "wt_step_vec4_kernel (4 envs per thread)" if name == "wt" else "ph_step_kernel<float> (x, A, B, index in fp64)",
                     "peak_source": pk["src"]}
        del env
        torch.cuda.empty_cache()
    return out


def run_train(args):
    """configs[4]: explore (one fused launch) -> update_net (values + GAE kernels; minibatch step: pime_ppo_step up to
    4096 rows, torch autograd above; flat grad all-reduce when distributed) per step; reports transitions/s end to end
    and the rollout share.  Not the bench line.  The reference's own shape (run_watertank_changing.sh: target_step 2000,
    batch 256, repeat 10): --envs 10 --batch-size 256 --repeat-times 10."""
    import torch
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    import pime_b200.gym_api as G
    import pime_b200.rl as R
    w = resolve(args, world)
    n, T, H = w["n"], w["T"], w["H"]
    env = R.PreprocessEnv(G.make(w["env"], num_envs=n, dtype=torch.float32))
    env.env.vec.env_offset = rank * n
    torch.manual_seed(0)
    torch.backends.cuda.matmul.allow_tf32 = bool(args.tf32)
    agent = R.AgentResidualIntegratorModularPPO()
    agent.learning_rate = 3e-4
    agent.init(H, env.state_dim, env.action_dim, env.n_integrator)
    agent.init_residual({"init_K": env.K.reshape(-1, 1)})
    buf = R.ReplayBuffer(n * T, env.state_dim, 1, True, False, True, num_envs=n)
    t_roll = t_upd = 0.0

    def step():
        nonlocal t_roll, t_upd
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        steps = agent.explore_env(env, buf, n * T, 1.0, 0.99)
        torch.cuda.synchronize()
        t1 = time.perf_counter()
        agent.update_net(buf, steps, args.batch_size, args.repeat_times)
        torch.cuda.synchronize()
        t_roll += t1 - t0
        t_upd += time.perf_counter() - t1

    for _ in range(args.warmup):
        step()
    if world > 1:
        dist.barrier()
    t_roll = t_upd = 0.0
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step()
    if world > 1:
        dist.barrier()
    dt = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(dt, op=dist.ReduceOp.MAX)
    if rank == 0:
        print(json.dumps({"metric": "PPO training transitions/sec (explore + update)", "value": world * n * T * args.steps / float(dt.item()),
                          "unit": "env-steps/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                          "config": {"workload": w["name"], "envs_per_gpu": n, "T": T, "actor": w["actor"], "batch_size": args.batch_size,
                                     "repeat_times": args.repeat_times,
                                     "minibatches_per_step": int(args.repeat_times * n * T / args.batch_size),
                                     "learner": "values + GAE: CUDA kernels; minibatch step: " + str(agent.learner_path)},
                          "rollout_share": t_roll / (t_roll + t_upd), "rollout_ms_per_step": 1e3 * t_roll / args.steps,
                          "update_ms_per_step": 1e3 * t_upd / args.steps}), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    args = parse()
    if args.impl == "reference":
        run_reference(args)
    elif args.workload == "train":
        run_train(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
