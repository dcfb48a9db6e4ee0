"""Per-step parity of the fused rollout kernel (rollout_kernel<Plant, KIND, H>, csrc/rollout_impl.cuh + tc_mlp.cuh) at every
compiled (plant, actor kind, H) and at multi-tile geometry, against independent references on every (step, live env) row.

The kernel is one persistent CTA per SM walking tiles of 256 envs as one sequence of network passes; at every tile boundary
the owners store one env, load the next and write its observation for the next pass.  The env counts are chosen against
that geometry (P = SM count of the device, read from torch like the launcher reads it):

  1            one live row, 255 dead ones shadowing it
  129          group 0 full, a single live row in group 1
  256 P + 1    CTA 0 gets a second tile holding one live env: uneven tile counts across CTAs
  3 * 256 P - 77   every CTA walks three tiles, the last one ragged

Small n run T >= max_step + 20 steps from a random initial t, so in-kernel resets land on different steps in different
envs; large n run a few steps, and T = 1 / T = 2 make every pass a tile boundary.  Each case asserts, on every row:

  1. routing, BITWISE: with deterministic=True (a_raw == a_avg) the recorded a_avg equals ActorPack.forward() of the recorded
     observation bit for bit.  Both kernels run the same tc::Engine, write_obs and read_out, and a tcgen05.mma output row
     does not depend on which lane / tile / pass it came from, so any row, group, tile or pass mix-up or stale operand shows;
  2. accuracy against a float64 torch forward (net64): per row 4e-3 + 1e-2 |want|, plus per-configuration RMS and
     |mean error| bounds (BOUNDS below, measured values beside them);
  3. stochastic runs (in-kernel Philox, auto-reset, two launches so that tick0 != 0): a_raw == forward(obs) + eps a_std within
     2 fp32 ulp, and eps equal to an fp64 Box-Muller of the oracle's Philox words within 1e-4 on >= 4096 (env, step) pairs
     that include the first and last rows of every tile of CTA 0;
  4. plant and bookkeeping from an open-loop replay of the recorded env_action through the oracle plant (fp64 plant:
     observations bit-identical, resets included; float plant: per-step bounds of test_gpu_01 / test_gpu_03 from the
     recorded float state), env_action == tanhf(a) + obs32 . priorK, reward / mask columns, final t / episode / ep_return,
     and the statistics block;
  5. dead tail rows write nothing (state arrays and replay rows padded with a sentinel, ld = n + pad);
  6. fidelity mode (rollout_fp32_kernel) bitwise against actor_forward_fp32_kernel and within 2e-5 of net64.

The replay helpers are pinned by test_replay_helpers_match_oracle_rollouts, which needs no GPU; every other test here is
marked gpu one by one for that reason (a module-level pytestmark would skip it too).
"""
import ctypes as C
import types

import numpy as np
import pytest
import torch

gpu = pytest.mark.gpu

HS = (32, 64, 128, 256)
WT_MAX, PH_MAX = 200, 50
K_WT = np.array([0.0, -0.4, 0.4, 0.0])     # priorK = -K of the reference scripts (obs . priorK = 0.4 (r - h2))
K_PH = np.array([0.02, -0.02, -0.035])
ATOL, RTOL = 4e-3, 1e-2                    # stated per-row bound of the throughput mode (test_gpu_02)

# (plant, observation, actor kind, H, num_stack, plant flavour)
CONFIGS = ([("wt", "integrator", "modular", H, 0, "f32") for H in HS]
           + [("wt", "integrator", "plain", H, 0, "f32") for H in HS]
           + [("wt", "goal", "plain", H, 0, "f32") for H in (64, 256)]
           + [("wt", "stacking", "plain", 256, k, "f32") for k in (1, 4, 10)]
           + [("ph", "integrator", "modular", H, 0, "f32") for H in HS]
           + [("wt", "stacking", "plain", H, 4, "f32") for H in (32, 64, 128)]
           + [("ph", "none", "plain", H, 0, "f32") for H in HS]
           + [("wt", "integrator", "modular", 256, 0, "f64"), ("ph", "integrator", "modular", 128, 0, "f64"),
              ("wt", "stacking", "plain", 256, 10, "f64")])
N_LABELS = ("1", "129", "tile+1", "3tiles-77")
SHORT = [(("wt", "integrator", "modular", H, 0, "f32"), T) for H in (32, 256) for T in (1, 2)]
BENCH = [(("wt", "integrator", "modular", 256, 0, "f32"), 1 << 20),    # headline Modular-256
         (("ph", "integrator", "modular", 128, 0, "f32"), 1 << 23),    # pH Modular-128
         (("wt", "stacking", "plain", 256, 10, "f32"), 1 << 19)]       # wts10: Stacking-10, plain-256, S = 30

# Bounds on (a_avg - net64) per configuration: (RMS, |mean|).  Set from one B200 run (NVIDIA B200, 1000 W power limit) at
# 1.5x the largest value measured over the configuration's cases; the comment gives the measured max |error|, RMS and
# |mean|.  The RMS bound holds for every case; the |mean| bound for the cases with >= 1e5 rows (the multi-tile, short-T and
# bench-geometry ones) -- at n = 1 and 129 the rows are one or a few correlated trajectories and their mean is no sharper
# than their RMS.  A bias error of +0.05 on one hidden unit moves the output by 3e-4 ... 1e-2.
MEAN_ROWS = 100_000
BOUNDS = {  # tag: (rms, |mean|),                 measured: max      rms      |mean|
    "wt-integrator-modular32-f32": (8.8e-05, 3.4e-05),  # 2.2e-04  5.8e-05  2.3e-05
    "wt-integrator-modular64-f32": (8.3e-05, 1.9e-05),  # 2.6e-04  5.5e-05  1.2e-05
    "wt-integrator-modular128-f32": (1.6e-04, 1.3e-04),  # 4.0e-04  1.0e-04  8.5e-05
    "wt-integrator-modular256-f32": (2.1e-04, 4.5e-05),  # 6.2e-04  1.4e-04  3.0e-05
    "wt-integrator-plain32-f32": (9.5e-05, 6.1e-05),  # 2.0e-04  6.3e-05  4.1e-05
    "wt-integrator-plain64-f32": (1.8e-04, 2.1e-05),  # 2.4e-04  1.2e-04  1.4e-05
    "wt-integrator-plain128-f32": (1.9e-04, 1.6e-04),  # 4.3e-04  1.2e-04  1.0e-04
    "wt-integrator-plain256-f32": (2.4e-04, 1.2e-04),  # 5.2e-04  1.5e-04  7.9e-05
    "wt-goal-plain64-f32": (1.4e-04, 4.9e-05),    # 2.6e-04  8.9e-05  3.2e-05
    "wt-goal-plain256-f32": (3.2e-04, 2.1e-04),   # 6.2e-04  2.1e-04  1.3e-04
    "wt-stacking1-plain256-f32": (1.7e-04, 6.7e-05),  # 5.3e-04  1.1e-04  4.5e-05
    "wt-stacking4-plain256-f32": (3.6e-04, 3.0e-04),  # 9.4e-04  2.4e-04  2.0e-04
    "wt-stacking10-plain256-f32": (4.0e-04, 3.2e-04),  # 1.2e-03  2.6e-04  2.1e-04
    "ph-integrator-modular32-f32": (1.6e-04, 5.7e-05),  # 2.0e-04  1.0e-04  3.7e-05
    "ph-integrator-modular64-f32": (1.7e-04, 1.5e-04),  # 3.2e-04  1.1e-04  9.8e-05
    "ph-integrator-modular128-f32": (1.8e-04, 1.4e-04),  # 4.1e-04  1.2e-04  9.1e-05
    "ph-integrator-modular256-f32": (3.7e-04, 3.1e-04),  # 7.3e-04  2.4e-04  2.0e-04
    "wt-stacking4-plain32-f32": (1.5e-04, 1.1e-04),  # 3.3e-04  9.5e-05  6.8e-05
    "wt-stacking4-plain64-f32": (1.5e-04, 1.2e-04),  # 3.1e-04  9.6e-05  7.8e-05
    "wt-stacking4-plain128-f32": (1.6e-04, 4.6e-06),  # 3.9e-04  1.1e-04  3.1e-06
    "ph-none-plain32-f32": (8.6e-05, 7.1e-05),    # 1.8e-04  5.7e-05  4.7e-05
    "ph-none-plain64-f32": (1.9e-04, 1.7e-04),    # 3.2e-04  1.2e-04  1.1e-04
    "ph-none-plain128-f32": (2.5e-04, 2.3e-04),   # 4.5e-04  1.7e-04  1.5e-04
    "ph-none-plain256-f32": (1.8e-04, 8.2e-05),   # 5.4e-04  1.2e-04  5.4e-05
    "wt-integrator-modular256-f64": (2.3e-04, 1.6e-04),  # 5.4e-04  1.5e-04  1.1e-04
    "ph-integrator-modular128-f64": (2.4e-04, 2.0e-04),  # 3.7e-04  1.6e-04  1.3e-04
    "wt-stacking10-plain256-f64": (3.0e-04, 2.0e-04),  # 1.3e-03  2.0e-04  1.3e-04
}


def tag(cfg):
    plant, obs, kind, H, k, dt = cfg
    return f"{plant}-{obs}{k or ''}-{kind}{H}-{dt}"


def state_dim(cfg):
    plant, obs, kind, H, k, dt = cfg
    if plant == "wt":
        return {"goal": 3, "integrator": 4}.get(obs, 3 * k)
    return 2 if obs == "none" else 3


def prior_k(cfg):
    plant, obs = cfg[:2]
    S = state_dim(cfg)
    if plant == "ph":
        return K_PH[:S].copy()
    if obs == "stacking":
        K = np.zeros(S)
        K[-3:] = K_WT[:3]   # the prior acts on the newest frame
        return K
    return K_WT[:S].copy()


def sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def n_of(label):
    P = sms()
    return {"1": 1, "129": 129, "tile+1": 256 * P + 1, "3tiles-77": 3 * 256 * P - 77}[label]


def f32(v):
    return np.asarray(v, np.float64).astype(np.float32).astype(np.float64)


# ------------------------------------------------------------------------------------------------ reference network
def actor_params(kind, H, S, seed, scale_last=0.1):
    """Random parameters at torch.nn.Linear's default scale in state_dict form; a non-trivial last layer."""
    rng = np.random.default_rng(seed)
    if kind == "modular":
        shapes = [("other_net.0", H, S - 1), ("other_net.2", H // 2, H), ("integrator_net.0", H, 1),
                  ("integrator_net.2", H // 2, H), ("net.0", H, H), ("net.2", 1, H)]
    else:
        shapes = [("net.0", H, S), ("net.2", H, H), ("net.4", H, H), ("net.6", 1, H)]
    sd = {}
    for name, o, i in shapes:
        b = 1.0 / np.sqrt(i)
        sd[name + ".weight"] = rng.uniform(-b, b, (o, i)).astype(np.float32)
        sd[name + ".bias"] = rng.uniform(-b, b, o).astype(np.float32)
    sd[shapes[-1][0] + ".weight"] = rng.normal(0, scale_last, (1, H)).astype(np.float32)
    return sd


def net64(kind, sd, obs):
    """a_avg = net(obs) in float64 on the GPU (torch), in chunks of at most 2^20 rows."""
    t = {k: torch.as_tensor(np.asarray(v), dtype=torch.float64, device=obs.device) for k, v in sd.items()}

    def lin(x, name):
        return x @ t[name + ".weight"].T + t[name + ".bias"]
    out = torch.empty(obs.shape[0], dtype=torch.float64, device=obs.device)
    for a in range(0, obs.shape[0], 1 << 20):
        x = obs[a:a + (1 << 20)].double()
        if kind == "modular":
            So = t["other_net.0.weight"].shape[1]
            u = torch.tanh(lin(torch.tanh(lin(x[:, :So], "other_net.0")), "other_net.2"))
            v = torch.tanh(lin(torch.tanh(lin(x[:, So:], "integrator_net.0")), "integrator_net.2"))
            y = lin(torch.tanh(lin(torch.cat([u, v], 1), "net.0")), "net.2")
        else:
            h = torch.tanh(lin(x, "net.0"))
            h = torch.tanh(lin(h, "net.2"))
            y = lin(torch.tanh(lin(h, "net.4")), "net.6")
        out[a:a + x.shape[0]] = y[:, 0]
    return out


def bitwise_equal(a, b):
    return a.contiguous().view(torch.int32) == b.contiguous().view(torch.int32)


# ------------------------------------------------------------------------------------------------ open-loop plant replay
def _lohi(lo, hi, u, flavour):
    """wt_reset's low + (high - low) u with the constants as the kernel folds them (WtConst<T>)."""
    if flavour == "f32":
        return float(np.float32(float(np.float32(lo)) + float(np.float32(hi - lo)) * u))
    return lo + (hi - lo) * u


def wt_replay(oracle, obs_mode, k, flavour, st0, act, seed, env_offset, pn=None, obs_rec=None, auto_reset=True):
    """Feed the recorded env_action [T, n] through oracle.wt_step from the initial state st0 (float64 arrays h1 h2 r I a1 a2
    Kp, int t, episode, frames [n, 3k]), one step at a time.  After a `done` (auto_reset) the env is reset from the Philox
    uniforms oracle.reset_uniforms(seed, env_offset + i, episode).  obs_rec (float flavour): the state at every step is
    re-read from the recorded float observation, which holds it exactly -- a local per-step check the loop cannot amplify.
    Returns obs [T, n, S] (float32, what the network saw), nxt [T, n, S] (float64, the observation after the step and any
    reset), rew, done [T, n] and the final state."""
    integ, stack = obs_mode == "integrator", obs_mode == "stacking"
    cfg = oracle.wt_cfg(reward_type="square_distance", has_integrator=integ)
    cast = f32 if flavour == "f32" else (lambda v: np.asarray(v, np.float64))
    T, n = act.shape
    s = {key: np.array(cast(st0[key]), np.float64) for key in ("h1", "h2", "r", "I", "a1", "a2", "Kp")}
    h1, h2, r, I, a1, a2, Kp = (s[key] for key in ("h1", "h2", "r", "I", "a1", "a2", "Kp"))
    t = np.array(st0["t"], np.int32)
    ep = np.array(st0["episode"], np.int64)
    fr = np.array(cast(st0["frames"]), np.float64) if stack else None
    S = 3 * k if stack else (4 if integ else 3)
    obs = np.empty((T, n, S), np.float32)
    nxt = np.empty((T, n, S), np.float64)
    rew = np.empty((T, n))
    done = np.empty((T, n), bool)

    def observe():
        return fr.copy() if stack else np.stack([h1, h2, r] + ([I] if integ else []), 1)
    for q in range(T):
        if obs_rec is not None:
            o = obs_rec[q].astype(np.float64)
            if stack:
                fr[:] = o
                h1[:], h2[:], r[:] = o[:, -3], o[:, -2], o[:, -1]
            else:
                h1[:], h2[:], r[:] = o[:, 0], o[:, 1], o[:, 2]
                if integ:
                    I[:] = o[:, 3]
        obs[q] = observe()
        p1 = None if pn is None else np.ascontiguousarray(pn[0][q], np.float64)
        p2 = None if pn is None else np.ascontiguousarray(pn[1][q], np.float64)
        rw, dn = oracle.wt_step(cfg, h1, h2, r, I if integ else None, t, a1, a2, Kp, np.ascontiguousarray(act[q], np.float64), p1, p2)
        if stack:   # frames.append(state)
            fr[:, :-3] = fr[:, 3:]
            fr[:, -3], fr[:, -2], fr[:, -1] = h1, h2, r
        for i in (np.flatnonzero(dn) if auto_reset else ()):
            u = oracle.reset_uniforms(seed, env_offset + int(i), int(ep[i]))
            a1[i], a2[i] = _lohi(0.0015, 0.0024, u[0], flavour), _lohi(0.0015, 0.0024, u[1], flavour)
            Kp[i] = _lohi(0.07, 0.17, u[2], flavour)
            h1[i], h2[i], r[i] = (_lohi(0.0, 10.0, u[j], flavour) for j in (3, 4, 5))
            I[i], t[i] = 0.0, 0
            ep[i] += 1
            if stack:
                fr[i] = np.tile([h1[i], h2[i], r[i]], k)
        nxt[q] = observe()
        rew[q], done[q] = rw, dn.astype(bool)
    return dict(obs=obs, nxt=nxt, rew=rew, done=done, t=t, episode=ep, **s, frames=fr)


def ph_replay(oracle, mode, flavour, st0, act, seed, env_offset, table, obs_rec=None, auto_reset=True):
    """The pH counterpart of wt_replay: oracle.ph_step on the device's own fp64 titration table, resets through
    oracle.reset_uniforms + oracle.ph_update_system + the table lookup.  x, A, B are fp64 in both flavours.  Also returns
    idx [T, n], the table entry read after each step (and reset)."""
    integ = mode != "none"
    cfg = oracle.ph_cfg(integrator_mode=1 if integ else 0)
    cast = f32 if flavour == "f32" else (lambda v: np.asarray(v, np.float64))
    T, n = act.shape
    s = {key: np.array(st0[key], np.float64) for key in ("x", "A", "B")}
    s.update({key: np.array(cast(st0[key]), np.float64) for key in ("y", "r", "I", "C", "qww_V", "qc_V")})
    x, y, r, I, A, B, Cc, qww, qc = (s[key] for key in ("x", "y", "r", "I", "A", "B", "C", "qww_V", "qc_V"))
    t = np.array(st0["t"], np.int32)
    ep = np.array(st0["episode"], np.int64)
    S = 3 if integ else 2
    obs = np.empty((T, n, S), np.float32)
    nxt = np.empty((T, n, S), np.float64)
    idx = np.empty((T, n), np.int64)
    rew = np.empty((T, n))
    done = np.empty((T, n), bool)

    def observe():
        return np.stack([y, r] + ([I] if integ else []), 1)
    for q in range(T):
        if obs_rec is not None:
            o = obs_rec[q].astype(np.float64)
            y[:], r[:] = o[:, 0], o[:, 1]
            if integ:
                I[:] = o[:, 2]
        obs[q] = observe()
        rw, dn = oracle.ph_step(cfg, table, x, y, r, I, t, A, B, Cc, np.ascontiguousarray(act[q], np.float64))
        for i in (np.flatnonzero(dn) if auto_reset else ()):
            u = oracle.reset_uniforms(seed, env_offset + int(i), int(ep[i]))
            qww[i], qc[i] = cast(0.005 + (0.015 - 0.005) * u[0]), cast(0.0015 + (0.0025 - 0.0015) * u[1])
            a_, b_, c_ = oracle.ph_update_system(qww[i:i + 1], qc[i:i + 1])
            A[i], B[i], Cc[i] = a_[0], b_[0], c_[0]
            x[i] = 0.0 + 50.0 * u[2]
            y[i] = table[int(np.rint(Cc[i] * x[i] * 1e5))]
            r[i] = cast(3.0 + (11.0 - 3.0) * u[3])
            I[i], t[i] = 0.0, 0
            ep[i] += 1
        idx[q] = np.rint(Cc * x * 1e5).astype(np.int64)
        nxt[q] = observe()
        rew[q], done[q] = rw, dn.astype(bool)
    return dict(obs=obs, nxt=nxt, idx=idx, rew=rew, done=done, t=t, episode=ep, **s)


def episode_returns(rew, done, ret0, flavour):
    """env.ret += rew every step, handed to the statistics and zeroed at a `done`, in the plant's arithmetic.
    Returns (final ep_return, the finished returns)."""
    dt = np.float32 if flavour == "f32" else np.float64
    ret = np.array(ret0, dt)
    fin = []
    for q in range(rew.shape[0]):
        ret = (ret + rew[q].astype(dt)).astype(dt)
        fin.append(ret[done[q]].astype(np.float64))
        ret[done[q]] = 0
    return ret, np.concatenate(fin) if fin else np.zeros(0)


def bm_ref(oracle, seed, index, tick):
    """fp64 Box-Muller of the per-step Philox block (stream 3): words 2,3 -> eps, words 0,1 -> process-noise pair."""
    w = oracle.philox4x32(seed, index, tick, 3)

    def pair(a, b):   # the uniforms as the kernel forms them, float((a >> 8) + 0.5) / 2^24; the rest in fp64
        u1 = float(np.float32(a >> 8) + np.float32(0.5)) / 16777216.0
        u2 = float(np.float32(b >> 8) + np.float32(0.5)) / 16777216.0
        rad = np.sqrt(-2.0 * np.log(u1))
        return rad * np.cos(2 * np.pi * u2), rad * np.sin(2 * np.pi * u2)
    return pair(w[2], w[3])[0], pair(w[0], w[1])


# ------------------------------------------------------------------------------------------------ CPU-only pin of the replay
def test_replay_helpers_match_oracle_rollouts(oracle, oracle_table):
    """Prior-only policies across an episode boundary: the replay helpers reproduce oracle.wt_rollout / oracle.ph_rollout
    bit for bit -- up to the `done`, and after it from the reset state drawn from the oracle's Philox uniforms."""
    rng = np.random.default_rng(3)
    n, seed, off = 5, 17, 1000
    for obs_mode, k in (("integrator", 0), ("stacking", 4), ("goal", 0)):
        S = 3 * k if k else (4 if obs_mode == "integrator" else 3)
        d = dict(h1=rng.uniform(0, 10, n), h2=rng.uniform(0, 10, n), r=rng.uniform(0, 10, n), I=rng.uniform(-5, 5, n),
                 a1=rng.uniform(0.0015, 0.0024, n), a2=rng.uniform(0.0015, 0.0024, n), Kp=rng.uniform(0.07, 0.17, n),
                 t=np.full(n, WT_MAX - 3, np.int32), episode=np.arange(1, n + 1), ep_return=np.zeros(n))
        if obs_mode != "integrator":
            d["I"] = np.zeros(n)
        d["frames"] = np.tile(np.stack([d["h1"], d["h2"], d["r"]], 1), (1, max(k, 1)))[:, :S]
        K = prior_k(("wt", obs_mode, "plain", 32, k, "f64"))
        pn = (rng.normal(0, 0.01, (8, n)), rng.normal(0, 0.01, (8, n)))
        mode = {"goal": 0, "integrator": 1, "stacking": 2}[obs_mode]
        cfg = oracle.wt_cfg(reward_type="square_distance", has_integrator=obs_mode == "integrator")

        def run(st, T, pn_):
            st = {key: np.array(v, np.float64) if key != "t" else np.array(v, np.int32) for key, v in st.items()}
            fr = np.ascontiguousarray(st["frames"]) if k else None
            o = oracle.wt_rollout(cfg, None, None, -0.5, K, mode, k, False, T, st["h1"], st["h2"], st["r"], st["I"], st["t"],
                                  st["a1"], st["a2"], st["Kp"], frames=fr, pn1=np.ascontiguousarray(pn_[0]),
                                  pn2=np.ascontiguousarray(pn_[1]), want_actions=True)
            return o
        oa = run(d, 3, (pn[0][:3], pn[1][:3]))
        d2 = dict(t=np.zeros(n, np.int32), I=np.zeros(n))
        cols = {key: np.empty(n) for key in ("a1", "a2", "Kp", "h1", "h2", "r")}
        for i in range(n):
            u = oracle.reset_uniforms(seed, off + i, int(d["episode"][i]))
            for j, key in enumerate(("a1", "a2", "Kp", "h1", "h2", "r")):
                lo, hi = {"a1": (0.0015, 0.0024), "a2": (0.0015, 0.0024), "Kp": (0.07, 0.17)}.get(key, (0.0, 10.0))
                cols[key][i] = lo + (hi - lo) * u[j]
        d2.update(cols)
        d2["frames"] = np.tile(np.stack([d2["h1"], d2["h2"], d2["r"]], 1), (1, max(k, 1)))[:, :S]
        ob = run(d2, 5, (pn[0][3:], pn[1][3:]))
        act = np.concatenate([oa["env_action"], ob["env_action"]])
        rp = wt_replay(oracle, obs_mode, k, "f64", d, act, seed, off, pn=pn)
        assert np.array_equal(rp["obs"], np.concatenate([oa["buf_state"], ob["buf_state"]])), obs_mode
        assert np.array_equal(rp["rew"].astype(np.float32), np.concatenate([oa["buf_other"], ob["buf_other"]])[..., 0])
        assert rp["done"][2].all() and not rp["done"][:2].any() and not rp["done"][3:].any()
        ret, fin = episode_returns(rp["rew"], rp["done"], d["ep_return"], "f64")
        assert np.array_equal(fin, oa["ep_return"]) and np.array_equal(ret, ob["ep_return"])
        assert np.array_equal(rp["episode"], d["episode"] + 1) and np.array_equal(rp["t"], np.full(n, 5))

    # pH: same construction through oracle.ph_rollout
    qww, qc = rng.uniform(0.005, 0.015, n), rng.uniform(0.0015, 0.0025, n)
    A, B, Cc = oracle.ph_update_system(qww, qc)
    x, r = rng.uniform(0, 50, n), rng.uniform(3, 11, n)
    y = oracle_table[np.rint(Cc * x * 1e5).astype(np.int64)]
    for integ in (1, 0):
        S = 3 if integ else 2
        d = dict(x=x, y=y, r=r, I=np.zeros(n), A=A, B=B, C=Cc, qww_V=qww, qc_V=qc, t=np.full(n, PH_MAX - 2, np.int32),
                 episode=np.ones(n, np.int64), ep_return=np.zeros(n))
        cfg = oracle.ph_cfg(integrator_mode=integ)

        def run(st, T):
            st = {key: np.array(v, np.float64) if key != "t" else np.array(v, np.int32) for key, v in st.items()}
            return oracle.ph_rollout(cfg, oracle_table, None, None, -0.5, -K_PH[:S], False, T, st["x"], st["y"], st["r"],
                                     st["I"], st["t"], st["A"], st["B"], st["C"], want_actions=True)
        oa = run(d, 2)
        d2 = dict(I=np.zeros(n), t=np.zeros(n, np.int32))
        us = [oracle.reset_uniforms(seed, off + i, 1) for i in range(n)]
        d2["qww_V"] = np.array([0.005 + (0.015 - 0.005) * u[0] for u in us])
        d2["qc_V"] = np.array([0.0015 + (0.0025 - 0.0015) * u[1] for u in us])
        d2["A"], d2["B"], d2["C"] = oracle.ph_update_system(d2["qww_V"], d2["qc_V"])
        d2["x"] = np.array([50.0 * u[2] for u in us])
        d2["r"] = np.array([3.0 + 8.0 * u[3] for u in us])
        d2["y"] = oracle_table[np.rint(d2["C"] * d2["x"] * 1e5).astype(np.int64)]
        ob = run(d2, 4)
        act = np.concatenate([oa["env_action"], ob["env_action"]])
        rp = ph_replay(oracle, "integrator" if integ else "none", "f64", d, act, seed, off, oracle_table)
        assert np.array_equal(rp["obs"], np.concatenate([oa["buf_state"], ob["buf_state"]])), integ
        assert np.array_equal(rp["rew"].astype(np.float32), np.concatenate([oa["buf_other"], ob["buf_other"]])[..., 0])
        assert rp["done"][1].all() and rp["done"].sum() == n
        ret, fin = episode_returns(rp["rew"], rp["done"], d["ep_return"], "f64")
        assert np.array_equal(fin, oa["ep_return"]) and np.array_equal(ret, ob["ep_return"])


def test_case_matrix_covers_every_compiled_shape():
    """The launcher compiles the plain and the modular actor at H = 32/64/128/256 for the water tank and the pH plant, and
    the plain one for the stacking water tank (rollout_wt.cuh / rollout_ph.cuh): each is in the matrix, both plant
    flavours are, and so are the three stacking depths (the three replay-row store branches of Stepper::finish)."""
    compiled = ({(p, kind, H) for p in ("wt", "ph") for kind in ("plain", "modular") for H in HS}
                | {("wt-stacking", "plain", H) for H in HS})
    covered = {(c[0] + ("-stacking" if c[1] == "stacking" else ""), c[2], c[3]) for c in CONFIGS}
    assert compiled <= covered, compiled - covered
    assert {c[5] for c in CONFIGS} == {"f32", "f64"}
    assert {state_dim(c) for c in CONFIGS} >= {2, 3, 4, 12, 30}
    print("\nrollout parity cases:")
    for c in CONFIGS:
        print(f"  {tag(c)}  x  n in {N_LABELS}")
    for c, T in SHORT:
        print(f"  {tag(c)}  x  n = 3 * 256 P - 77, T = {T}")
    for c, n in BENCH:
        print(f"  {tag(c)}  x  n = {n} (bench geometry), T = 4")


# ------------------------------------------------------------------------------------------------ GPU cases
@pytest.fixture(scope="module")
def V():
    import pime_b200.vec as vec
    return vec


def make_env(V, cfg, n, seed, env_offset=0):
    plant, obs, kind, H, k, dt = cfg
    dtype = torch.float32 if dt == "f32" else torch.float64
    if plant == "wt":
        env = V.WaterTankVec(n, dtype=dtype, obs_mode=obs, num_stack=k, seed=seed, env_offset=env_offset)
    else:
        env = V.PHVec(n, dtype=dtype, integrator=obs, seed=seed, env_offset=env_offset)
    env.reset()
    return env


def state_fields(cfg):
    if cfg[0] == "wt":
        return ("h1", "h2", "r", "I", "a1", "a2", "Kp", "t", "episode", "ep_return") + (("frames",) if cfg[1] == "stacking" else ())
    return ("x", "y", "r", "I", "A", "B", "C", "qww_V", "qc_V", "t", "episode", "ep_return")


def snapshot(env, cfg):
    st = {}
    for key in state_fields(cfg):
        v = getattr(env, key).detach().cpu().numpy()
        st[key] = v.T.copy() if key == "frames" else v.astype(np.int64) if key in ("t", "episode") else v.astype(np.float64)
    return st


def rollout(env, cfg, T, pack, deterministic, pn=None):
    kw = dict(actor=pack, deterministic=deterministic, auto_reset=True, replay=True, want_actions=True)
    if pn is not None:
        kw["pnoise"] = pn
    out = env.rollout(T, prior_k(cfg), **kw)
    env.check_status()
    return out


def check_network(cfg, kind, sd, pack, out, S, errs):
    """Items 1 and 2: bitwise routing, accuracy against net64 (errors collected in errs for the RMS / mean bounds)."""
    bs, bo = out["buf_state"].reshape(-1, S), out["buf_other"].reshape(-1, 4)
    a = bo[:, 2].contiguous()
    fwd = pack.forward(bs)
    bad = ~bitwise_equal(a, fwd)
    if bool(bad.any()):
        first = int(torch.nonzero(bad)[0])
        n = out["buf_state"].shape[1]
        raise AssertionError(f"{tag(cfg)}: {int(bad.sum())} rows of a_avg differ from ActorPack.forward(obs) in their bits; "
                             f"first at (step, env) = {divmod(first, n)}: {float(a[first])!r} vs {float(fwd[first])!r}")
    want = net64(kind, sd, bs)
    err = a.double() - want
    over = err.abs() > ATOL + RTOL * want.abs()
    assert not bool(over.any()), f"{tag(cfg)}: {int(over.sum())} rows beyond 4e-3 + 1e-2 |want|, max {float(err.abs().max()):.3e}"
    errs.append(err)


def check_stochastic(oracle, cfg, pack, out, S, seed, env_offset, tick0, a_std, dtype, rng, st0=None):
    """Item 3 on one stochastic launch, plus the action arithmetic of item 4."""
    T, n = out["buf_state"].shape[:2]
    bs, bo = out["buf_state"].reshape(-1, S), out["buf_other"].reshape(-1, 4)
    a_raw, eps = bo[:, 2], bo[:, 3]
    fwd = pack.forward(bs)
    ref = fwd.double() + eps.double() * a_std
    m = torch.maximum(torch.maximum(a_raw.abs(), fwd.abs()), (eps * a_std).abs())
    ulp = (torch.nextafter(m, torch.full_like(m, float("inf"))) - m).double()
    off = (a_raw.double() - ref).abs() > 2 * ulp
    assert not bool(off.any()), f"{tag(cfg)}: a_raw != forward(obs) + eps a_std within 2 ulp on {int(off.sum())} rows"
    # env_action = tanhf(a_raw) + obs32 . priorK, in the flavour's arithmetic (up to tanhf / summation rounding)
    K = torch.as_tensor(prior_k(cfg).astype(np.float32).astype(np.float64) if dtype == torch.float32 else prior_k(cfg),
                        device=bs.device)
    terms = bs.double() * K
    want = torch.tanh(a_raw.double()) + terms.sum(1)
    tol = 1e-6 * (1.0 + terms.abs().sum(1))
    act = out["env_action"].reshape(-1).double()
    assert bool(((act - want).abs() <= tol).all()), f"{tag(cfg)}: env_action off by {float((act - want).abs().max()):.3e}"
    # eps vs the fp64 Box-Muller reference on >= 4096 (env, step) pairs incl. the first / last rows of CTA 0's tiles
    tiles = (n + 255) // 256
    G = min(tiles, sms())
    rows = set()
    for tl in range(0, tiles, G):
        lo = tl * 256
        rows.update(i for i in (lo, lo + 127, lo + 128, min(lo + 255, n - 1)) if i < n)
    pairs = {(q, i) for i in rows for q in range(T)}
    if n * T <= 4096:
        pairs = {(q, i) for i in range(n) for q in range(T)}
    while len(pairs) < min(4096, n * T):
        pairs.add((int(rng.integers(T)), int(rng.integers(n))))
    pairs = sorted(pairs)
    qi = torch.as_tensor([p[0] for p in pairs], device=bs.device)
    ii = torch.as_tensor([p[1] for p in pairs], device=bs.device)
    got = out["buf_other"][..., 3][qi, ii].cpu().numpy()
    ref = np.array([bm_ref(oracle, seed, env_offset + i, tick0 + q)[0] for q, i in pairs])
    err = np.abs(got.astype(np.float64) - ref)
    assert err.max() <= 1e-4, f"{tag(cfg)}: eps differs from Box-Muller(Philox) by {err.max():.2e} at {pairs[int(err.argmax())]}"
    if cfg[0] == "wt" and dtype == torch.float32 and st0 is not None:
        check_process_noise(oracle, cfg, out, st0, pairs, seed, env_offset, tick0)


def check_process_noise(oracle, cfg, out, st0, pairs, seed, env_offset, tick0, sigma=0.01):
    """In-kernel process noise of the float water tank (noise_scale = sigma, nothing injected).  The float state is
    observed exactly, so one oracle step from the recorded observation of step q, with the recorded action and sigma times
    the fp64 Box-Muller pair of Philox words 0 and 1, must give the observation of step q + 1 within the per-step plant
    bound.  (env, step) pairs whose env finished an episode by step q are left out: their parameters were re-drawn."""
    obs_mode, k = cfg[1], cfg[4]
    integ, stack = obs_mode == "integrator", obs_mode == "stacking"
    bs = out["buf_state"].cpu().numpy()
    mask = out["buf_other"][..., 1].cpu().numpy()
    act = out["env_action"].cpu().numpy().astype(np.float64)
    T = bs.shape[0]
    alive = np.cumsum(mask == 0, axis=0) == 0
    sel = [(q, i) for q, i in pairs if q + 1 < T and alive[q, i]]
    if not sel:
        return
    q, i = np.array([p[0] for p in sel]), np.array([p[1] for p in sel])
    o = bs[q, i].astype(np.float64)
    c = (o.shape[1] - 3, o.shape[1] - 2, o.shape[1] - 1) if stack else (0, 1, 2)
    h1, h2, r = (np.ascontiguousarray(o[:, j]) for j in c)
    I = np.ascontiguousarray(o[:, 3]) if integ else None
    z = np.array([bm_ref(oracle, seed, env_offset + int(ii), tick0 + int(qq))[1] for qq, ii in sel])
    ocfg = oracle.wt_cfg(reward_type="square_distance", has_integrator=integ)
    oracle.wt_step(ocfg, h1, h2, r, I, np.zeros(len(sel), np.int32), *(np.ascontiguousarray(st0[key][i]) for key in ("a1", "a2", "Kp")),
                   np.ascontiguousarray(act[q, i]), np.ascontiguousarray(sigma * z[:, 0]), np.ascontiguousarray(sigma * z[:, 1]))
    nxt = bs[q + 1, i].astype(np.float64)
    for j, want in zip(c[:2], (h1, h2)):
        err = np.abs(nxt[:, j] - want)
        assert (err <= 2e-5 * np.maximum(np.abs(want), 0.1)).all(), \
            f"{tag(cfg)}: process noise: level {j} off by {err.max():.2e} at (step, env) {sel[int(err.argmax())]}"


def check_plant(oracle, V, cfg, env, st0, out, pn, seed, env_offset, S):
    """Item 4 from the replay: observations, reward / mask columns, final state, statistics."""
    plant, obs_mode, kind, H, k, flav = cfg
    bs, bo = out["buf_state"].cpu().numpy(), out["buf_other"].cpu().numpy()
    act = out["env_action"].cpu().numpy().astype(np.float64)
    T, n = act.shape
    rec = bs if flav == "f32" else None
    if plant == "wt":
        pnh = None if pn is None else (pn[0].cpu().numpy(), pn[1].cpu().numpy())
        rp = wt_replay(oracle, obs_mode, k, flav, st0, act, seed, env_offset, pn=pnh, obs_rec=rec)
    else:
        t64, t32 = (x.cpu().numpy() for x in V.ph_table(env.cfg, env.device))
        rp = ph_replay(oracle, obs_mode, flav, st0, act, seed, env_offset, t64, obs_rec=rec)
    done = rp["done"]
    # env_action = tanhf(a_avg) + obs32 . float(priorK), added in fp32 (Stepper::prepare), up to tanhf / summation rounding
    terms = bs.astype(np.float64) * prior_k(cfg).astype(np.float32).astype(np.float64)
    want_a = np.tanh(bo[..., 2].astype(np.float64)) + terms.sum(-1)
    assert (np.abs(act - want_a) <= 1e-6 * (1.0 + np.abs(terms).sum(-1))).all(), f"{tag(cfg)}: deterministic env_action"
    # observations
    if flav == "f64":
        bad = np.argwhere(~(rp["obs"] == bs).all(2))
        assert bad.size == 0, f"{tag(cfg)}: observation differs from the oracle plant at (step, env) {tuple(bad[0])}"
    else:
        want, got = rp["nxt"][:-1], bs[1:].astype(np.float64)
        if plant == "wt":   # measured: <= 8e-7 absolute on levels below 0.1 (the fp32 Euler chain near an empty tank)
            tol = 2e-5 * np.maximum(np.abs(want), 0.1)
            if obs_mode == "integrator":
                tol[..., 3] = 1e-4 + 1e-5 * np.abs(want[..., 3])
        else:
            tol = np.zeros_like(want)
            if obs_mode == "integrator":
                tol[..., 2] = 2e-5
            assert np.array_equal(got[..., 0], t32[rp["idx"][:-1]]), f"{tag(cfg)}: pH y is not the replay's table entry"
            want = want.copy()
            want[..., 0] = got[..., 0]
        bad = np.argwhere(~(np.abs(got - want) <= tol).all(2))
        assert bad.size == 0, (f"{tag(cfg)}: one-step plant replay off at (step, env) {tuple(bad[0] + [1, 0])}: "
                               f"{got[tuple(bad[0])]} vs {want[tuple(bad[0])]}")
    # reward and mask columns
    if flav == "f64":
        np.testing.assert_allclose(bo[..., 0], rp["rew"], rtol=1e-6, atol=1e-7)
    else:
        np.testing.assert_allclose(bo[..., 0], rp["rew"], rtol=1e-5, atol=1e-4)
    assert np.array_equal(bo[..., 1], np.where(done, np.float32(0.0), np.float32(0.99))), f"{tag(cfg)}: mask column"
    # final state
    fin = snapshot(env, cfg)
    assert np.array_equal(fin["t"], rp["t"]) and np.array_equal(fin["episode"], rp["episode"]), f"{tag(cfg)}: t / episode"
    ret, done_rets = episode_returns(bo[..., 0].astype(np.float64) if flav == "f32" else rp["rew"], done, st0["ep_return"], flav)
    if flav == "f64":
        np.testing.assert_allclose(fin["ep_return"], ret, rtol=1e-12, atol=1e-12)
    else:
        assert np.array_equal(fin["ep_return"].astype(np.float32), ret), f"{tag(cfg)}: ep_return"
    last = rp["nxt"][-1]
    if plant == "wt":
        for key in ("a1", "a2", "Kp"):
            assert np.array_equal(fin[key], rp[key]), key
        got_last = fin["frames"] if obs_mode == "stacking" else np.stack(
            [fin["h1"], fin["h2"], fin["r"]] + ([fin["I"]] if obs_mode == "integrator" else []), 1)
        if flav == "f64":
            assert np.array_equal(got_last, last)
        else:
            tol = 2e-5 * np.maximum(np.abs(last), 0.1)
            if obs_mode == "integrator":
                tol[:, 3] = 1e-4 + 1e-5 * np.abs(last[:, 3])
            assert (np.abs(got_last - last) <= tol).all(), f"{tag(cfg)}: final state"
    else:
        np.testing.assert_allclose(fin["x"], rp["x"], rtol=1e-12)
        assert np.array_equal(fin["qww_V"], rp["qww_V"]) and np.array_equal(fin["qc_V"], rp["qc_V"])
        np.testing.assert_allclose(fin["A"], rp["A"], rtol=1e-15)
        np.testing.assert_allclose(fin["B"], rp["B"], rtol=1e-14)
    # statistics
    st = out["stats"].cpu().numpy()
    assert st[2] == done.sum() and st[5] == n * T, f"{tag(cfg)}: stats dones {st[2]} vs {done.sum()}, steps {st[5]} vs {n * T}"
    np.testing.assert_allclose(st[0], done_rets.sum(), rtol=1e-9, atol=1e-9)
    np.testing.assert_allclose(st[1], (done_rets ** 2).sum(), rtol=1e-9, atol=1e-9)
    rsum = bo[..., 0].astype(np.float64).sum() if flav == "f32" else rp["rew"].sum()
    np.testing.assert_allclose(st[4], rsum, rtol=1e-9 if flav == "f32" else 1e-12, atol=1e-9)
    if flav == "f32":
        # and against fp64 sums of the replay's own rewards: within the per-step reward bound above, summed over the
        # steps of each episode, plus the fp32 accumulation (<= T ulp of the running sum; every reward here is <= 0)
        slack = 1e-4 + 1e-5 * np.abs(rp["rew"])
        r64, fin64 = episode_returns(rp["rew"], done, st0["ep_return"], "f64")
        sl, fin_sl = episode_returns(slack, done, np.zeros(n), "f64")
        assert (np.abs(fin["ep_return"] - r64) <= sl + 2e-5 * np.abs(r64) + 1e-6).all(), f"{tag(cfg)}: ep_return vs fp64 replay"
        assert abs(st[0] - fin64.sum()) <= fin_sl.sum() + 2e-5 * np.abs(fin64).sum() + 1e-6, f"{tag(cfg)}: stats[0] vs fp64"
        assert abs(st[1] - (fin64 ** 2).sum()) <= (fin_sl * (2 * np.abs(fin64) + fin_sl)).sum() + 4e-5 * (fin64 ** 2).sum() + 1e-6
        assert abs(st[4] - rp["rew"].sum()) <= slack.sum() + 2e-5 * np.abs(rp["rew"]).sum(), f"{tag(cfg)}: stats[4] vs fp64"


def run_case(V, oracle, cfg, n, T, errs, random_t=True):
    plant, obs_mode, kind, H, k, flav = cfg
    S = state_dim(cfg)
    seed = 1 + sum(map(ord, tag(cfg))) + n
    env_offset = 7 * n
    rng = np.random.default_rng(seed)
    sd = actor_params(kind, H, S, seed)
    pack = V.ActorPack(kind, S, H, 1 if kind == "modular" else 0).update(sd)
    env = make_env(V, cfg, n, seed, env_offset)
    if random_t:
        env.t.copy_(torch.as_tensor(rng.integers(0, WT_MAX if plant == "wt" else PH_MAX, n), dtype=torch.int32))
    saved = {key: getattr(env, key).clone() for key in state_fields(cfg)}
    st0 = snapshot(env, cfg)
    pn = None
    if plant == "wt":
        g = torch.Generator(device="cuda").manual_seed(seed)
        pn = tuple(torch.randn((T, n), generator=g, device="cuda", dtype=env.dtype) * 0.01 for _ in range(2))
    # deterministic run: routing, accuracy, plant
    out = rollout(env, cfg, T, pack, True, pn)
    check_network(cfg, kind, sd, pack, out, S, errs)
    check_plant(oracle, V, cfg, env, st0, out, pn, seed, env_offset, S)
    del out
    # stochastic runs from the same state: in-kernel Philox (exploration and process noise), two launches (tick0 = 0, T)
    for key, v in saved.items():
        getattr(env, key).copy_(v)
    env.tick = 0
    a_std = float(np.float32(np.exp(np.float32(pack.a_std_log))))
    for launch in range(2):
        tick0 = env.tick
        out = rollout(env, cfg, T, pack, False)
        check_stochastic(oracle, cfg, pack, out, S, seed, env_offset, tick0, a_std, env.dtype, rng, st0 if launch == 0 else None)
        del out


def report(cfg, errs, label):
    e = torch.cat(errs)
    mx, rms, mean = float(e.abs().max()), float(e.pow(2).mean().sqrt()), float(e.mean())
    print(f"\n{tag(cfg)} [{label}]: rows {e.numel()}, a_avg - net64: max {mx:.3e} rms {rms:.3e} mean {mean:+.3e}")
    return rms, mean, e.numel()


def check_bounds(cfg, rms, mean, rows):
    rb, mb = BOUNDS[tag(cfg)]
    assert rms <= rb, f"{tag(cfg)}: RMS error {rms:.3e} > {rb:.1e}"
    if rows >= MEAN_ROWS:
        assert abs(mean) <= mb, f"{tag(cfg)}: |mean error| {abs(mean):.3e} > {mb:.1e}"


@gpu
@pytest.mark.parametrize("n_label", N_LABELS)
@pytest.mark.parametrize("cfg", CONFIGS, ids=tag)
def test_rollout_parity(V, oracle, cfg, n_label):
    n = n_of(n_label)
    T = (WT_MAX if cfg[0] == "wt" else PH_MAX) + 20 if n <= 129 else 3
    errs = []
    run_case(V, oracle, cfg, n, T, errs)
    check_bounds(cfg, *report(cfg, errs, f"n={n} T={T}"))


@gpu
@pytest.mark.parametrize("cfg,T", SHORT, ids=[f"{tag(c)}-T{T}" for c, T in SHORT])
def test_rollout_parity_every_pass_a_tile_boundary(V, oracle, cfg, T):
    """T = 1 / 2 at 3 tiles per CTA: every network pass starts or ends a tile (the short-pass regime)."""
    n = n_of("3tiles-77")
    errs = []
    run_case(V, oracle, cfg, n, T, errs)
    check_bounds(cfg, *report(cfg, errs, f"n={n} T={T}"))


@gpu
@pytest.mark.parametrize("cfg,n", BENCH, ids=[f"{tag(c)}-{n}" for c, n in BENCH])
def test_rollout_parity_bench_geometry(V, oracle, cfg, n):
    """The env counts of the rollout benchmarks, 4 steps from the freshly reset state."""
    errs = []
    run_case(V, oracle, cfg, n, 4, errs, random_t=False)
    check_bounds(cfg, *report(cfg, errs, f"n={n} T=4"))


# ------------------------------------------------------------------------------------------------ dead rows
SENTINEL = 0x7FC0DEAD   # a quiet NaN no kernel computes


@gpu
@pytest.mark.parametrize("n_label", ("1", "129", "tile+1", "3tiles-77"))
@pytest.mark.parametrize("plant", ("wt", "ph"))
def test_dead_rows_write_nothing(V, plant, n_label):
    """Tail rows shadow the last env and write nothing: state arrays of n + pad entries and replay rows of length
    ld = n + pad, all padding filled with a sentinel, rollout over the first n.  Every pad entry keeps its sentinel and
    every live row is written."""
    import pime_b200._lib as L
    n, pad, T = n_of(n_label), 300, 3
    ld = n + pad
    cfg = ("wt", "integrator", "modular", 64, 0, "f32") if plant == "wt" else ("ph", "integrator", "modular", 32, 0, "f32")
    S = state_dim(cfg)
    pack = V.ActorPack("modular", S, cfg[3], 1).update(actor_params("modular", cfg[3], S, 5))
    env = make_env(V, cfg, ld, seed=9)
    env.t[:n].copy_(torch.as_tensor(np.random.default_rng(n).integers(0, WT_MAX if plant == "wt" else PH_MAX, n), dtype=torch.int32))
    for key in state_fields(cfg):
        v = getattr(env, key)
        v.view(torch.int64 if v.element_size() == 8 else torch.int32)[n:] = SENTINEL
    before = {key: getattr(env, key).clone() for key in state_fields(cfg)}
    bs = torch.full((T, ld, S), SENTINEL, dtype=torch.int32, device="cuda").view(torch.float32)
    bo = torch.full((T, ld, 4), SENTINEL, dtype=torch.int32, device="cuda").view(torch.float32)
    act = torch.full((T, ld), SENTINEL, dtype=torch.int32, device="cuda").view(torch.float32)
    shim = types.SimpleNamespace(n=n, state_dim=S, seed=env.seed, env_offset=env.env_offset, tick=0, dtype=env.dtype,
                                 device=env.device, status=env.status)
    keep = []
    a, out = V._rollout_args(shim, T, pack, prior_k(cfg), False, True, 1.0, 0.99, None, None, None, False, None, keep)
    a.buf_state, a.buf_other, a.env_action, a.ld = L.ptr(bs), L.ptr(bo), L.ptr(act), ld
    if plant == "wt":
        rc = L.lib().pime_wt_rollout_f32(C.byref(env.cfg), C.c_int64(n), C.byref(env._st), C.byref(a), L.stream_ptr())
    else:
        rc = L.lib().pime_ph_rollout_f32(C.byref(env.cfg), L.ptr(env.table), C.c_int64(n), C.byref(env._st), C.byref(a),
                                         L.stream_ptr())
    L.check(rc)
    env.check_status()
    for key, v in before.items():
        got = getattr(env, key)
        assert torch.equal(got[n:].view(torch.int32 if got.element_size() == 4 else torch.int64),
                           v[n:].view(torch.int32 if v.element_size() == 4 else torch.int64)), f"pad of {key} written"
        if key in ("t", "h1", "x"):
            assert not torch.equal(got[:n], v[:n]), f"live {key} not written"
    for name, buf in (("buf_state", bs), ("buf_other", bo), ("env_action", act)):
        bits = buf.view(torch.int32)
        assert bool((bits[:, n:] == SENTINEL).all()), f"{name}: a dead row wrote past n"
        assert not bool((bits[:, :n] == SENTINEL).any()), f"{name}: a live row was not written"
    st = out["stats"].cpu().numpy()
    assert st[5] == n * T


# ------------------------------------------------------------------------------------------------ fidelity mode
@gpu
@pytest.mark.parametrize("n", (33, 4099))
@pytest.mark.parametrize("cfg", [("wt", "integrator", "modular", 256, 0, "f32"), ("ph", "none", "plain", 128, 0, "f64")], ids=tag)
def test_fidelity_rollout_matches_fidelity_forward(V, cfg, n):
    """rollout_fp32_kernel (32 envs per CTA, fp32 CUDA cores): a_avg bit-identical to actor_forward_fp32_kernel on the
    recorded observations, and within 2e-5 of net64."""
    plant, obs_mode, kind, H, k, flav = cfg
    S = state_dim(cfg)
    sd = actor_params(kind, H, S, n + H)
    pack = V.ActorPack(kind, S, H, 1 if kind == "modular" else 0, precision="fp32").update(sd)
    env = make_env(V, cfg, n, seed=n)
    env.t.copy_(torch.as_tensor(np.random.default_rng(n).integers(0, WT_MAX if plant == "wt" else PH_MAX, n), dtype=torch.int32))
    T = 60
    out = rollout(env, cfg, T, pack, True)
    bs, a = out["buf_state"].reshape(-1, S), out["buf_other"][..., 2].reshape(-1).contiguous()
    assert bool(bitwise_equal(a, pack.forward(bs)).all())
    err = float((a.double() - net64(kind, sd, bs)).abs().max())
    print(f"\nfidelity {tag(cfg)} n={n}: max |a_avg - net64| = {err:.2e}")
    assert err <= 2e-5
