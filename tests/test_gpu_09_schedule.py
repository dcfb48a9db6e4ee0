"""GPU tests of the scheduled rollout (pime_*_rollout_schedule_*, vec.rollout_schedule, scenarios.staircase_metrics /
robust_map): the set-point staircase as one fused launch.

  1. bit-identity with the per-segment protocol it replaces (reset -> restore the plant state -> set_r -> rollout, one
     launch per segment): replay rows, env_action and every array of the final env state, for every kernel (prior-only,
     tcgen05 plain / modular at H = 32 ... 256, fidelity), both plant flavours, reset_r and reset_all segment begins and
     the env counts of test_gpu_08 (a partial tile, a second tile on CTA 0);
  2. the per-env metrics against an fp64 recomputation (f32 plant: from the replay rows and the per-segment states; f64
     plant: from an open-loop replay of the recorded env_action through vec.step);
  3. robust_map against the CPU oracle's staircase;
  4. env-range shards with env_offset give the metrics of one launch; dead tail rows write nothing;
  5. a 2^20-member robustness map with the Modular-256 actor in bounded memory.
"""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

K_WT = np.array([0.0, -0.4, 0.4, 0.0])     # priorK of the reference scripts (obs . priorK = 0.4 (r - h2))
K_PH = np.array([0.02, -0.02, -0.035])
WT_SP, PH_SP = (3.0, 6.0, 9.0, 4.0), (10.0, 6.0, 3.0, 8.0)
N_LABELS = ("1", "129", "tile+1")

# (plant, observation, actor kind or None, H, num_stack, flavour, actor precision, step limit below L + reset_from_last)
CASES = [
    ("wt", "integrator", None, 0, 0, "f32", "tc", False),
    ("wt", "goal", None, 0, 0, "f64", "tc", False),
    ("wt", "stacking", None, 0, 4, "f32", "tc", True),
    ("ph", "none", None, 0, 0, "f64", "tc", False),
    ("wt", "integrator", "modular", 32, 0, "f32", "tc", False),
    ("wt", "integrator", "modular", 64, 0, "f64", "tc", False),
    ("wt", "integrator", "modular", 128, 0, "f32", "tc", True),
    ("wt", "integrator", "modular", 256, 0, "f32", "tc", False),
    ("wt", "goal", "plain", 32, 0, "f32", "tc", False),
    ("wt", "goal", "plain", 256, 0, "f64", "tc", False),
    ("wt", "stacking", "plain", 64, 1, "f32", "tc", True),
    ("wt", "stacking", "plain", 128, 4, "f64", "tc", False),
    ("wt", "stacking", "plain", 256, 10, "f32", "tc", False),
    ("ph", "integrator", "modular", 32, 0, "f32", "tc", True),
    ("ph", "integrator", "modular", 128, 0, "f64", "tc", False),
    ("ph", "nobound", "plain", 64, 0, "f32", "tc", False),
    ("ph", "nobound", "modular", 256, 0, "f32", "tc", False),
    ("ph", "none", "plain", 128, 0, "f32", "tc", False),
    ("ph", "none", "plain", 256, 0, "f64", "tc", True),
    ("wt", "integrator", "modular", 64, 0, "f32", "fp32", False),
    ("wt", "stacking", "plain", 32, 10, "f64", "fp32", False),
    ("ph", "nobound", "plain", 128, 0, "f32", "fp32", True),
]
# sampled cross product: each case gets one env count, one segment-begin kind and one policy noise setting
SAMPLED = [(c, N_LABELS[i % 3], i % 2, i % 4 != 3) for i, c in enumerate(CASES)]
NSEG, SEG_L, LIMIT = 4, 9, 5


def tag(c):
    plant, obs, kind, H, k, dt, prec, fl = c
    return f"{plant}-{obs}{k or ''}-{kind or 'prior'}{H or ''}-{dt}-{prec}{'-fromlast' if fl else ''}"


def state_dim(c):
    plant, obs, k = c[0], c[1], c[4]
    if plant == "wt":
        return {"goal": 3, "integrator": 4}.get(obs, 3 * k)
    return 2 if obs == "none" else 3


def prior_k(c):
    S = state_dim(c)
    if c[0] == "ph":
        return K_PH[:S].copy()
    if c[1] == "stacking":
        K = np.zeros(S)
        K[-3:] = K_WT[:3]   # the prior acts on the newest frame
        return K
    return K_WT[:S].copy()


def n_of(label):
    P = torch.cuda.get_device_properties(0).multi_processor_count
    return {"1": 1, "129": 129, "tile+1": 256 * P + 1}[label]


def actor_params(kind, H, S, seed):
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
    sd[shapes[-1][0] + ".weight"] = rng.normal(0, 0.1, (1, H)).astype(np.float32)
    return sd


def make_pack(V, c, seed=7):
    plant, obs, kind, H, k, dt, prec, fl = c
    if kind is None:
        return None
    S = state_dim(c)
    return V.ActorPack(kind, S, H, 1 if kind == "modular" else 0, precision=prec).update(actor_params(kind, H, S, seed))


def make_env(V, c, n, seed=11, env_offset=0):
    """A reset env with random levels / x and step counters, so that the restore and t = 0 of a segment begin show."""
    plant, obs, kind, H, k, dt, prec, fl = c
    dtype = torch.float32 if dt == "f32" else torch.float64
    g = torch.Generator(device="cuda").manual_seed(seed)
    if plant == "wt":
        kw = dict(max_step=LIMIT) if fl else {}
        env = V.WaterTankVec(n, dtype=dtype, obs_mode=obs, num_stack=k, seed=seed, env_offset=env_offset,
                             reset_from_last_state=fl, **kw)
        env.reset()
        env.h1.copy_(torch.rand(n, generator=g, device="cuda", dtype=torch.float64) * 10)
        env.h2.copy_(torch.rand(n, generator=g, device="cuda", dtype=torch.float64) * 10)
    else:
        kw = dict(max_episode_steps=LIMIT) if fl else {}
        env = V.PHVec(n, dtype=dtype, integrator=obs, seed=seed, env_offset=env_offset, reset_from_last_state=fl, **kw)
        env.reset()
        env.x.copy_(torch.rand(n, generator=g, device="cuda", dtype=torch.float64) * 40)
    env.t.copy_(torch.randint(0, 3, (n,), generator=g, device="cuda", dtype=torch.int32))
    return env


def fields(env):
    if hasattr(env, "h1"):
        names = ("h1", "h2", "r", "I", "a1", "a2", "Kp", "t", "episode", "ep_return", "frames", "last_h1", "last_h2")
    else:
        names = ("x", "y", "r", "I", "A", "B", "C", "qww_V", "qc_V", "t", "episode", "ep_return", "last_x")
    return {k: getattr(env, k) for k in names if getattr(env, k) is not None}


def bits(t):
    """The bytes of a tensor as integers (NaN == NaN, -0 != +0)."""
    return t.contiguous().view({4: torch.int32, 8: torch.int64}[t.element_size()])


def output(env):
    return env.h2 if hasattr(env, "h1") else env.y


def begin_segment(env, r, resample):
    """The per-segment protocol the scheduled launch replaces (utils/test.py:102-106, :1386-1388): reset(), set_state(the
    plant state before it), set_r(r)."""
    if hasattr(env, "h1"):
        keep = (env.h1.clone(), env.h2.clone())
        env.reset(resample_params=resample)
        env.set_state(*keep)
        env.set_r(r)
    else:
        keep = env.x.clone()
        env.reset(resample_params=resample)
        env.x.copy_(keep)
        idx = torch.round(env.C * env.x * 1e5).long().clamp_(0, env.table.numel() - 1)
        env.y.copy_(env.table[idx])
        env.r.fill_(float(r))


def per_segment(env, c, setpoints, L, pack, deterministic, resample):
    """One rollout launch per segment; returns the concatenated rows and the output y right after each segment begin
    and after each segment's last step (float64)."""
    outs, y0, y1 = [], [], []
    for r in setpoints:
        begin_segment(env, r, resample)
        y0.append(output(env).double().clone())
        outs.append(env.rollout(L, prior_k(c), actor=pack, deterministic=deterministic, replay=True, want_actions=True))
        y1.append(output(env).double().clone())
        env.check_status()
    cat = {k: torch.cat([o[k] for o in outs]) for k in ("buf_state", "buf_other", "env_action")}
    return cat, torch.stack(y0), torch.stack(y1)


def metrics_from(y, r, rew, y_begin, K, L):
    """fp64 metrics from y [T, n] after every step, r [T, n], rewards [T, n] and y at each segment begin [K, n]."""
    n = y.shape[1]
    y, r, rew = (a.reshape(K, L, n) for a in (y, r, rew))
    e = r - y
    up = (r[:, 0] >= y_begin)[:, None]
    ovs = torch.where(up, y - r, r - y).amax(1).clamp_min(0.0)
    return torch.stack([rew.sum(1), e.abs().sum(1), e[:, -1].abs(), ovs])


def obs_y(c, obs):
    """The controlled output in a replay row: y (pH), h2 of the newest frame (stacking), h2."""
    if c[0] == "ph":
        return obs[..., 0]
    return obs[..., -2] if c[1] == "stacking" else obs[..., 1]


@pytest.fixture(scope="module")
def V():
    import pime_b200.vec as vec
    return vec


@pytest.mark.parametrize("case,n_label,resample,deterministic", SAMPLED,
                         ids=[f"{tag(c)}-n{nl}-rs{rs}-{'det' if d else 'sto'}" for c, nl, rs, d in SAMPLED])
def test_schedule_equals_per_segment_protocol(V, case, n_label, resample, deterministic):
    n = n_of(n_label)
    setpoints = WT_SP if case[0] == "wt" else PH_SP
    pack = make_pack(V, case)
    sched, ref = make_env(V, case, n), make_env(V, case, n)
    st0 = {k: v.clone() for k, v in fields(sched).items()}
    tick0 = sched.tick
    out = sched.rollout_schedule(setpoints, SEG_L, prior_k(case), actor=pack, deterministic=deterministic, replay=True,
                                 want_actions=True, resample_params=bool(resample))
    sched.check_status()
    want, y_begin, y_end = per_segment(ref, case, setpoints, SEG_L, pack, deterministic, bool(resample))
    for k in ("buf_state", "buf_other", "env_action"):
        assert torch.equal(bits(out[k]), bits(want[k])), k
    for k, v in fields(ref).items():
        assert torch.equal(bits(getattr(sched, k)), bits(v)), k
    assert sched.tick == ref.tick == tick0 + NSEG * SEG_L

    # metrics against an fp64 recomputation
    got = out["metrics"]
    assert got.shape == (4, NSEG, n) and got.dtype == torch.float64
    T = NSEG * SEG_L
    if case[5] == "f32":
        # y after step s: the next row's observation inside a segment, the per-segment state after its last step; r: the
        # set-point in the plant's precision (a stacking row shows the reset's frames at a segment's first step)
        y_obs = obs_y(case, out["buf_state"]).double()
        y = torch.cat([y_obs[1:], y_obs[:1]]).reshape(NSEG, SEG_L, n)
        y[:, -1] = y_end
        r = torch.tensor(setpoints, dtype=sched.dtype, device="cuda").double().repeat_interleave(SEG_L)[:, None].expand(T, n)
        ref_m = metrics_from(y.reshape(T, n), r, out["buf_other"][..., 0].double(), y_begin, NSEG, SEG_L)
    else:
        # open-loop replay of the recorded plant actions through the step kernel, from the initial state
        rep = make_env(V, case, n)
        for k, v in fields(rep).items():
            v.copy_(st0[k])
        rep.tick = tick0
        ys, rs, rews, yb = [], [], [], []
        for s in range(T):
            if s % SEG_L == 0:
                begin_segment(rep, setpoints[s // SEG_L], bool(resample))
                yb.append(output(rep).double().clone())
            _, rew, _ = rep.step(out["env_action"][s])
            ys.append(output(rep).double().clone()); rs.append(rep.r.double().clone()); rews.append(rew.double())
        rep.check_status()
        ref_m = metrics_from(torch.stack(ys), torch.stack(rs), torch.stack(rews), torch.stack(yb), NSEG, SEG_L)
    torch.testing.assert_close(got, ref_m, rtol=1e-12, atol=0)
    assert torch.equal(sched.r, torch.full_like(sched.r, setpoints[-1]))


def _fma_prior_f32(obs32, pk):
    """obs32 . priorK as the kernel's chain of fmaf (one rounding per term): exact products in fp64, rounded to fp32."""
    acc = np.zeros(obs32.shape[0], np.float32)
    for k in range(pk.shape[0]):
        acc = (obs32[:, k].astype(np.float64) * np.float64(np.float32(pk[k])) + acc.astype(np.float64)).astype(np.float32)
    return acc


def test_robust_map_matches_the_oracle_staircase(oracle):
    """robust_map (water tank, f64, prior-only, no noise) against the CPU oracle stepping the same staircase: reset_r keeps
    (a1, a2, Kp), the levels carry over, I and t restart, r steps through 3, 6, 9, 4, 2."""
    import pime_b200.scenarios as SC
    steps = 60
    m, params = SC.robust_map(-K_WT, SC.ROBUST_TESTS, plant="wt", steps=steps, dtype=torch.float64, noise_scale=0.0)
    n = params.shape[0]
    cfg = oracle.wt_cfg(reward_type="square_distance")
    cfg.max_step = 2 ** 30
    h1, h2 = np.zeros(n), np.zeros(n)
    a1, a2, Kp = (np.ascontiguousarray(params[:, j]) for j in range(3))
    want = np.zeros((4, 5, n))
    for k, r_ in enumerate(SC.WT_INTEGRATOR_SETPOINTS):
        r, I, t = np.full(n, float(r_)), np.zeros(n), np.zeros(n, np.int32)
        up = r >= h2
        for _ in range(steps):
            obs32 = np.stack([h1, h2, r, I], 1).astype(np.float32)
            a = _fma_prior_f32(obs32, K_WT).astype(np.float64)     # tanh(0) + obs32 . priorK, priorK = -K
            rew, _ = oracle.wt_step(cfg, h1, h2, r, I, t, a1, a2, Kp, a)
            e = r - h2
            want[0, k] += rew
            want[1, k] += np.abs(e)
            want[2, k] = np.abs(e)
            want[3, k] = np.maximum(want[3, k], np.where(up, h2 - r, r - h2))
    for j, name in enumerate(SC.METRICS):
        np.testing.assert_allclose(m[name].cpu().numpy(), want[j], rtol=1e-9, atol=1e-12, err_msg=name)
    assert (m["ret"] < 0).all() and (m["iae"] > 0).all()


def test_staircase_metrics_of_env_range_shards_equal_one_launch(V):
    """Two launches over the halves of the env range (env_offset) give bit for bit the metrics of one launch: every random
    stream (reset, exploration, process noise) is keyed by the global env id."""
    import pime_b200.scenarios as SC
    c = ("wt", "integrator", "modular", 64, 0, "f32", "tc", False)
    n, h = 1000, 437
    pack = make_pack(V, c)
    whole = make_env(V, c, n, seed=3)
    parts = [make_env(V, c, h, seed=3), make_env(V, c, n - h, seed=3, env_offset=h)]
    # make_env draws its random start from a per-env-count generator: give the shards the whole range's start
    for k, v in fields(whole).items():
        getattr(parts[0], k).copy_(v[:h])
        getattr(parts[1], k).copy_(v[h:])
    kw = dict(actor=pack, setpoints=WT_SP, steps=13, resample_params=True, start=(1.0, 2.0))
    one = SC.staircase_metrics(whole, K_WT * -1, **kw)
    two = [SC.staircase_metrics(p, K_WT * -1, **kw) for p in parts]
    for name in SC.METRICS:
        assert one[name].shape == (4, n)
        assert torch.equal(bits(one[name]), bits(torch.cat([two[0][name], two[1][name]], 1))), name
    # stochastic policy through vec.rollout_schedule directly
    outs = [e.rollout_schedule(WT_SP, 7, prior_k(c), actor=pack, deterministic=False) for e in [whole] + parts]
    assert torch.equal(bits(outs[0]["metrics"]), bits(torch.cat([outs[1]["metrics"], outs[2]["metrics"]], 2)))


SENTINEL = -1234.5


@pytest.mark.parametrize("case,n", [(("wt", "integrator", "modular", 128, 0, "f32", "tc", False), 129),
                                    (("wt", "integrator", "modular", 32, 0, "f32", "tc", False), "tile+1"),
                                    (("ph", "nobound", "plain", 64, 0, "f64", "fp32", False), 33),
                                    (("ph", "none", None, 0, 0, "f32", "tc", False), 129)], ids=lambda v: str(v))
def test_dead_tail_rows_write_no_metrics(V, case, n):
    """A metrics buffer padded past 4 K n keeps its sentinel; every element of [4][K][n] is written."""
    n = n_of(n) if isinstance(n, str) else n
    env = make_env(V, case, n)
    setpoints = WT_SP if case[0] == "wt" else PH_SP
    buf = torch.full((4 * NSEG * n + 999,), SENTINEL, dtype=torch.float64, device="cuda")
    env.rollout_schedule(setpoints, 5, prior_k(case), actor=make_pack(V, case), deterministic=True,
                         metrics=buf[: 4 * NSEG * n].view(4, NSEG, n))
    env.check_status()
    assert (buf[4 * NSEG * n:] == SENTINEL).all()
    assert (buf[: 4 * NSEG * n] != SENTINEL).all() and torch.isfinite(buf[: 4 * NSEG * n]).all()


def test_robust_map_of_a_million_members_in_bounded_memory(V):
    """2^20 water-tank parameter sets, the Modular-256 actor, 5 x 500 steps: finite metrics, and the launch allocates no
    trajectory buffers (the replay rows of this staircase would be ~70 GB)."""
    import pime_b200.scenarios as SC
    n = 1 << 20
    rng = np.random.default_rng(0)
    params = np.stack([rng.uniform(0.0015, 0.0024, n), rng.uniform(0.0015, 0.0024, n), rng.uniform(0.07, 0.17, n)], 1)
    pack = V.ActorPack("modular", 4, 256, 1).update(actor_params("modular", 256, 4, 5))
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    m, p = SC.robust_map(-K_WT, params, actor=pack, plant="wt", steps=500)
    torch.cuda.synchronize()
    peak = torch.cuda.max_memory_allocated() - base
    env_state = n * 4 * 16            # the WaterTankVec's per-env arrays (fp32 / int32)
    assert peak < env_state + (1 << 30), peak
    assert p.shape == (n, 3)
    for name in SC.METRICS:
        assert m[name].shape == (5, n) and torch.isfinite(m[name]).all(), name
