"""GPU tests of the scheduled rollout with an extension block (pime_*_rollout_schedule_ext_*, vec.rollout_schedule with
a [K, n] set-point matrix or policy='linear', scenarios.staircase_metrics / robust_map with policy and per-env
set-points):

  1. per-env set-points: one launch where env i tracks sequence i % 3 equals, bit for bit, three launches of the shared
     schedule on identical env copies (replay rows, env_action, metrics, every final state array), on the sampled cases
     of test_gpu_09; a matrix of equal columns equals the shared schedule;
  2. the linear policy in f64 equals scenarios.staircase(policy='linear') (the per-step loop of the prior and step
     kernels) bit for bit on every observation of both plants, process noise included; its metrics match an fp64
     recomputation;
  3. the linear policy in f32: every action is, bit for bit, clip(row . priorK) of its replay row as an fp32
     fused-multiply-add chain (what prior_kernel<float> computes), the metrics match an fp64 recomputation from the
     replay rows, and rows, actions, rewards and final state equal the f32 per-step loop bit for bit;
  4. robust_map(policy='linear') against the CPU oracle's clipped linear staircase;
  5. env-range shards with column slices of the set-point matrix give the metrics of one launch, for both policies;
  6. 2^23-member pH and 2^20-member water-tank maps over random per-env staircases in bounded memory.
"""
import numpy as np
import pytest
import torch

from test_gpu_09_schedule import (K_PH, K_WT, NSEG, SAMPLED, SEG_L, actor_params, begin_segment, bits, fields,
                                  make_env, make_pack, metrics_from, n_of, output, prior_k, tag)

pytestmark = pytest.mark.gpu

WT_SEQS = ((3.0, 6.0, 9.0, 4.0), (8.0, 2.0, 5.0, 7.0), (1.0, 9.5, 4.0, 6.0))
PH_SEQS = ((10.0, 6.0, 3.0, 8.0), (5.0, 9.0, 4.0, 7.0), (8.0, 3.5, 10.0, 6.0))


@pytest.fixture(scope="module")
def V():
    import pime_b200.vec as vec
    return vec


def seq_matrix(seqs, n):
    """[K, n] float64: column i is seqs[i % len(seqs)]."""
    s = torch.tensor(seqs, dtype=torch.float64, device="cuda")
    return s[torch.arange(n, device="cuda") % len(seqs)].t().contiguous()


@pytest.mark.parametrize("case,n_label,resample,deterministic", SAMPLED,
                         ids=[f"{tag(c)}-n{nl}-rs{rs}-{'det' if d else 'sto'}" for c, nl, rs, d in SAMPLED])
def test_per_env_setpoints_equal_shared_launches(V, case, n_label, resample, deterministic):
    n = n_of(n_label)
    seqs = WT_SEQS if case[0] == "wt" else PH_SEQS
    pack = make_pack(V, case)
    kw = dict(actor=pack, deterministic=deterministic, replay=True, want_actions=True, resample_params=bool(resample))
    per_env = make_env(V, case, n)
    out = per_env.rollout_schedule(seq_matrix(seqs, n), SEG_L, prior_k(case), **kw)
    per_env.check_status()
    assert out["metrics"].shape == (4, NSEG, n)
    env_id = torch.arange(n, device="cuda")
    for j, seq in enumerate(seqs):
        ref = make_env(V, case, n)
        want = ref.rollout_schedule(seq, SEG_L, prior_k(case), **kw)
        ref.check_status()
        mask = env_id % 3 == j
        for k in ("buf_state", "buf_other", "env_action"):
            assert torch.equal(bits(out[k][:, mask]), bits(want[k][:, mask])), (j, k)
        assert torch.equal(bits(out["metrics"][..., mask]), bits(want["metrics"][..., mask])), j
        for k, v in fields(ref).items():
            got = getattr(per_env, k)
            assert torch.equal(bits(got[..., mask]), bits(v[..., mask])), (j, k)
        if j == 0:   # equal columns: the same launch as the shared schedule
            eq = make_env(V, case, n)
            got = eq.rollout_schedule(torch.tensor(seq, dtype=torch.float64).reshape(-1, 1).expand(NSEG, n), SEG_L,
                                      prior_k(case), **kw)
            eq.check_status()
            for k in ("buf_state", "buf_other", "env_action", "metrics"):
                assert torch.equal(bits(got[k]), bits(want[k])), k
            for k, v in fields(ref).items():
                assert torch.equal(bits(getattr(eq, k)), bits(v)), k


# ------------------------------------------------------------------------------------------------ linear policy
# (plant, observation, num_stack); K is the reference's K (the action is clip(-obs . K))
LINEAR_CASES = [("wt", "goal", 0), ("wt", "integrator", 0), ("wt", "stacking", 4), ("ph", "none", 0),
                ("ph", "integrator", 0), ("ph", "nobound", 0)]
LIN_L, LIN_N = 40, 300


def lin_case(plant, obs, k, dt):
    return (plant, obs, None, 0, k, dt, "tc", False)


def start_of(env):
    return (1.5, 0.5) if hasattr(env, "h1") else (14.0,)


def set_start(env, start):
    if hasattr(env, "h1"):
        env.set_state(*start)
    else:
        env.x.fill_(float(start[0]))


def fused_linear(V, c, seqs_or_seq, n, noise):
    """the linear staircase as one scheduled launch from start_of(env), step limit lifted as scenarios.staircase does"""
    env = make_lin_env(V, c, n, noise)
    set_start(env, start_of(env))
    st0 = {k: v.clone() for k, v in fields(env).items()}
    tick0 = env.tick
    out = env.rollout_schedule(seqs_or_seq, LIN_L, prior_k(c), deterministic=True, replay=True, want_actions=True,
                               policy="linear")
    env.check_status()
    return env, out, st0, tick0


def make_lin_env(V, c, n, noise):
    env = make_env(V, c, n)
    if hasattr(env, "h1"):
        env.cfg.max_step = 2 ** 30
        env.cfg.noise_scale = 0.01 if noise else 0.0
    else:
        env.cfg.max_episode_steps = 2 ** 30
    return env


@pytest.mark.parametrize("plant,obs,k", LINEAR_CASES, ids=[f"{p}-{o}{k or ''}" for p, o, k in LINEAR_CASES])
def test_linear_policy_f64_equals_the_per_step_staircase(V, plant, obs, k):
    import pime_b200.scenarios as SC
    c = lin_case(plant, obs, k, "f64")
    seq = WT_SEQS[0] if plant == "wt" else PH_SEQS[0]
    for noise in ((False, True) if plant == "wt" else (False,)):
        env, out, st0, tick0 = fused_linear(V, c, seq, LIN_N, noise)
        ref = make_lin_env(V, c, LIN_N, noise)
        K = -prior_k(c)
        res = SC.staircase(ref, "linear", K, setpoints=seq, steps=LIN_L, start=start_of(ref))
        ref.check_status()
        assert torch.equal(bits(out["buf_state"]), bits(res["obs"])), noise
        assert torch.equal(bits(out["env_action"].float()), bits(res["actions"])), noise
        assert torch.equal(bits(out["buf_other"][..., 0]), bits(res["rewards"])), noise
        assert (out["buf_other"][..., 1:] == torch.tensor([0.99, 0.0, 0.0], device="cuda")).all()
        for name, v in fields(ref).items():
            assert torch.equal(bits(getattr(env, name)), bits(v)), (noise, name)
        if plant == "wt":
            assert (out["env_action"].abs() <= 1).all()
        # metrics: fp64 recomputation from an open-loop replay of env_action through the step kernel
        rep = make_lin_env(V, c, LIN_N, noise)
        for name, v in fields(rep).items():
            v.copy_(st0[name])
        rep.tick = tick0
        T = NSEG * LIN_L
        ys, rs, rews, yb = [], [], [], []
        for s in range(T):
            if s % LIN_L == 0:
                begin_segment(rep, seq[s // LIN_L], False)
                yb.append(output(rep).double().clone())
            _, rew, _ = rep.step(out["env_action"][s])
            ys.append(output(rep).double().clone()); rs.append(rep.r.double().clone()); rews.append(rew.double())
        rep.check_status()
        want = metrics_from(torch.stack(ys), torch.stack(rs), torch.stack(rews), torch.stack(yb), NSEG, LIN_L)
        torch.testing.assert_close(out["metrics"], want, rtol=1e-12, atol=0)


def fmaf(a, b, c):
    """fp32 fused multiply-add, correctly rounded: a b is exact in fp64; TwoSum gives a b + c = s + e exactly, and the
    fp64 sum s rounds to the fp32 nearest to a b + c except on an fp32 tie, which the sign of e breaks."""
    a, b, c = (np.asarray(v, np.float32) for v in (a, b, c))
    p, c64 = a.astype(np.float64) * b.astype(np.float64), c.astype(np.float64)
    s = p + c64
    bv = s - p
    e = (p - (s - bv)) + (c64 - bv)
    r = s.astype(np.float32)
    r64 = r.astype(np.float64)
    other = np.nextafter(r, np.where(s > r64, np.float32(np.inf), np.float32(-np.inf))).astype(np.float32)
    o64 = other.astype(np.float64)
    tie = (s != r64) & (2.0 * s == r64 + o64)
    return np.where(tie & (e != 0) & (np.sign(e) == np.sign(o64 - s)), other, r)


def _linear_f32(rows, K):
    """-(row . K) in fp32 as prior_kernel<float> forms it: one fused multiply-add per term in k order, unclipped"""
    acc = np.zeros(rows.shape[:-1], np.float32)
    for j in range(rows.shape[-1]):
        acc = fmaf(rows[..., j], np.float32(K[j]), acc)
    return -acc


@pytest.mark.parametrize("plant,obs,k", LINEAR_CASES, ids=[f"{p}-{o}{k or ''}" for p, o, k in LINEAR_CASES])
def test_linear_policy_f32_actions_and_metrics_from_replay_rows(V, plant, obs, k):
    import pime_b200.scenarios as SC
    c = lin_case(plant, obs, k, "f32")
    seqs = WT_SEQS if plant == "wt" else PH_SEQS
    env, out, st0, tick0 = fused_linear(V, c, seq_matrix(seqs, LIN_N), LIN_N, True)
    K = -prior_k(c)
    rows = out["buf_state"].cpu().numpy()
    act = out["env_action"].cpu().numpy()
    lin = _linear_f32(rows, K)
    want = np.clip(lin, -1, 1) if plant == "wt" else lin
    assert np.array_equal(act.view(np.int32), want.view(np.int32)), np.abs(act - want).max()
    assert (out["buf_other"][..., 2:] == 0).all()
    T = NSEG * LIN_L
    if obs != "stacking":
        # y after step s: the next row's output (a reset_r segment begin keeps h1, h2 / x and C); after the last step: the
        # final state.  r: the row's set-point; y at a segment begin: its first row.
        o = out["buf_state"].double()
        yi, ri = (1, 2) if plant == "wt" else (0, 1)
        y = torch.cat([o[1:, :, yi], output(env).double()[None]])
        ref_m = metrics_from(y, o[:, :, ri], out["buf_other"][..., 0].double(), o[::LIN_L, :, yi], NSEG, LIN_L)
        torch.testing.assert_close(out["metrics"], ref_m, rtol=1e-12, atol=0)
    # the f32 per-step loop of scenarios.staircase, env by env on its own sequence: bit for bit the same (the fused
    # plant and the step kernel agree in f32 on these cases, and both policies form the same FMA chain)
    for j, seq in enumerate(seqs):
        ref = make_lin_env(V, c, LIN_N, True)
        res = SC.staircase(ref, "linear", K, setpoints=seq, steps=LIN_L, start=start_of(ref))
        ref.check_status()
        mask = torch.arange(LIN_N, device="cuda") % 3 == j
        assert torch.equal(bits(out["buf_state"][:, mask]), bits(res["obs"][:, mask])), j
        assert torch.equal(bits(out["env_action"][:, mask]), bits(res["actions"][:, mask])), j
        assert torch.equal(bits(out["buf_other"][:, mask, 0]), bits(res["rewards"][:, mask])), j
        for name, v in fields(ref).items():
            assert torch.equal(bits(getattr(env, name)[..., mask]), bits(v[..., mask])), (j, name)


# ------------------------------------------------------------------------------------------------ maps
def test_robust_map_linear_matches_the_oracle_staircase(V, oracle):
    """robust_map(policy='linear'), water tank f64, no noise, against the oracle stepping clip(-obs . K, -1, 1) in fp64."""
    import pime_b200.scenarios as SC
    steps = 60
    K = -K_WT
    m, params = SC.robust_map(K, SC.ROBUST_TESTS, plant="wt", steps=steps, dtype=torch.float64, noise_scale=0.0,
                              policy="linear")
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
            a = np.clip(-(np.stack([h1, h2, r, I], 1) @ K), -1.0, 1.0)
            rew, _ = oracle.wt_step(cfg, h1, h2, r, I, t, a1, a2, Kp, a)
            e = r - h2
            want[0, k] += rew
            want[1, k] += np.abs(e)
            want[2, k] = np.abs(e)
            want[3, k] = np.maximum(want[3, k], np.where(up, h2 - r, r - h2))
    for j, name in enumerate(SC.METRICS):
        np.testing.assert_allclose(m[name].cpu().numpy(), want[j], rtol=1e-9, atol=1e-12, err_msg=name)
    # the first action: 0.4 (3 - 0) = 1.2 for the agent's prior term, clipped to 1.0 by the linear policy
    first = {}
    for policy in ("actor", "linear"):
        env = V.WaterTankVec(n, dtype=torch.float64, max_step=2 ** 30, noise_scale=0.0)
        env.reset()
        env.reset_changable_parameters(*(torch.as_tensor(params[:, j]) for j in range(3)))
        env.set_state(0.0, 0.0)
        first[policy] = env.rollout_schedule(SC.WT_INTEGRATOR_SETPOINTS, 1, -K, deterministic=True, want_actions=True,
                                             policy=policy)["env_action"][0]
    assert (first["linear"] == 1.0).all()
    torch.testing.assert_close(first["actor"], torch.full_like(first["actor"], 1.2), rtol=1e-6, atol=1e-6)


@pytest.mark.parametrize("policy", ["agent", "linear"])
def test_shards_with_setpoint_column_slices_equal_one_launch(V, policy):
    import pime_b200.scenarios as SC
    c = ("wt", "integrator", "modular", 64, 0, "f32", "tc", False)
    n, h = 1000, 437
    pack = make_pack(V, c) if policy == "agent" else None
    whole = make_env(V, c, n, seed=3)
    parts = [make_env(V, c, h, seed=3), make_env(V, c, n - h, seed=3, env_offset=h)]
    for k, v in fields(whole).items():
        getattr(parts[0], k).copy_(v[..., :h])
        getattr(parts[1], k).copy_(v[..., h:])
    g = torch.Generator(device="cuda").manual_seed(5)
    sp = torch.rand((4, n), generator=g, device="cuda", dtype=torch.float64) * 10
    kw = dict(actor=pack, steps=13, resample_params=True, start=(1.0, 2.0), policy=policy)
    one = SC.staircase_metrics(whole, -K_WT, setpoints=sp, **kw)
    two = [SC.staircase_metrics(parts[0], -K_WT, setpoints=sp[:, :h], **kw),
           SC.staircase_metrics(parts[1], -K_WT, setpoints=sp[:, h:], **kw)]
    for name in SC.METRICS:
        assert one[name].shape == (4, n)
        assert torch.equal(bits(one[name]), bits(torch.cat([two[0][name], two[1][name]], 1))), name


@pytest.mark.parametrize("plant,policy", [("ph", "linear"), ("ph", "agent"), ("wt", "linear"), ("wt", "agent")])
def test_maps_over_random_per_env_staircases_in_bounded_memory(V, plant, policy):
    """2^23 pH members (5 x 50 steps, Modular-128) or 2^20 water-tank members (5 x 500 steps, Modular-256), each with its
    own random staircase in [r_lo, r_hi]: finite metrics and no trajectory buffers."""
    import pime_b200._lib as L
    import pime_b200.scenarios as SC
    n = 1 << (23 if plant == "ph" else 20)
    rng = np.random.default_rng(0)
    if plant == "ph":
        params = np.stack([rng.uniform(0.005, 0.015, n), rng.uniform(0.0015, 0.0025, n)], 1)
        cfg, S, H, K = L.ph_config(), 3, 128, -K_PH
    else:
        params = np.stack([rng.uniform(0.0015, 0.0024, n), rng.uniform(0.0015, 0.0024, n), rng.uniform(0.07, 0.17, n)], 1)
        cfg, S, H, K = L.wt_config(), 4, 256, -K_WT
    pack = V.ActorPack("modular", S, H, 1).update(actor_params("modular", H, S, 5)) if policy == "agent" else None
    g = torch.Generator(device="cuda").manual_seed(9)
    sp = cfg.r_lo + (cfg.r_hi - cfg.r_lo) * torch.rand((5, n), generator=g, device="cuda", dtype=torch.float64)
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    m, p = SC.robust_map(K, params, actor=pack, plant=plant, setpoints=sp, policy=policy)
    torch.cuda.synchronize()
    peak = torch.cuda.max_memory_allocated() - base
    env_state = n * (60 if plant == "ph" else 4 * 16)   # the vec's per-env arrays
    assert peak < env_state + sp.numel() * 8 + 4 * 5 * n * 8 + (1 << 30), peak
    assert p.shape[0] == n
    for name in SC.METRICS:
        assert m[name].shape == (5, n) and torch.isfinite(m[name]).all(), name
