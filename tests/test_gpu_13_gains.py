"""GPU tests of the scheduled rollout with per-env controller gains (pime_*_rollout_schedule_gains_*, vec.rollout_schedule
with a [S, n] priorK, scenarios.staircase_metrics / robust_map with a [S, n] K):

  1. a gain matrix whose columns all equal priorK is the _response launch with that priorK, bit for bit: replay rows,
     env_action, metrics, response, final state, stats and status -- on the non-stacking sampled cases of test_gpu_09 and
     the non-stacking linear cases of test_gpu_10 (both plants, every other observation, f32 and f64, the tcgen05,
     fidelity and prior-only kernels, deterministic and stochastic agent, linear policy, shared and per-env set-points,
     reset_r and reset_all);
  2. mixed gains: every env's outputs equal those of the shared-K launch run with its own gain, bit for bit;
  3. robust_map(policy='linear') over a (kp, ki) grid x plant rows against the fp64 CPU oracle's staircase stepped with
     each env's own K, for both plants;
  4. env-range shards with column slices of the gain matrix give the one-launch result; dead tail rows write nothing;
  5. a 2^20-member water-tank map (64 x 64 gains x 256 plants, Modular-256) and a 2^23-member pH map (linear) in bounded
     memory, whose nominal-gain envs equal a shared-K launch over the same plants;
  6. the Python layer's rejections.
"""
import numpy as np
import pytest
import torch

from test_gpu_09_schedule import (K_PH, K_WT, NSEG, PH_SP, SAMPLED, SEG_L, WT_SP, actor_params, bits, fields, make_env,
                                  make_pack, n_of, prior_k, tag)
from test_gpu_10_schedule_ext import (LIN_L, LIN_N, LINEAR_CASES, PH_SEQS, WT_SEQS, lin_case, make_lin_env, seq_matrix,
                                      set_start, start_of)

pytestmark = pytest.mark.gpu

OUTPUTS = ("buf_state", "buf_other", "env_action", "metrics", "response")
SAMPLED_NS = [s for s in SAMPLED if s[0][1] != "stacking"]
LINEAR_NS = [c for c in LINEAR_CASES if c[1] != "stacking"]


@pytest.fixture(scope="module")
def V():
    import pime_b200.vec as vec
    return vec


def columns(priorK, n):
    """[S, n] float64 on the device, every column priorK"""
    return torch.as_tensor(np.asarray(priorK, np.float64), device="cuda")[:, None].expand(len(priorK), n).contiguous()


def same_outputs(out, want, env, ref, mask=None):
    """bit-identical outputs and final state (of the envs in mask, or all with their stats: the sums are atomics over
    CTAs, whose order differs from launch to launch)"""
    def pick(t, time_major):
        if mask is None:
            return t
        return t[:, mask] if time_major else t[..., mask]
    for k in OUTPUTS:
        if k in want:
            tm = k in ("buf_state", "buf_other")
            assert torch.equal(bits(pick(out[k], tm)), bits(pick(want[k], tm))), k
    if mask is None:
        assert torch.equal(out["stats"][[2, 5]], want["stats"][[2, 5]])
        torch.testing.assert_close(out["stats"], want["stats"], rtol=1e-12, atol=1e-300)
    for k, v in fields(ref).items():
        assert torch.equal(bits(pick(getattr(env, k), False)), bits(pick(v, False))), k


def checked(env, fn):
    out = fn()
    torch.cuda.synchronize()
    status = int(env.status.item())
    env.check_status()
    return out, status


# ------------------------------------------------------------------------------------------------ 1. uniform gains
@pytest.mark.parametrize("case,n_label,resample,deterministic", SAMPLED_NS,
                         ids=[f"{tag(c)}-n{nl}-rs{rs}-{'det' if d else 'sto'}" for c, nl, rs, d in SAMPLED_NS])
def test_uniform_gains_equal_the_shared_launch(V, case, n_label, resample, deterministic):
    n = n_of(n_label)
    seqs = WT_SEQS if case[0] == "wt" else PH_SEQS
    sp = seq_matrix(seqs, n) if resample else (WT_SP if case[0] == "wt" else PH_SP)
    pack = make_pack(V, case)
    kw = dict(actor=pack, deterministic=deterministic, replay=True, want_actions=True, resample_params=bool(resample),
              response=True)
    env, ref = make_env(V, case, n), make_env(V, case, n)
    out, s1 = checked(env, lambda: env.rollout_schedule(sp, SEG_L, columns(prior_k(case), n), **kw))
    want, s0 = checked(ref, lambda: ref.rollout_schedule(sp, SEG_L, prior_k(case), **kw))
    assert s1 == s0
    same_outputs(out, want, env, ref)


@pytest.mark.parametrize("dt", ["f32", "f64"])
@pytest.mark.parametrize("plant,obs,k", LINEAR_NS, ids=[f"{p}-{o}" for p, o, k in LINEAR_NS])
def test_uniform_gains_equal_the_shared_linear_launch(V, plant, obs, k, dt):
    """f32: per-env set-points; f64: one shared staircase (with process noise on the water tank)"""
    c = lin_case(plant, obs, k, dt)
    seqs = WT_SEQS if plant == "wt" else PH_SEQS
    sp = seq_matrix(seqs, LIN_N) if dt == "f32" else seqs[0]

    def make():
        e = make_lin_env(V, c, LIN_N, True)
        set_start(e, start_of(e))
        return e

    env, ref = make(), make()
    kw = dict(deterministic=True, replay=True, want_actions=True, policy="linear", response=True)
    out, s1 = checked(env, lambda: env.rollout_schedule(sp, LIN_L, columns(prior_k(c), LIN_N), **kw))
    want, s0 = checked(ref, lambda: ref.rollout_schedule(sp, LIN_L, prior_k(c), **kw))
    assert s1 == s0
    same_outputs(out, want, env, ref)


# ------------------------------------------------------------------------------------------------ 2. mixed gains
MIXED = [("wt", "integrator", "modular", 64, 0, "f32", "tc", False, "agent", True),
         ("wt", "goal", "plain", 128, 0, "f64", "tc", False, "agent", False),
         ("ph", "integrator", "modular", 32, 0, "f32", "tc", False, "agent", False),
         ("ph", "nobound", "plain", 64, 0, "f64", "fp32", False, "agent", True),
         ("wt", "integrator", None, 0, 0, "f32", "tc", False, "linear", True),
         ("ph", "none", None, 0, 0, "f64", "tc", False, "agent", True)]


def gain_set(case, G):
    """G distinct priorK vectors around the reference's"""
    base = prior_k(case)
    return [base * (1.0 + 0.25 * g) + 0.01 * g * np.sign(base) for g in range(G)]


@pytest.mark.parametrize("n_label", ["1", "129", "tile+1"])
@pytest.mark.parametrize("mc", MIXED, ids=lambda m: f"{tag(m[:8])}-{m[8]}")
def test_mixed_gains_equal_one_launch_per_gain(V, mc, n_label):
    case, policy, deterministic = mc[:8], mc[8], mc[9]
    n = n_of(n_label)
    G = 3 + len(n_label) % 3   # 3 .. 5 gains
    gains = gain_set(case, G)
    # a seeded permutation: neighbouring rows of a 128-row group get different gains
    assign = torch.as_tensor(np.random.default_rng(n).permutation(n) % G, device="cuda")
    Kmat = torch.stack([torch.as_tensor(g, device="cuda") for g in gains], 1)[:, assign].contiguous()
    sp = WT_SP if case[0] == "wt" else PH_SP
    pack = make_pack(V, case)
    kw = dict(actor=pack, deterministic=deterministic, replay=True, want_actions=True, response=True,
              policy="actor" if policy == "agent" else "linear")
    env = make_env(V, case, n)
    out, _ = checked(env, lambda: env.rollout_schedule(sp, SEG_L, Kmat, **kw))
    for g, K in enumerate(gains):
        ref = make_env(V, case, n)
        want, _ = checked(ref, lambda: ref.rollout_schedule(sp, SEG_L, K, **kw))
        mask = assign == g
        if mask.any():
            same_outputs(out, want, env, ref, mask)


# ------------------------------------------------------------------------------------------------ 3. CPU oracle
def _grid(kps, kis, builder):
    kp, ki = np.meshgrid(kps, kis, indexing="ij")
    return np.stack([builder(a, b) for a, b in zip(kp.ravel(), ki.ravel())], 1)   # [S, G]


def _oracle_staircase(oracle, plant, K, params, setpoints, steps, cfg=None, table=None, sample_t=20.0):
    """fp64 linear staircase stepped by the CPU oracle with each env's own K ([S, n], reference sign): metrics and response
    [8, len(setpoints), n] in the order METRICS + RESPONSE.  cfg (oracle.wt_cfg / ph_cfg, its step limit is lifted here),
    table and sample_t (pH): the plant's configuration, by default the registered one."""
    n = params.shape[0]
    out = np.zeros((8, len(setpoints), n))
    j1 = np.arange(1, steps + 1)[:, None]
    if plant == "wt":
        cfg = cfg or oracle.wt_cfg(reward_type="square_distance")
        cfg.max_step = 2 ** 30
        h1, h2 = np.zeros(n), np.zeros(n)
        a1, a2, Kp = (np.ascontiguousarray(params[:, j]) for j in range(3))
    else:
        cfg = cfg or oracle.ph_cfg()
        cfg.max_episode_steps = 2 ** 30
        table = oracle.ph_table() if table is None else table
        A, B, Cc = oracle.ph_update_system(params[:, 0], params[:, 1], sample_t)
        x = np.zeros(n)
    for k, r_ in enumerate(setpoints):
        r, I, t = np.full(n, float(r_)), np.zeros(n), np.zeros(n, np.int32)
        if plant == "ph":
            y = np.array([table[oracle.ph_index(cfg, Cc[i] * x[i])] for i in range(n)])
        yb = (h2 if plant == "wt" else y).copy()
        up = r >= yb
        ret, iae, ovs = np.zeros(n), np.zeros(n), np.zeros(n)
        ys, us = [], []
        for _ in range(steps):
            st = np.stack([h1, h2, r, I] if plant == "wt" else [y, r, I])
            acc = np.zeros(n)
            for k_ in range(st.shape[0]):   # in k order, a rounded product and a rounded sum per term, as the kernel
                acc = acc + st[k_] * K[k_]
            a = -acc
            if plant == "wt":
                a = np.clip(a, -1.0, 1.0)
                rew, _ = oracle.wt_step(cfg, h1, h2, r, I, t, a1, a2, Kp, a)
                yy = h2
            else:
                rew, _ = oracle.ph_step(cfg, table, x, y, r, I, t, A, B, Cc, a)
                yy = y
            e = np.abs(r - yy)
            ret += rew; iae += e
            ovs = np.maximum(ovs, np.where(up, yy - r, r - yy))
            ys.append(yy.copy()); us.append(a)
        yv, u = np.array(ys), np.array(us)
        d = np.abs(r - yb)
        outside = np.abs(r - yv) > 0.02 * d
        reach = np.where(up, yv - yb, yb - yv) >= 0.9 * d
        out[:4, k] = ret, iae, e, ovs
        out[4, k] = np.where(outside, j1, 0).max(0)
        out[5, k] = np.where(d == 0, 0, np.where(reach.any(0), np.where(reach, j1, steps + 1).min(0), -1))
        out[6, k] = np.abs(np.diff(u, axis=0)).sum(0)
        out[7, k] = np.abs(u).max(0)
    return out


@pytest.mark.parametrize("plant", ["wt", "ph"])
def test_gain_map_matches_the_oracle_staircase(V, oracle, plant):
    import pime_b200.scenarios as SC
    steps = 40
    if plant == "wt":
        Kg = _grid([0.1, 0.4, 0.8, 1.5], [0.0, 0.01, 0.03, 0.08], lambda kp, ki: [0.0, kp, -kp, -ki])
        P = np.asarray(SC.ROBUST_TESTS)
        sp = SC.WT_INTEGRATOR_SETPOINTS
        kw = dict(noise_scale=0.0)
    else:
        Kg = _grid([0.01, 0.02, 0.03, 0.05], [0.0, 0.02, 0.035, 0.06], lambda kp, ki: [-kp, kp, ki])
        P = np.array([[0.01, 0.002], [0.012, 0.0018], [0.008, 0.0022]])
        sp = SC.PH_SETPOINTS
        kw = {}
    G, m = Kg.shape[1], P.shape[0]
    K = np.repeat(Kg, m, axis=1)
    params = np.tile(P, (G, 1))
    got, p = SC.robust_map(K, params, plant=plant, steps=steps, dtype=torch.float64, policy="linear", response=True,
                           setpoints=sp, **kw)
    assert p.shape == (G * m, P.shape[1])
    want = _oracle_staircase(oracle, plant, K, p, sp, steps)
    for j, name in enumerate(SC.METRICS + SC.RESPONSE):
        g = got[name].cpu().numpy()
        assert g.shape == (len(sp), G * m)
        if name in ("settle", "rise"):
            np.testing.assert_array_equal(g, want[j], err_msg=name)
        elif name == "peak_action":
            # the fp64 plants round like the oracle's to the last bits only: equal where the clip saturates, else 1e-12
            if plant == "wt":
                np.testing.assert_array_equal(g == 1.0, want[j] == 1.0, err_msg=name)
            np.testing.assert_allclose(g, want[j], rtol=1e-12, atol=0, err_msg=name)
        else:
            np.testing.assert_allclose(g, want[j], rtol=1e-9, atol=1e-12, err_msg=name)
    # the map is not flat: every (gain, plant) pair tracks differently
    assert len(np.unique(got["iae"].cpu().numpy()[0])) == G * m


# ------------------------------------------------------------------------------------------------ 4. shards and tails
@pytest.mark.parametrize("policy", ["agent", "linear"])
def test_shards_give_the_result_of_one_launch(V, policy):
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
    K = -torch.as_tensor(K_WT, device="cuda")[:, None] * (0.5 + torch.rand((1, n), generator=g, device="cuda",
                                                                            dtype=torch.float64))
    K[3] = -0.05 * torch.rand(n, generator=g, device="cuda", dtype=torch.float64)
    kw = dict(actor=pack, steps=13, resample_params=True, start=(1.0, 2.0), policy=policy, response=True)
    one = SC.staircase_metrics(whole, K, **kw)
    two = [SC.staircase_metrics(parts[0], K[:, :h], **kw), SC.staircase_metrics(parts[1], K[:, h:], **kw)]
    for name in SC.METRICS + SC.RESPONSE:
        assert one[name].shape == (len(SC.WT_INTEGRATOR_SETPOINTS), n)
        assert torch.equal(bits(one[name]), bits(torch.cat([two[0][name], two[1][name]], 1))), name
    for k, v in fields(whole).items():
        assert torch.equal(bits(v), bits(torch.cat([getattr(parts[0], k), getattr(parts[1], k)], -1))), k


SENTINEL = -1234.5


@pytest.mark.parametrize("case", [("wt", "integrator", "modular", 32, 0, "f32", "tc", False),
                                  ("ph", "nobound", "plain", 64, 0, "f64", "fp32", False),
                                  ("ph", "none", None, 0, 0, "f32", "tc", False)], ids=tag)
def test_dead_tail_rows_write_nothing(V, case):
    """n = 256 P + 1: metrics and response buffers padded past 4 K n keep their sentinel; every element is written."""
    n = n_of("tile+1")
    env = make_env(V, case, n)
    setpoints = WT_SP if case[0] == "wt" else PH_SP
    m = 4 * NSEG * n
    mbuf = torch.full((m + 999,), SENTINEL, dtype=torch.float64, device="cuda")
    rbuf = torch.full((m + 999,), SENTINEL, dtype=torch.float64, device="cuda")
    out = env.rollout_schedule(setpoints, 5, columns(prior_k(case), n), actor=make_pack(V, case), deterministic=True,
                               metrics=mbuf[:m].view(4, NSEG, n), response=rbuf[:m].view(4, NSEG, n))
    env.check_status()
    assert out["response"].data_ptr() == rbuf.data_ptr() and out["metrics"].data_ptr() == mbuf.data_ptr()
    for buf in (mbuf, rbuf):
        assert (buf[m:] == SENTINEL).all()
        assert (buf[:m] != SENTINEL).all() and torch.isfinite(buf[:m]).all()


# ------------------------------------------------------------------------------------------------ 5. scale
@pytest.mark.parametrize("plant", ["wt", "ph"])
def test_gain_maps_in_bounded_memory(V, plant):
    """water tank: 64 x 64 (kp, ki) x 256 plants = 2^20 envs, Modular-256 agent, 5 x 500 steps; pH: 2^23 envs, linear,
    5 x 50 steps.  Finite outputs in range; the envs with the nominal gain equal a shared-K launch over the same plants."""
    import pime_b200._lib as L
    import pime_b200.scenarios as SC
    rng = np.random.default_rng(0)
    if plant == "wt":
        m = 256
        P = np.stack([rng.uniform(0.0015, 0.0024, m), rng.uniform(0.0015, 0.0024, m), rng.uniform(0.07, 0.17, m)], 1)
        Kg = _grid(np.linspace(0.05, 1.6, 64), np.linspace(0.0, 0.06, 64), lambda kp, ki: [0.0, kp, -kp, -ki])
        Kg[:, 0] = -K_WT   # the nominal gain
        S, steps, policy = 4, 500, "agent"
        pack = V.ActorPack("modular", S, 256, 1).update(actor_params("modular", 256, S, 5))
    else:
        m = 512
        P = np.stack([rng.uniform(0.005, 0.015, m), rng.uniform(0.0015, 0.0025, m)], 1)
        Kg = _grid(np.linspace(0.005, 0.05, 128), np.linspace(0.0, 0.07, 128), lambda kp, ki: [-kp, kp, ki])
        Kg[:, 0] = -K_PH
        S, steps, policy, pack = 3, L.ph_config().max_episode_steps, "linear", None
    G = Kg.shape[1]
    n = G * m
    assert n == 1 << (20 if plant == "wt" else 23)
    params = np.tile(P, (G, 1))
    K = torch.as_tensor(np.repeat(Kg, m, axis=1), device="cuda")
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    got, p = SC.robust_map(K, params, actor=pack, plant=plant, policy=policy, response=True)
    torch.cuda.synchronize()
    peak = torch.cuda.max_memory_allocated() - base
    env_state = n * (60 if plant == "ph" else 4 * 16)
    assert peak < env_state + 2 * 4 * 5 * n * 8 + 2 * S * n * 8 + (1 << 30), peak
    for name in SC.METRICS + SC.RESPONSE:
        assert got[name].shape == (5, n) and torch.isfinite(got[name]).all(), name
    assert ((got["settle"] >= 0) & (got["settle"] <= steps)).all()
    assert ((got["rise"] >= -1) & (got["rise"] <= steps)).all()
    del K
    want, _ = SC.robust_map(-(K_WT if plant == "wt" else K_PH), params, actor=pack, plant=plant, policy=policy,
                            response=True)
    for name in SC.METRICS + SC.RESPONSE:   # gain 0 is the nominal one: rows 0 .. m - 1
        assert torch.equal(bits(got[name][:, :m]), bits(want[name][:, :m])), name


# ------------------------------------------------------------------------------------------------ 6. Python rejections
def test_python_rejections(V):
    import pime_b200.scenarios as SC
    env = V.WaterTankVec(8)
    env.reset()
    for bad in (np.zeros((3, 8)), np.zeros((4, 7)), np.zeros((4, 8, 1)), torch.zeros((8, 4))):
        with pytest.raises(ValueError):
            env.rollout_schedule(WT_SP, 5, bad)
        with pytest.raises(ValueError):
            SC.staircase_metrics(env, bad, steps=5)
    st = V.WaterTankVec(8, obs_mode="stacking", num_stack=2)
    st.reset()
    with pytest.raises(ValueError):
        st.rollout_schedule(WT_SP, 5, np.zeros((6, 8)))
    with pytest.raises(ValueError):
        SC.staircase(env, "linear", np.zeros((4, 8)), steps=5)
    ph = V.PHVec(8)
    ph.reset()
    with pytest.raises(ValueError):
        ph.rollout_schedule(PH_SP, 5, np.zeros((4, 8)))
    # a 2-D K goes through the fused launch for the agent policy
    res = SC.staircase(env, "agent", np.tile(-K_WT[:, None], (1, 8)), steps=5)
    assert res["actions"].shape == (5 * len(SC.WT_INTEGRATOR_SETPOINTS), 8)
