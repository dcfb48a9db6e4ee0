"""GPU tests of the step response of a scheduled rollout (pime_*_rollout_schedule_response_*, vec.rollout_schedule with
response=True, scenarios.staircase_metrics / robust_map with response=True):

  1. the launch with the response is the launch without it: bit-identical replay rows, env_action, metrics and final
     state, on every sampled case of test_gpu_09 and on the linear cases of test_gpu_10;
  2. settle, rise and peak_action equal, and effort matches to 1e-12, an fp64 recomputation from y after every step, y at
     each segment begin and the actions fed to the plant -- both plants, every observation, f32 and f64, the tcgen05,
     fidelity and prior-only kernels, both policies, shared and per-env set-points, reset_r and reset_all;
  3. robust_map(response=True) against the CPU oracle's staircase, for the clipped linear baseline (segments that never
     settle and never reach 90 %) and the prior-only agent (a first action of 1.2);
  4. env-range shards give the response of one launch bit for bit; dead tail rows write nothing;
  5. 2^20-member water-tank and 2^23-member pH maps with the response in bounded memory.
"""
import numpy as np
import pytest
import torch

from test_gpu_09_schedule import (K_PH, K_WT, NSEG, PH_SP, SAMPLED, SEG_L, WT_SP, _fma_prior_f32, actor_params,
                                  begin_segment, bits, fields, make_env, make_pack, n_of, obs_y, output, per_segment, prior_k,
                                  tag)
from test_gpu_10_schedule_ext import (LIN_L, LIN_N, LINEAR_CASES, PH_SEQS, WT_SEQS, lin_case, make_lin_env, seq_matrix,
                                      set_start, start_of)

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def V():
    import pime_b200.vec as vec
    return vec


def response_from(y, u, y_begin, r, K, L, band=0.02):
    """fp64 step response [4, K, n] from y [T, n] after every step, the actions u [T, n], y at each segment begin
    [K, n] and r [T, n], as include/pime_b200.h defines it."""
    n = y.shape[1]
    y, u, r = (a.double().reshape(K, L, n) for a in (y, u, r))
    r = r[:, 0]
    d = (r - y_begin).abs()
    j1 = torch.arange(1, L + 1, device=y.device, dtype=torch.float64)[None, :, None]
    outside = (r[:, None] - y).abs() > (band * d)[:, None]
    settle = torch.where(outside, j1, 0.0).amax(1)
    progress = torch.where((r >= y_begin)[:, None], y - y_begin[:, None], y_begin[:, None] - y)
    first = torch.where(progress >= (0.9 * d)[:, None], j1, float(L + 1)).amin(1)
    rise = torch.where(d == 0, 0.0, torch.where(first > L, -1.0, first))
    effort = torch.zeros_like(d)
    for j in range(1, L):   # in j order, as the kernel sums
        effort = effort + (u[:, j] - u[:, j - 1]).abs()
    return torch.stack([settle, rise, effort, u.abs().amax(1)])


def check_response(got, want):
    assert got.shape == want.shape and got.dtype == torch.float64
    for m in (0, 1, 3):
        assert torch.equal(got[m], want[m]), (m, (got[m] != want[m]).sum().item())
    torch.testing.assert_close(got[2], want[2], rtol=1e-12, atol=0)


def same_launch(out, want, env, ref):
    """the launch with the response is the launch without it"""
    for k in ("buf_state", "buf_other", "env_action", "metrics"):
        assert torch.equal(bits(out[k]), bits(want[k])), k
    # the episode / step counts are exact; the sums are atomics over CTAs, whose order differs from launch to launch
    assert torch.equal(out["stats"][[2, 5]], want["stats"][[2, 5]])
    torch.testing.assert_close(out["stats"], want["stats"], rtol=1e-12, atol=1e-300)
    for k, v in fields(ref).items():
        assert torch.equal(bits(getattr(env, k)), bits(v)), k


def replay(V, make, st0, tick0, actions, sp, L, resample):
    """Open-loop replay of the recorded plant actions through the step kernel from the initial state, segment k beginning
    as the scheduled launch does with r = sp[k] ([K, n]).  Returns y after every step, r and y at each segment begin."""
    rep = make()
    for k, v in fields(rep).items():
        v.copy_(st0[k])
    rep.tick = tick0
    ys, rs, yb = [], [], []
    for s in range(actions.shape[0]):
        if s % L == 0:
            begin_segment(rep, 0.0, resample)
            rep.r.copy_(sp[s // L])
            yb.append(output(rep).double().clone())
        rep.step(actions[s])
        ys.append(output(rep).double().clone()); rs.append(rep.r.double().clone())
    rep.check_status()
    return torch.stack(ys), torch.stack(rs), torch.stack(yb)


@pytest.mark.parametrize("case,n_label,resample,deterministic", SAMPLED,
                         ids=[f"{tag(c)}-n{nl}-rs{rs}-{'det' if d else 'sto'}" for c, nl, rs, d in SAMPLED])
def test_response_of_the_agent_policy(V, case, n_label, resample, deterministic):
    n = n_of(n_label)
    setpoints = WT_SP if case[0] == "wt" else PH_SP
    pack = make_pack(V, case)
    kw = dict(actor=pack, deterministic=deterministic, replay=True, want_actions=True, resample_params=bool(resample))
    env, ref = make_env(V, case, n), make_env(V, case, n)
    st0 = {k: v.clone() for k, v in fields(env).items()}
    tick0 = env.tick
    out = env.rollout_schedule(setpoints, SEG_L, prior_k(case), response=True, **kw)
    env.check_status()
    want = ref.rollout_schedule(setpoints, SEG_L, prior_k(case), **kw)
    ref.check_status()
    assert "response" not in want
    same_launch(out, want, env, ref)

    T = NSEG * SEG_L
    u = out["env_action"]
    if case[5] == "f32":
        # y after step s: the next row's observation inside a segment, the per-segment state after its last step (as
        # test_gpu_09 recomputes the metrics)
        _, y_begin, y_end = per_segment(make_env(V, case, n), case, setpoints, SEG_L, pack, deterministic, bool(resample))
        y_obs = obs_y(case, out["buf_state"]).double()
        y = torch.cat([y_obs[1:], y_obs[:1]]).reshape(NSEG, SEG_L, n)
        y[:, -1] = y_end
        y = y.reshape(T, n)
        r = torch.tensor(setpoints, dtype=env.dtype, device="cuda").double().repeat_interleave(SEG_L)[:, None].expand(T, n)
    else:
        sp = torch.tensor(setpoints, dtype=torch.float64, device="cuda")[:, None].expand(NSEG, n)
        y, r, y_begin = replay(V, lambda: make_env(V, case, n), st0, tick0, u, sp, SEG_L, bool(resample))
    got = out["response"]
    check_response(got, response_from(y, u, y_begin, r, NSEG, SEG_L))
    assert ((got[0] >= 0) & (got[0] <= SEG_L)).all() and ((got[1] >= -1) & (got[1] <= SEG_L)).all()
    if case[0] == "wt" and n > 1:   # the unclipped residual action exceeds the pump's range somewhere
        assert (got[3] > 1).any()


@pytest.mark.parametrize("dt", ["f32", "f64"])
@pytest.mark.parametrize("plant,obs,k", LINEAR_CASES, ids=[f"{p}-{o}{k or ''}" for p, o, k in LINEAR_CASES])
def test_response_of_the_linear_policy(V, plant, obs, k, dt):
    """f32: per-env set-points, settle band 0.02; f64: one shared staircase, settle band 0.1."""
    c = lin_case(plant, obs, k, dt)
    seqs = WT_SEQS if plant == "wt" else PH_SEQS
    sp = seq_matrix(seqs, LIN_N) if dt == "f32" else seqs[0]
    band = 0.02 if dt == "f32" else 0.1

    def make():
        e = make_lin_env(V, c, LIN_N, True)
        set_start(e, start_of(e))
        return e

    env, ref = make(), make()
    st0 = {name: v.clone() for name, v in fields(env).items()}
    tick0 = env.tick
    kw = dict(deterministic=True, replay=True, want_actions=True, policy="linear")
    out = env.rollout_schedule(sp, LIN_L, prior_k(c), response=True, settle_band=band, **kw)
    env.check_status()
    want = ref.rollout_schedule(sp, LIN_L, prior_k(c), **kw)
    ref.check_status()
    same_launch(out, want, env, ref)
    # the fused linear staircase equals the per-step loop of the step kernel bit for bit on these cases (test_gpu_10)
    spm = torch.as_tensor(sp, dtype=torch.float64, device="cuda")
    spm = spm if spm.ndim == 2 else spm[:, None].expand(NSEG, LIN_N)
    y, r, y_begin = replay(V, make, st0, tick0, out["env_action"], spm, LIN_L, False)
    got = out["response"]
    check_response(got, response_from(y, out["env_action"], y_begin, r, NSEG, LIN_L, band))
    if plant == "wt":
        assert (got[3] <= 1).all()


# ------------------------------------------------------------------------------------------------ known answer
def _oracle_response(oracle, params, steps, policy):
    """The water-tank staircase stepped by the CPU oracle in fp64 (reset_r: (a1, a2, Kp) kept, levels carried over, I
    and t restarted), with the step response of each segment: [4, 5, n]."""
    import pime_b200.scenarios as SC
    n = params.shape[0]
    cfg = oracle.wt_cfg(reward_type="square_distance")
    cfg.max_step = 2 ** 30
    h1, h2 = np.zeros(n), np.zeros(n)
    a1, a2, Kp = (np.ascontiguousarray(params[:, j]) for j in range(3))
    want = np.zeros((4, 5, n))
    j1 = np.arange(1, steps + 1)[:, None]
    for k, r_ in enumerate(SC.WT_INTEGRATOR_SETPOINTS):
        r, I, t = np.full(n, float(r_)), np.zeros(n), np.zeros(n, np.int32)
        yb, ys, us = h2.copy(), [], []
        for _ in range(steps):
            if policy == "linear":
                a = np.clip(np.stack([h1, h2, r, I], 1) @ K_WT, -1.0, 1.0)
            else:    # tanh(0) + obs32 . priorK, unclipped
                a = _fma_prior_f32(np.stack([h1, h2, r, I], 1).astype(np.float32), K_WT).astype(np.float64)
            oracle.wt_step(cfg, h1, h2, r, I, t, a1, a2, Kp, a)
            ys.append(h2.copy()); us.append(a)
        y, u = np.array(ys), np.array(us)
        d = np.abs(r - yb)
        outside = np.abs(r - y) > 0.02 * d
        reach = np.where(r >= yb, y - yb, yb - y) >= 0.9 * d
        want[0, k] = np.where(outside, j1, 0).max(0)
        want[1, k] = np.where(d == 0, 0, np.where(reach.any(0), np.where(reach, j1, steps + 1).min(0), -1))
        want[2, k] = np.abs(np.diff(u, axis=0)).sum(0)
        want[3, k] = np.abs(u).max(0)
    return want


@pytest.mark.parametrize("policy", ["linear", "agent"])
def test_robust_map_response_matches_the_oracle_staircase(V, oracle, policy):
    import pime_b200.scenarios as SC
    steps = 60
    m, params = SC.robust_map(-K_WT, SC.ROBUST_TESTS, plant="wt", steps=steps, dtype=torch.float64, noise_scale=0.0,
                              policy=policy, response=True)
    want = _oracle_response(oracle, params, steps, policy)
    for j, name in enumerate(SC.RESPONSE):
        got = m[name].cpu().numpy()
        if name in ("settle", "rise"):
            np.testing.assert_array_equal(got, want[j], err_msg=name)
        else:
            np.testing.assert_allclose(got, want[j], rtol=1e-9, atol=1e-12, err_msg=name)
    for name in SC.METRICS:
        assert m[name].shape == (5, params.shape[0])
    if policy == "linear":
        # the proportional baseline keeps a steady-state error: some segments never settle and never reach 90 %
        assert ((m["settle"] == steps) & (m["rise"] == -1)).any()
        assert (m["peak_action"] == 1.0).any() and (m["peak_action"] <= 1.0).all()
    else:
        # 0.4 (3 - 0) = 1.2: the first action is beyond the pump's range
        assert (m["peak_action"][0] >= 1.2 - 1e-6).all()


# ------------------------------------------------------------------------------------------------ invariance and tails
@pytest.mark.parametrize("policy", ["agent", "linear"])
def test_shards_give_the_response_of_one_launch(V, policy):
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
    kw = dict(actor=pack, steps=13, resample_params=True, start=(1.0, 2.0), policy=policy, response=True)
    one = SC.staircase_metrics(whole, -K_WT, setpoints=sp, **kw)
    two = [SC.staircase_metrics(parts[0], -K_WT, setpoints=sp[:, :h], **kw),
           SC.staircase_metrics(parts[1], -K_WT, setpoints=sp[:, h:], **kw)]
    for name in SC.METRICS + SC.RESPONSE:
        assert one[name].shape == (4, n)
        assert torch.equal(bits(one[name]), bits(torch.cat([two[0][name], two[1][name]], 1))), name


SENTINEL = -1234.5


@pytest.mark.parametrize("case", [("wt", "integrator", "modular", 32, 0, "f32", "tc", False),
                                  ("wt", "stacking", "plain", 64, 4, "f32", "tc", False),
                                  ("ph", "nobound", "plain", 64, 0, "f64", "fp32", False),
                                  ("ph", "none", None, 0, 0, "f32", "tc", False)], ids=tag)
def test_dead_tail_rows_write_no_response(V, case):
    """n = 256 P + 1: a response buffer padded past 4 K n keeps its sentinel; every element of [4][K][n] is written."""
    n = n_of("tile+1")
    env = make_env(V, case, n)
    setpoints = WT_SP if case[0] == "wt" else PH_SP
    buf = torch.full((4 * NSEG * n + 999,), SENTINEL, dtype=torch.float64, device="cuda")
    out = env.rollout_schedule(setpoints, 5, prior_k(case), actor=make_pack(V, case), deterministic=True,
                               response=buf[: 4 * NSEG * n].view(4, NSEG, n))
    env.check_status()
    assert out["response"].data_ptr() == buf.data_ptr()
    assert (buf[4 * NSEG * n:] == SENTINEL).all()
    assert (buf[: 4 * NSEG * n] != SENTINEL).all() and torch.isfinite(buf[: 4 * NSEG * n]).all()


# ------------------------------------------------------------------------------------------------ scale
@pytest.mark.parametrize("plant", ["wt", "ph"])
def test_maps_with_the_response_in_bounded_memory(V, plant):
    """2^20 water-tank members (5 x 500 steps, Modular-256) or 2^23 pH members (5 x 50 steps, Modular-128) with the step
    response: finite values in range, and no trajectory buffers."""
    import pime_b200._lib as L
    import pime_b200.scenarios as SC
    n = 1 << (23 if plant == "ph" else 20)
    rng = np.random.default_rng(0)
    if plant == "ph":
        params = np.stack([rng.uniform(0.005, 0.015, n), rng.uniform(0.0015, 0.0025, n)], 1)
        S, H, K, steps = 3, 128, -K_PH, L.ph_config().max_episode_steps
    else:
        params = np.stack([rng.uniform(0.0015, 0.0024, n), rng.uniform(0.0015, 0.0024, n), rng.uniform(0.07, 0.17, n)], 1)
        S, H, K, steps = 4, 256, -K_WT, 500
    pack = V.ActorPack("modular", S, H, 1).update(actor_params("modular", H, S, 5))
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    m, p = SC.robust_map(K, params, actor=pack, plant=plant, response=True)
    torch.cuda.synchronize()
    peak = torch.cuda.max_memory_allocated() - base
    env_state = n * (60 if plant == "ph" else 4 * 16)   # the vec's per-env arrays
    assert peak < env_state + 2 * 4 * 5 * n * 8 + (1 << 30), peak
    assert p.shape[0] == n
    for name in SC.METRICS + SC.RESPONSE:
        assert m[name].shape == (5, n) and torch.isfinite(m[name]).all(), name
    assert ((m["settle"] >= 0) & (m["settle"] <= steps)).all()
    assert ((m["rise"] >= -1) & (m["rise"] <= steps)).all()
    assert (m["effort"] >= 0).all() and (m["peak_action"] >= 0).all()
