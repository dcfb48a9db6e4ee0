"""Both PPO minibatch steps against an fp64 reference of AgentPPO.update_net's minibatch (elegantrl/agent.py:635-652), at the
batch sizes the steps serve, at return scales of real replays, and at the edges of the kernels' row tiling.

* SIMT step (csrc/learner.cu, pime_ppo_step in grad_out mode): H 32..256, B 2..4096 (R = 2, 4, 8 rows per CTA, ragged last CTA).
* Tensor-core step (csrc/learner_tc.cu, pime_ppo_grad_tc): H 128 / 256, B 2048..2^20 (ragged last row tile).
* A sweep of std(r_sum) over 1e-2..1e4, mean(r_sum) in {0, -10 std} and a_std_log in {-3, -0.5, 1} on both steps.
* One real water-tank replay (explore_env + update_net's value / GAE pre-pass) on the tensor-core step.
* pime_ppo_apply_grad against an fp64 Adam (torch's fused formula), pime_gae_scan against an fp64 reverse recursion.

The reference runs float64 copies of the nets on the exact fp32 inputs the kernels read.  The bounds are fixed, the same at
every return scale, a_std_log and B: a bound that had to grow with the scale would be hiding a precision bug.

Some decisions switch a row's gradient on or off (the clipped-surrogate min, SmoothL1's |e| < 1, each critic ReLU); a row
that fp32 and fp64 decide differently moves a gradient entry by a whole row's contribution.  The minibatch is therefore
drawn only from rows whose decisions are clear of their thresholds (see _clear_rows); the count of excluded rows is printed.

Error metric: max |err| / max |ref| per gradient tensor.  A tensor of one element (a_std_log, the output-layer biases) and the
four objectives are single sums over the batch whose terms cancel; their error is measured against the sum of the absolute
row terms, which is what fp32 summation error scales with."""
import copy

import numpy as np
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

SIMT_BOUND = 2e-5
TC_BOUND = 5e-5
OBJ_BOUND = 1e-5
CHUNK = 1 << 16

# The tensor-core step's actor output carries the error of its fp16 hi + lo forward (a few 1e-6 absolute).  The log-prob
# amplifies it by |a - mean| / exp(a_std_log)^2, which at a_std_log = -3 is ~1e3: the ratio, and through it every actor
# gradient, then differs from fp64 by more than the step's own arithmetic does.  Those cases are checked twice: against an
# fp64 reference evaluated at the kernel's own actor output (TC_BOUND: the backward, carried gradients included, is exact
# to that bound), and against the plain fp64 reference with this named, fixed bound on the forward's amplified error.
TC_SMALL_STD = -3.0
TC_SMALL_STD_BOUND = 1e-3


# ------------------------------------------------------------------------------------------------ agents and data
_AGENTS = {}


def _agent(kind, S, H):
    """A fresh agent (cached per shape; callers deep-copy it) with a non-zero actor output layer."""
    import pime_b200.rl as R
    key = (kind, S, H)
    if key not in _AGENTS:
        torch.manual_seed(1000 * H + 10 * S + (kind == "modular"))
        agent = R.AgentResidualIntegratorModularPPO() if kind == "modular" else R.AgentResidualPPO()
        agent.init(H, S, 1, 1) if kind == "modular" else agent.init(H, S, 1)
        with torch.no_grad():
            agent.act.net[-1].weight.normal_(0, 0.1)
            agent.act.net[-1].bias.normal_(0, 0.1)
        _AGENTS[key] = agent
    agent = copy.copy(_AGENTS[key])
    agent.act, agent.cri = copy.deepcopy(agent.act), copy.deepcopy(agent.cri)
    agent._fused = None
    return agent


def _nets64(agent):
    act, cri = copy.deepcopy(agent.act).double(), copy.deepcopy(agent.cri).double()
    for p in list(act.parameters()) + list(cri.parameters()):
        p.grad = None
    return act, cri


def _data(agent, S, L, mean=-50.0, std=30.0, adv_scale=1.0, a_std_log=-0.5, lp_spread=0.3, seed=0):
    """L candidate rows: states on the plants' ranges (levels / set-points in [0, 12], the integrator column in +-25), actions
    drawn from the actor's own Gaussian, old log-probs off the new ones by N(0, lp_spread) (the ratio crosses both clip
    edges), r_sum ~ N(mean, std), advantages ~ N(0, adv_scale)."""
    with torch.no_grad():
        agent.act.a_std_log.fill_(a_std_log)
    dev = agent.device
    g = torch.Generator(device=dev).manual_seed(seed)
    state = torch.rand(L, S, device=dev, generator=g) * 12
    state[:, -1] = torch.rand(L, device=dev, generator=g) * 50 - 25
    std_a = float(np.exp(np.float32(a_std_log)))
    with torch.no_grad():
        a_avg = agent.act.a_avg(state).reshape(-1)
    noise = torch.randn(L, device=dev, generator=g)
    action = (a_avg + noise * std_a).contiguous()
    logprob = -(noise.pow(2) * 0.5 + a_std_log + agent.act.sqrt_2pi_log) + torch.randn(L, device=dev, generator=g) * lp_spread
    r_sum = torch.randn(L, device=dev, generator=g) * std + mean
    adv = torch.randn(L, device=dev, generator=g) * adv_scale
    return state.contiguous(), action, r_sum.contiguous(), logprob.contiguous(), adv.contiguous()


# ------------------------------------------------------------------------------------------------ fp64 reference
def _objective_sums(act, cri, x, action, r_sum, logprob, adv, B, cs, clip, lam, shift=None):
    """The objectives of agent.py:635-652 over rows x of a B-row minibatch whose r_sum.std() is cs: each mean is a sum / B,
    so a minibatch can be evaluated in row chunks whose losses (and gradients) add up.  Also returns the sums of the
    absolute row terms of each objective and the row terms of d united / d a_std_log and d united / d (output bias).
    shift (optional, per row, no gradient) moves the actor's output, e.g. onto the value a kernel computed."""
    mean = act.a_avg(x).reshape(-1)
    if shift is not None:
        mean = mean + shift
    asl = act.a_std_log.reshape(())
    new_lp = -(asl + act.sqrt_2pi_log + ((mean - action) / asl.exp()).pow(2) * 0.5)     # compute_logprob (net_residual.py:62-66)
    ratio = (new_lp - logprob).exp()
    s1, s2 = adv * ratio, adv * ratio.clamp(1 - clip, 1 + clip)
    sur_rows = -torch.min(s1, s2)
    ent_rows = new_lp.exp() * new_lp
    value = cri(x).squeeze(1)
    cri_rows = F.smooth_l1_loss(value, r_sum, reduction="none")
    oa = (sur_rows + ent_rows * lam).sum() / B
    oc = cri_rows.sum() / B
    ou = oa + oc / (cs + 1e-5)
    oe = ent_rows.sum() / B
    with torch.no_grad():
        std = act.a_std_log.exp().reshape(())
        dd = (mean - action) / std
        g_lp = (-torch.where(s1 <= s2, s1, torch.zeros_like(s1)) + lam * (ent_rows + new_lp.exp())) / B
        d_act = g_lp * (-dd / std)
        d_cri = (value - r_sum).clamp(-1, 1) / B / (cs + 1e-5)
        absum = {"united": float(((sur_rows + ent_rows * lam).abs().sum() + cri_rows.sum() / (cs + 1e-5)) / B),
                 "actor": float((sur_rows + ent_rows * lam).abs().sum() / B), "critic": float(cri_rows.sum() / B),
                 "entropy": float(ent_rows.abs().sum() / B), "a_std_log": float((g_lp * (dd * dd - 1)).abs().sum()),
                 "act_out_bias": float(d_act.abs().sum()), "cri_out_bias": float(d_cri.abs().sum())}
    return (oa, oc, ou, oe), absum


def _reference(act, cri, x, action, r_sum, logprob, adv, clip, lam, shift=None):
    """fp64 objectives, gradients (in act / cri .grad) and absolute-term sums of one minibatch, in chunks of CHUNK rows."""
    B = x.shape[0]
    cs = float(r_sum.std())
    tot = np.zeros(4)
    absum = {}
    for lo in range(0, B, CHUNK):
        sl = slice(lo, lo + CHUNK)
        objs, ab = _objective_sums(act, cri, x[sl], action[sl], r_sum[sl], logprob[sl], adv[sl], B, cs, clip, lam,
                                   None if shift is None else shift[sl])
        objs[2].backward()
        tot += [objs[2].item(), objs[0].item(), objs[1].item(), objs[3].item()]
        for k, v in ab.items():
            absum[k] = absum.get(k, 0.0) + v
    return tot, absum, cs


def _critic_preacts(cri, x):
    out, h = [], x
    for i in (0, 2, 4):
        z = cri.net[i](h)
        out.append(z)
        h = torch.relu(z)
    return out


def _clear_rows(agent, data, clip):
    """Rows whose branch decisions are clear of their thresholds in fp64: |ratio - (1 +- clip)| > 1e-4, ||e| - 1| > 1e-4 and
    every critic pre-activation |z| > 1e-5 max |z| of its layer (the maxima over all candidate rows)."""
    act, cri = _nets64(agent)
    state, action, r_sum, logprob, adv = (t.double() for t in data)
    L = state.shape[0]
    with torch.no_grad():
        zmax = [0.0, 0.0, 0.0]
        for lo in range(0, L, CHUNK):
            for i, z in enumerate(_critic_preacts(cri, state[lo:lo + CHUNK])):
                zmax[i] = max(zmax[i], float(z.abs().max()))
        keep = torch.empty(L, dtype=torch.bool, device=state.device)
        for lo in range(0, L, CHUNK):
            sl = slice(lo, lo + CHUNK)
            x = state[sl]
            ratio = (act.compute_logprob(x, action[sl].unsqueeze(1)) - logprob[sl]).exp()
            ok = ((ratio - (1 + clip)).abs() > 1e-4) & ((ratio - (1 - clip)).abs() > 1e-4)
            zs = _critic_preacts(cri, x)
            ok &= (cri(x).squeeze(1) - r_sum[sl]).abs().sub(1).abs() > 1e-4
            for i, z in enumerate(zs):
                ok &= (z.abs() > 1e-5 * zmax[i]).all(1)
            keep[sl] = ok
    return torch.nonzero(keep).reshape(-1), L - int(keep.sum())


def _draw(agent, data, B, clip, seed):
    rows, excluded = _clear_rows(agent, data, clip)
    g = torch.Generator(device=rows.device).manual_seed(seed)
    idx = rows[torch.randint(rows.numel(), size=(B,), device=rows.device, generator=g)].contiguous()
    return idx, excluded


# ------------------------------------------------------------------------------------------------ the kernels
def _decode(work, off, row_tiles, units):
    """T-format (tiles of 128 rows x 64 units, hi block + lo block, each [8 unit groups][128 rows][8 fp16]) -> [rows, units] fp32."""
    nb = row_tiles * (units // 64) * 2 * 16384
    raw = work[off:off + nb].view(torch.float16).view(row_tiles, units // 64, 2, 8, 128, 8).float()
    x = raw[:, :, 0] + raw[:, :, 1]
    return x.permute(0, 3, 1, 2, 4).reshape(row_tiles * 128, units)


def _kernel_grad(agent, data, idx, tc, want_out=False):
    """One step's flat gradient and loss row from pime_ppo_grad_tc (tc) or pime_ppo_step(grad_out); with want_out, the
    tensor-core step's actor output per row (its last hidden activation from the work buffer, times the output layer)."""
    import ctypes as C
    import pime_b200._lib as L
    import pime_b200.rl as R
    S, H = agent.state_dim, agent.net_dim
    f = R.FusedLearner(agent.act, agent.cri, S, H, agent.device)
    f.load(agent.act, agent.cri)
    grad = torch.zeros_like(f.theta)
    if tc:
        args = f._bind(data, idx, agent, True)
        L.check(L.lib().pime_ppo_grad_tc(args, L.ptr(f.work_tc), L.ptr(grad), L.stream_ptr()))
    else:
        f.step(data, idx, agent, grad_out=grad)
    torch.cuda.synchronize()
    losses = f.losses(0, 1)[0].double().cpu().numpy()
    slices = f._slices(agent.act, agent.cri)
    out = None
    if want_out:
        B = idx.numel()
        lay = (C.c_int64 * 34)()
        L.check(L.lib().pime_ppo_tc_layout(C.byref(f.cfg), C.c_int32(B), lay))
        last = _decode(f.work_tc, lay[2 + 2 * 4], (B + 127) // 128, agent.net_dim)[:B].double()
        w = agent.act.net[-1]
        out = last @ w.weight.detach().double().reshape(-1) + w.bias.detach().double().reshape(())
        del last
    f.work_tc = f.work = f._args = None
    return grad, losses, slices, out


def _check(agent, data, idx, tc, label, excluded):
    """Kernel step vs fp64 on rows idx: the four objectives and every gradient tensor.  Returns the worst gradient error.
    Tensor-core step at a_std_log = TC_SMALL_STD: see TC_SMALL_STD_BOUND."""
    small_std = tc and float(agent.act.a_std_log.detach().reshape(-1)[0]) == TC_SMALL_STD
    grad, losses, slices, out = _kernel_grad(agent, data, idx, tc, want_out=small_std)
    sub = [t[idx].double() for t in data]
    if small_std:
        act64, cri64 = _nets64(agent)
        with torch.no_grad():
            out64 = torch.cat([act64.a_avg(sub[0][lo:lo + CHUNK]).reshape(-1) for lo in range(0, idx.numel(), CHUNK)])
        shift = out - out64
        std = float(np.exp(np.float32(TC_SMALL_STD)))
        print(f"{label}: actor output err {float(shift.abs().max()):.2e}, ratio err (to first order) "
              f"{float((shift * (out64 - sub[1]).abs()).abs().max()) / std ** 2:.2e}")
        own = _compare(agent, act64, cri64, sub, grad, losses, slices, TC_BOUND, label + " at the kernel's actor output", excluded, shift)
        plain = _compare(agent, *_nets64(agent), sub, grad, losses, slices, TC_SMALL_STD_BOUND, label, excluded, None, objectives=False)
        return max(own, plain)
    return _compare(agent, *_nets64(agent), sub, grad, losses, slices, TC_BOUND if tc else SIMT_BOUND, label, excluded, None)


def _compare(agent, act64, cri64, sub, grad, losses, slices, bound, label, excluded, shift, objectives=True):
    ref, absum, cs = _reference(act64, cri64, *sub, agent.ratio_clip, agent.lambda_entropy, shift)
    names = ["united", "actor", "critic", "entropy"]
    obj_err = {n: abs(losses[i] - ref[i]) / max(abs(ref[i]), absum[n]) for i, n in enumerate(names)}
    # flat-layout order (actor tensors, critic tensors, a_std_log) -> the fp64 copies
    p64 = {id(p): ("act." + n, q) for (n, p), q in zip(agent.act.named_parameters(), act64.parameters())}
    p64.update({id(p): ("cri." + n, q) for (n, p), q in zip(agent.cri.named_parameters(), cri64.parameters())})
    sums = {"act.net.%d.bias" % (2 if agent.act.kind == "modular" else 6): "act_out_bias", "cri.net.6.bias": "cri_out_bias",
            "act.a_std_log": "a_std_log"}
    worst, worst_name, errs = 0.0, "", {}
    for t, o in slices:
        name, q = p64[id(t)]
        got = grad[o:o + t.numel()].double().view_as(t)
        want = q.grad.view_as(t)
        scale = absum[sums[name]] if name in sums else float(want.abs().max())
        err = float((got - want).abs().max())
        rel = err / scale if scale > 0 else (0.0 if err == 0 else float("inf"))
        errs[name] = rel
        if rel > worst:
            worst, worst_name = rel, name
    print(f"{label}: excluded {excluded} rows, std(r_sum) {cs:.3g}, worst gradient err {worst:.2e} ({worst_name}), "
          f"objectives {max(obj_err.values()):.2e}")
    bad = {k: f"{v:.2e}" for k, v in errs.items() if not v <= bound}
    assert not bad, f"{label}: gradient errors over {bound:g}: {bad}"
    bad = {k: f"{v:.2e}" for k, v in obj_err.items() if not v <= OBJ_BOUND}
    assert not (objectives and bad), f"{label}: objective errors over {OBJ_BOUND:g}: {bad}"
    return worst


def _case(kind, S, H, B, tc, seed=0, L=None, **gen):
    agent = _agent(kind, S, H)
    data = _data(agent, S, L or max(4 * B, 8192), seed=seed, **gen)
    idx, excluded = _draw(agent, data, B, agent.ratio_clip, seed + 1)
    tag = ", ".join(f"{k}={v:g}" for k, v in gen.items())
    return _check(agent, data, idx, tc, f"{'tc' if tc else 'simt'} {kind}-{H} S={S} B={B}" + (f" ({tag})" if tag else ""), excluded)


# ------------------------------------------------------------------------------------------------ the reference itself
@pytest.mark.parametrize("kind", ["modular", "plain"])
def test_reference_helper_equals_agent_objectives_in_fp64(kind):
    """The chunked helper is AgentPPO.ppo_objectives: same objectives and gradients in float64 (<= 1e-12)."""
    import types

    import pime_b200.rl as R
    agent = _agent(kind, 4, 32)
    data = _data(agent, 4, 300, mean=-500.0, std=200.0)
    x, action, r_sum, logprob, adv = (t.double() for t in data)
    act1, cri1 = _nets64(agent)
    ns = types.SimpleNamespace(act=act1, cri=cri1, criterion=torch.nn.SmoothL1Loss(), ratio_clip=agent.ratio_clip,
                               lambda_entropy=agent.lambda_entropy)
    oa, oc, ou, oe = R.AgentPPO.ppo_objectives(ns, x, action.unsqueeze(1), r_sum, logprob, adv)
    ou.backward()
    act2, cri2 = _nets64(agent)
    global CHUNK
    keep, CHUNK = CHUNK, 64                   # five chunks, the last one ragged
    try:
        ref, _, _ = _reference(act2, cri2, x, action, r_sum, logprob, adv, agent.ratio_clip, agent.lambda_entropy)
    finally:
        CHUNK = keep
    np.testing.assert_allclose(ref, [ou.item(), oa.item(), oc.item(), oe.item()], rtol=1e-12, atol=0)
    for p1, p2 in zip(list(act1.parameters()) + list(cri1.parameters()), list(act2.parameters()) + list(cri2.parameters())):
        if p1.grad is None:
            assert p2.grad is None
            continue
        assert float((p1.grad - p2.grad).abs().max()) <= 1e-12 * max(float(p1.grad.abs().max()), 1e-300)


# ------------------------------------------------------------------------------------------------ SIMT step
def _cover(Hs, Bs):
    """Every (H, B) pair once, S and the actor kind varying with both H and B (S = 30 on the plain actor only), plus the
    largest B with the modular actor and S = 4 at every H."""
    out = []
    for hi, H in enumerate(Hs):
        for bi, B in enumerate(Bs):
            S = (3, 4, 30)[(bi + hi) % 3]
            out.append(("plain" if S == 30 or (bi // 2 + hi) % 2 else "modular", S, H, B))
        if ("modular", 4, H, Bs[-1]) not in out:
            out.append(("modular", 4, H, Bs[-1]))
    return out


_SIMT = _cover((32, 64, 128, 256), (2, 3, 129, 257, 1000, 4096))


@pytest.mark.parametrize("kind,S,H,B", _SIMT)
def test_simt_step_matches_fp64(kind, S, H, B):
    _case(kind, S, H, B, tc=False, seed=B + H)


# ------------------------------------------------------------------------------------------------ tensor-core step
@pytest.mark.parametrize("kind,S,H,B", _cover((128, 256), (2048, 2049, 33000, 1 << 17)))
def test_tc_step_matches_fp64(kind, S, H, B):
    _case(kind, S, H, B, tc=True, seed=B + H)


def test_tc_step_matches_fp64_at_the_largest_batch():
    """2^20 rows, the entry's limit (8192 row tiles; the weight-gradient row split grows to 256)."""
    _case("modular", 4, 256, 1 << 20, tc=True, seed=7, L=1 << 18)
    torch.cuda.empty_cache()


# ------------------------------------------------------------------------------------------------ return-scale sweep
_SWEEP = [(s, m, a) for s in (1e-2, 1.0, 1e2, 1e3, 1e4) for m in (0.0, -10.0) for a in (-3.0, -0.5, 1.0)]


@pytest.mark.parametrize("std,mean_over_std,a_std_log", _SWEEP)
def test_simt_step_across_return_scales(std, mean_over_std, a_std_log):
    _case("modular", 4, 128, 1000, tc=False, seed=11, std=std, mean=mean_over_std * std, a_std_log=a_std_log)


@pytest.mark.parametrize("std,mean_over_std,a_std_log", _SWEEP)
def test_tc_step_across_return_scales(std, mean_over_std, a_std_log):
    _case("modular", 4, 256, 8192, tc=True, seed=12, std=std, mean=mean_over_std * std, a_std_log=a_std_log)


# ------------------------------------------------------------------------------------------------ a real replay
def test_tc_step_on_a_water_tank_replay():
    """configs[4]'s data in miniature: 2^12 water tanks x 200 steps from a fresh Modular-256 agent with its prior
    (reward_scale 1, gamma 0.99), values and GAE by update_net's own pre-pass, then one 2^17-row step against fp64."""
    import pime_b200.gym_api as G
    import pime_b200.rl as R
    n = 1 << 12
    env = R.PreprocessEnv(G.make("NonLinearWaterTankChangingParamUniformGoalIntegrator-SquareDistance-v2", num_envs=n, dtype=torch.float32))
    torch.manual_seed(0)
    agent = R.AgentResidualIntegratorModularPPO()
    agent.init(256, env.state_dim, env.action_dim, env.n_integrator)
    agent.init_residual({"init_K": env.K.reshape(-1, 1)})
    buf = R.ReplayBuffer(n * env.max_step, env.state_dim, 1, True, False, True, num_envs=n)
    agent.explore_env(env, buf, n * env.max_step, 1.0, 0.99)
    buf.update_now_len_before_sample()
    with torch.no_grad():                                  # update_net's pre-pass (rl.py, agent.py:611-633)
        buf_reward, buf_mask, buf_action, buf_noise, buf_state = buf.sample_all()
        buf_value = agent._values(buf_state)
        buf_logprob = -(buf_noise.pow(2) * 0.5 + agent.act.a_std_log + agent.act.sqrt_2pi_log).sum(1)
        buf_r_sum, buf_adv = agent.compute_reward(buf.now_len, buf_reward, buf_mask, buf_value, buf.num_envs)
        agent.act.net[-1].weight.normal_(0, 0.01)          # the prior alone leaves the actor's hidden gradients at zero
    data = (buf_state.contiguous(),) + tuple(t.reshape(-1).contiguous() for t in (buf_action, buf_r_sum, buf_logprob, buf_adv))
    del buf, buf_reward, buf_mask, buf_noise, buf_value
    print(f"water-tank replay: {data[0].shape[0]} rows, std(r_sum) {float(data[2].std()):.4g}, |mean(r_sum)| {abs(float(data[2].mean())):.4g}, "
          f"max |r_sum| {float(data[2].abs().max()):.4g}")
    idx, excluded = _draw(agent, data, 1 << 17, agent.ratio_clip, 5)
    _check(agent, data, idx, True, "tc modular-256 water-tank replay B=131072", excluded)


# ------------------------------------------------------------------------------------------------ Adam
@pytest.mark.parametrize("scale", [1.0, 0.5])
def test_apply_grad_matches_fp64_adam(scale):
    """pime_ppo_apply_grad on a fixed gradient sequence vs torch's fused-Adam formula in fp64, one step at a time from the
    kernel's own fp32 state, at steps 1, 2 and 1000 (bias corrections): |d theta - d theta_64| <= 1e-5 lr + ulp(theta).
    The bias corrections are those adam_prepare writes at the start of the step (here by a 2-row pime_ppo_step)."""
    import pime_b200._lib as L
    import pime_b200.rl as R
    agent = _agent("modular", 4, 64)
    data = _data(agent, 4, 64)
    f = R.FusedLearner(agent.act, agent.cri, 4, 64, agent.device)
    f.load(agent.act, agent.cri)
    sink = torch.zeros_like(f.theta)
    idx = torch.arange(2, device="cuda")
    grp = agent.optimizer.param_groups[0]
    lr, b1, b2, eps = (float(np.float32(v)) for v in (grp["lr"], grp["betas"][0], grp["betas"][1], grp["eps"]))
    live = torch.zeros_like(f.theta, dtype=torch.bool)
    for t, o in f._slices(agent.act, agent.cri):
        live[o:o + t.numel()] = True
    n = f.theta.numel()
    g = torch.Generator(device="cuda").manual_seed(3)
    mags = 10.0 ** (torch.rand(n, device="cuda", generator=g) * 6 - 4)        # 1e-4 .. 1e2 per element
    for step in range(1, 1001):
        grad = (torch.randn(n, device="cuda", generator=g) * mags).float()
        grad[::97] = 0.0
        f.step(data, idx, agent, grad_out=sink)                              # adam_prepare for this step, then close it
        check = step in (1, 2, 1000)
        if check:
            th0, m0, v0 = f.theta.double(), f.m.double(), f.v.double()
        args = f._bind(data, idx, agent, False, sink)
        L.check(L.lib().pime_ppo_apply_grad(args, L.ptr(grad), ctypes_float(scale), L.stream_ptr()))
        if not check:
            continue
        torch.cuda.synchronize()
        gd = grad.double() * scale
        m = m0 + (gd - m0) * (1 - b1)                                          # lerp(exp_avg, grad, 1 - beta1)
        v = v0 * b2 + (1 - b2) * gd * gd
        bc1, bc2 = 1 - b1 ** step, 1 - b2 ** step
        th = th0 - (lr / bc1) * m / (v.sqrt() / np.sqrt(bc2) + eps)
        got = f.theta.double()
        ulp = torch.from_numpy(np.spacing(np.abs(f.theta.cpu().numpy()))).double().cuda()
        err = ((got - th0) - (th - th0)).abs()
        worst = float((err / (1e-5 * lr + ulp))[live].max())
        # moments: a few fp32 roundings of terms of size |m0| + |g| and v
        mv = max(float(((f.m.double() - m).abs() / (2.4e-7 * (m0.abs() + gd.abs()) + 1e-30))[live].max()),
                 float(((f.v.double() - v).abs() / (2.4e-7 * v + 1e-30))[live].max()))
        print(f"adam scale={scale} step {step}: worst |d theta err| / (1e-5 lr + ulp) {worst:.3f}, moments {mv:.3f} of their bound")
        assert worst <= 1.0 and mv <= 1.0, step
        assert torch.equal(f.theta[~live], th0[~live].float())
    assert int(f.state[0]) == 1000


def ctypes_float(x):
    import ctypes
    return ctypes.c_float(x)


# ------------------------------------------------------------------------------------------------ GAE scan
@pytest.mark.parametrize("lam", [0.0, 0.95, 0.99])
@pytest.mark.parametrize("strided", [False, True])
def test_gae_scan_matches_fp64_recursion(lam, strided):
    """pime_gae_scan (through V.gae_scan) vs the reverse recursion of agent.py:685-708 in fp64: 200 steps x 2^16 + 3 env
    columns, rewards in [-100, 0], episode ends inside the columns; also on the stride-4 view into a [T n, 4] replay
    buffer.  Bound: 2e-5 of the column's largest |r_sum|."""
    import pime_b200.vec as V
    T, n = 200, (1 << 16) + 3
    g = torch.Generator(device="cuda").manual_seed(int(lam * 100) + strided)
    reward = -torch.rand(T, n, device="cuda", generator=g) * 100
    mask = torch.full((T, n), 0.99, device="cuda")
    mask[torch.rand(T, n, device="cuda", generator=g) < 0.02] = 0.0
    mask[-1] = 0.0
    value = -torch.rand(T, n, device="cuda", generator=g) * 5000
    if strided:
        buf = torch.randn(T * n, 4, device="cuda", generator=g)
        buf[:, 0], buf[:, 1] = reward.reshape(-1), mask.reshape(-1)
        r_sum, adv = V.gae_scan(buf[:, 0], buf[:, 1], value, lam, stride=4)
    else:
        r_sum, adv = V.gae_scan(reward, mask, value, lam)
    torch.cuda.synchronize()
    r, m, v = reward.double(), mask.double(), value.double()
    lam32 = float(np.float32(lam))
    rs, ad = torch.empty_like(r), torch.empty_like(r)
    pre_r = torch.zeros(n, dtype=torch.float64, device="cuda")
    pre_a = torch.zeros_like(pre_r)
    for s in range(T - 1, -1, -1):
        rs[s] = r[s] + m[s] * pre_r
        pre_r = rs[s]
        ad[s] = r[s] + m[s] * (pre_a - v[s])
        pre_a = v[s] + ad[s] * lam32
    col = rs.abs().amax(0)
    e_r = float(((r_sum.double() - rs).abs() / col).max())
    e_a = float(((adv.double() - ad).abs() / col).max())
    print(f"gae lam={lam} stride={4 if strided else 1}: r_sum err {e_r:.2e}, adv err {e_a:.2e} (of the column's max |r_sum|)")
    assert e_r <= 2e-5 and e_a <= 2e-5
