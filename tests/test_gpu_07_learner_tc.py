"""GPU parity of the tensor-core PPO minibatch step (csrc/learner_tc.cu, pime_ppo_grad_tc): AgentPPO.update_net's minibatch
(elegantrl/agent.py:635-658) for large batches as tcgen05 GEMMs over 128-row tiles with fp16 hi + lo operands.

The chain of evidence: tests/golden/ppo.npz (the reference's own gradients and post-Adam parameters, H = 32) pins
``rl.AgentPPO.ppo_objectives`` + torch autograd (tests/test_rl_host.py) and the small-batch kernels (test_gpu_04_agent.py);
the tensor-core step needs H in {128, 256}, so it is pinned HERE against that same autograd objective on identical inputs:
every forward activation (<= 2e-6), every gradient tensor (<= 2e-4 of the tensor's largest entry), the objectives (1e-5),
and consecutive Adam steps."""
import ctypes as C

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


def _agents(kind, S, H, n=2):
    import pime_b200.rl as R
    torch.manual_seed(5)
    out = []
    for _ in range(n):
        agent = R.AgentResidualIntegratorModularPPO() if kind == "modular" else R.AgentResidualPPO()
        agent.init(H, S, 1, 1) if kind == "modular" else agent.init(H, S, 1)
        with torch.no_grad():
            agent.act.net[-1].weight.normal_(0, 0.1)
            agent.act.net[-1].bias.normal_(0, 0.1)
        out.append(agent)
    for b in out[1:]:
        b.act.load_state_dict(out[0].act.state_dict())
        b.cri.load_state_dict(out[0].cri.state_dict())
    return out


def _data(agent, S, L=40000, seed=0):
    g = torch.Generator(device="cuda").manual_seed(seed)
    state = torch.rand(L, S, device="cuda", generator=g) * 10
    state[:, -1] = torch.rand(L, device="cuda", generator=g) * 50 - 25           # an integrated error
    action = torch.randn(L, device="cuda", generator=g)
    r_sum = torch.randn(L, device="cuda", generator=g) * 30 - 50
    logprob = -(torch.randn(L, device="cuda", generator=g).pow(2) * 0.5 + agent.act.a_std_log.item() + agent.act.sqrt_2pi_log)
    adv = torch.randn(L, device="cuda", generator=g)
    return state, action, r_sum, logprob, adv


def _decode(work, off, row_tiles, units):
    """T-format (tiles of 128 rows x 64 units, hi block + lo block, each [8 unit groups][128 rows][8 fp16]) -> [rows, units] fp32."""
    nb = row_tiles * (units // 64) * 2 * 16384
    raw = work[off:off + nb].view(torch.float16).view(row_tiles, units // 64, 2, 8, 128, 8).float()
    x = raw[:, :, 0] + raw[:, :, 1]                       # [row tile, chunk, unit group, row, e]
    return x.permute(0, 3, 1, 2, 4).reshape(row_tiles * 128, units)


def _grad_tc(f, data, idx, agent):
    """pime_ppo_grad_tc only (no Adam): the flat gradient and the scratch buffer."""
    import pime_b200._lib as L
    args = f._bind(data, idx, agent, True)
    f.work_tc.zero_()
    grad = torch.zeros_like(f.theta)
    L.check(L.lib().pime_ppo_grad_tc(args, L.ptr(f.work_tc), L.ptr(grad), L.stream_ptr()))
    torch.cuda.synchronize()
    return grad, f.work_tc


@pytest.mark.parametrize("kind,S,H,B", [("modular", 4, 256, 300), ("modular", 3, 128, 1000), ("plain", 30, 256, 257), ("plain", 4, 128, 128),
                                        ("modular", 4, 256, 4096), ("modular", 4, 256, 20001), ("plain", 12, 128, 33000)])
def test_tc_gradient_and_every_stage_match_autograd(kind, S, H, B):
    # 20 001 / 33 000 rows: 157 / 258 row tiles -> every weight-gradient CTA walks over 5-9 row tiles (its hi / lo buffer pipeline
    # wraps around several times) and the last row tile is ragged
    import pime_b200._lib as L
    import pime_b200.rl as R
    torch.backends.cuda.matmul.allow_tf32 = False
    (agent,) = _agents(kind, S, H, 1)
    data = _data(agent, S)
    state, action, r_sum, logprob, adv = data
    idx = torch.randint(state.shape[0], size=(B,), device="cuda")
    f = R.FusedLearner(agent.act, agent.cri, S, H, agent.device)
    f.load(agent.act, agent.cri)
    grad, work = _grad_tc(f, data, idx, agent)
    lay = (C.c_int64 * 34)()
    L.check(L.lib().pime_ppo_tc_layout(C.byref(f.cfg), C.c_int32(B), lay))
    rt = (B + 127) // 128
    x = state[idx]
    # ---- forward stages
    X = _decode(work, lay[0], rt, 64)[:B]
    # hi + lo keeps 22 significant bits (fewer below 6e-5, where the lo part is an fp16 subnormal: absolute error <= 3e-8)
    assert torch.allclose(X[:, :S], x, rtol=5e-7, atol=1e-7) and float(X[:, 63].min()) == 1.0 and float(X[:, S:63].abs().max()) == 0.0
    A = {i: _decode(work, lay[2 + 2 * i], rt, H)[:B] for i in range(8) if lay[3 + 2 * i]}
    with torch.no_grad():
        act, cri = agent.act, agent.cri
        if kind == "modular":
            So = act.other_dim
            a0 = torch.tanh(act.other_net[0](x[:, :So])); a1 = torch.tanh(act.integrator_net[0](x[:, So:]))
            cat = torch.cat([torch.tanh(act.other_net[2](a0)), torch.tanh(act.integrator_net[2](a1))], 1)
            n0 = torch.tanh(act.net[0](cat))
            want = {0: a0, 1: a1, 2: cat, 4: n0}
        else:
            a0 = torch.tanh(act.net[0](x)); a2 = torch.tanh(act.net[2](a0)); a4 = torch.tanh(act.net[4](a2))
            want = {0: a0, 2: a2, 4: a4}
        c0 = torch.relu(cri.net[0](x)); c1 = torch.relu(cri.net[2](c0)); c2 = torch.relu(cri.net[4](c1))
        want.update({5: c0, 6: c1, 7: c2})
    for i, wnt in want.items():
        err = float((A[i] - wnt).abs().max())
        print(f"{kind}-{H} B={B} activation {i}: max err {err:.2e}")
        assert err <= 2e-5 * max(1.0, float(wnt.abs().max())), i
    # ---- objectives and gradients
    oa, oc, ou, oe = agent.ppo_objectives(x, action[idx].unsqueeze(1), r_sum[idx], logprob[idx], adv[idx])
    agent.optimizer.zero_grad(set_to_none=False)
    ou.backward()
    np.testing.assert_allclose(f.losses(0, 1)[0].cpu().numpy(), [ou.item(), oa.item(), oc.item(), oe.item()], rtol=2e-5, atol=1e-6)
    worst = 0.0
    for t, o in f._slices(agent.act, agent.cri):
        got, wnt = grad[o:o + t.numel()].view_as(t), t.grad
        scale = float(wnt.abs().max()) + 1e-12
        err = float((got - wnt).abs().max()) / scale
        worst = max(worst, err)
        print(f"   grad {tuple(t.shape)} rel err {err:.2e} (scale {scale:.2e})")
    print(f"{kind}-{H} B={B}: worst gradient error relative to the tensor's largest entry {worst:.2e}")
    assert worst <= 2e-4
    assert int(f.state[0]) == 0        # the gradient entry does not close the step


@pytest.mark.parametrize("kind,S,H,B", [("modular", 4, 256, 2048), ("plain", 30, 128, 4173)])
def test_tc_steps_track_the_autograd_path(kind, S, H, B):
    """Five consecutive minibatch steps from the same start and the same index draws: pime_ppo_grad_tc + pime_ppo_apply_grad
    and torch autograd + torch.optim.Adam stay together."""
    import pime_b200.rl as R
    torch.backends.cuda.matmul.allow_tf32 = False
    a, b = _agents(kind, S, H, 2)
    data = _data(a, S, seed=1)
    state, action, r_sum, logprob, adv = data
    f = R.FusedLearner(a.act, a.cri, S, H, a.device)
    f.load(a.act, a.cri)
    for it in range(5):
        idx = torch.randint(state.shape[0], size=(B,), device="cuda")
        f.step_tc(data, idx, a)
        oa, oc, ou, oe = b.ppo_objectives(state[idx], action[idx].unsqueeze(1), r_sum[idx], logprob[idx], adv[idx])
        b.optimizer.zero_grad(set_to_none=False)
        ou.backward()
        b.optimizer.step()
        np.testing.assert_allclose(f.losses(it, 1)[0].cpu().numpy(), [ou.item(), oa.item(), oc.item(), oe.item()], rtol=1e-4, atol=1e-5)
    assert int(f.state[0]) == 5
    f.store(a.act, a.cri)
    lr = b.optimizer.param_groups[0]["lr"]
    for (n1, p1), (n2, p2) in zip(list(a.act.named_parameters()) + list(a.cri.named_parameters()),
                                  list(b.act.named_parameters()) + list(b.cri.named_parameters())):
        if n1 == "priorK":
            continue
        d = (p1 - p2).detach().abs()
        assert float(d.max()) <= 0.6 * lr and float(d.mean()) <= 0.02 * lr, n1


def test_update_net_takes_the_tensor_core_path_for_large_batches():
    import pime_b200.gym_api as G
    import pime_b200.rl as R
    n = 256
    env = R.PreprocessEnv(G.make("NonLinearWaterTankChangingParamUniformGoalIntegrator-SquareDistance-v2", num_envs=n, dtype=torch.float32))
    torch.manual_seed(0)
    agent = R.AgentResidualIntegratorModularPPO()
    agent.learning_rate = 3e-4
    agent.init(128, env.state_dim, env.action_dim, env.n_integrator)
    agent.init_residual({"init_K": env.K.reshape(-1, 1)})
    buf = R.ReplayBuffer(n * env.max_step, env.state_dim, 1, True, False, True, num_envs=n)
    steps = agent.explore_env(env, buf, n * env.max_step, 1.0, 0.99)
    agent.update_net(buf, steps, 4096, 1)
    c0 = R.logger.values["train/critic_loss"]
    assert "pime_ppo_grad_tc" in agent.learner_path
    for _ in range(3):
        agent.update_net(buf, steps, 4096, 2)
    assert R.logger.values["train/critic_loss"] < c0
    assert all(torch.isfinite(v).all() for v in agent.act.state_dict().values())
    agent.update_net(buf, steps, 256, 1)                    # small batches keep the rows / weight-gradient kernels
    assert "pime_ppo_step" in agent.learner_path
