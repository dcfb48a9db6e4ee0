"""GPU tests of the agent / buffer / trainer surface (pime_b200.rl): the reference's PPO pre-pass (values, GAE, plain
advantage -- fixtures from the reference's own compute_reward_* in tests/golden/ppo.npz) through the CUDA kernels,
the fused explore_env into the HBM-resident replay, the learner step and the train loop."""
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

WT = "NonLinearWaterTankChangingParamUniformGoalIntegrator-SquareDistance-v2"
PH = "PH1DChangingParamUniformGoalIntegrator-SqaureDistance-v35"


def _agent_from_fixture(g, tag):
    import pime_b200.rl as R
    if tag == "modular":
        agent = R.AgentResidualIntegratorModularPPO()
        agent.init(32, 4, 1, 1)
    else:
        agent = R.AgentResidualPPO()
        agent.init(32, 3, 1)
    agent.lambda_gae_adv, agent.ratio_clip, agent.lambda_entropy = 0.95, 0.25, 0.02
    agent.init_residual({"init_K": g[f"{tag}.K"]})
    agent.act.load_state_dict({k[len(tag) + 6:]: torch.as_tensor(g[k]) for k in g.files if k.startswith(f"{tag}.act0.")})
    agent.cri.load_state_dict({k[len(tag) + 6:]: torch.as_tensor(g[k]) for k in g.files if k.startswith(f"{tag}.cri0.")})
    return agent


@pytest.mark.parametrize("tag", ["modular", "plain"])
def test_value_gae_and_plain_advantage_match_reference(golden, tag):
    """agent.py:617-624,666-708: critic values by the tcgen05 kernel (fp16 operands: 2e-3), reward-to-go / GAE by the
    scan kernel on the reference's own values (fp32: 1e-5 relative), both buffer orders (reference order = one env,
    and the time-major order of a 6-env batch)."""
    g = golden("ppo")
    agent = _agent_from_fixture(g, tag)
    state = torch.as_tensor(g[f"{tag}.state"]).cuda()
    val = agent._values(state).cpu().numpy()
    assert np.abs(val - g[f"{tag}.value"]).max() <= 2e-3 * max(1.0, np.abs(g[f"{tag}.value"]).max())
    reward, mask = torch.as_tensor(g[f"{tag}.reward"]).cuda(), torch.as_tensor(g[f"{tag}.mask"]).cuda()
    value = torch.as_tensor(g[f"{tag}.value"]).cuda()
    L, n, T = reward.numel(), 6, 20
    for num_envs in (1, n):
        if num_envs == 1:
            r_, m_, v_ = reward, mask, value
            back = lambda x: x
        else:   # episode-major [n, T] -> time-major [T, n] and back
            tm = lambda x: x.view(n, T).t().contiguous().view(-1)
            r_, m_, v_ = tm(reward), tm(mask), tm(value)
            back = lambda x: x.view(T, n).t().contiguous().view(-1)
        r_sum, adv = agent.compute_reward_gae(L, r_, m_, v_, num_envs)
        np.testing.assert_allclose(back(r_sum).cpu().numpy(), g[f"{tag}.r_sum"], rtol=1e-5, atol=1e-4)
        np.testing.assert_allclose(back(adv).cpu().numpy(), g[f"{tag}.adv_gae"], rtol=1e-4, atol=2e-5)
        r_sum2, adv2 = agent.compute_reward_adv(L, r_, m_, v_, num_envs)
        np.testing.assert_allclose(back(r_sum2).cpu().numpy(), g[f"{tag}.r_sum"], rtol=1e-5, atol=1e-4)
        np.testing.assert_allclose(back(adv2).cpu().numpy(), g[f"{tag}.adv_plain"], rtol=1e-4, atol=2e-5)


def _make(env_id, num_envs, dtype=torch.float32, **kw):
    import pime_b200.gym_api as G
    import pime_b200.rl as R
    return R.PreprocessEnv(G.make(env_id, num_envs=num_envs, dtype=dtype, **kw))


@pytest.mark.parametrize("env_id,algo,H", [(WT, "residualintegratormodularppo", 64), (PH, "residualintegratormodularppo", 32),
                                           ("NonLinearWaterTankChangingParamUniformGoalStacking4-SquareDistance-v2", "residualppo", 32),
                                           (WT, "ppo", 32)])
def test_explore_env_fills_the_hbm_replay(env_id, algo, H):
    """agent_residual.py:52-69 as ONE launch per episode batch: row layout, masks, reward scale, a_raw = net(s) + eps*std."""
    import pime_b200.rl as R
    n = 300
    env = _make(env_id, n)
    agent = R.MODELS[algo]()
    if "modular" in algo:
        agent.init(H, env.state_dim, env.action_dim, env.n_integrator)
    else:
        agent.init(H, env.state_dim, env.action_dim)
    if "residual" in algo:
        agent.init_residual({"init_K": env.K.reshape(-1, 1)})
    with torch.no_grad():
        agent.act.net[-1].weight.normal_(0, 0.1)
    T = env.max_step
    buf = R.ReplayBuffer(2 * n * T, env.state_dim, 1, True, False, True, num_envs=n)
    steps = agent.explore_env(env, buf, n * T + 1, reward_scale=0.5, gamma=0.97)
    assert steps == 2 * n * T                                   # whole episode batches until >= target_step
    buf.update_now_len_before_sample()
    assert buf.now_len == steps
    r, m, a, nz, s = buf.sample_all()
    m_ = m.view(2 * T, n).cpu().numpy()
    assert np.all(m_[T - 1] == 0) and np.all(m_[2 * T - 1] == 0) and np.all(np.delete(m_, [T - 1, 2 * T - 1], 0) == np.float32(0.97))
    assert torch.isfinite(s).all() and torch.isfinite(r).all() and float(r.max()) <= 0.0
    with torch.no_grad():
        a_net = agent.act.a_avg(s)
    std = float(agent.act.a_std_log.detach().exp())
    assert float((a - nz * std - a_net).abs().max()) <= 2e-3    # fp16 tensor-core operands vs torch fp32
    assert 0.9 < float(nz.std()) < 1.1 and abs(float(nz.mean())) < 0.02
    if "Stacking" not in env_id:
        s0 = s.view(2 * T, n, -1)[0]
        assert float(s0[:, -1].abs().max()) == 0.0 if "Integrator" in env_id else True   # I = 0 after reset


def test_update_net_learns_and_checkpoint_roundtrip(tmp_path):
    import pime_b200.rl as R
    torch.manual_seed(0)
    n = 256
    env = _make(WT, n)
    agent = R.AgentResidualIntegratorModularPPO()
    agent.learning_rate = 3e-4
    agent.init(64, env.state_dim, env.action_dim, env.n_integrator)
    agent.init_residual({"init_K": env.K.reshape(-1, 1)})
    buf = R.ReplayBuffer(n * env.max_step, env.state_dim, 1, True, False, True, num_envs=n)
    before = {k: v.clone() for k, v in agent.act.state_dict().items()}
    steps = agent.explore_env(env, buf, n * env.max_step, 1.0, 0.99)
    obj_a, obj_c = agent.update_net(buf, steps, batch_size=4096, repeat_times=2)
    assert np.isfinite(obj_a) and np.isfinite(obj_c)
    after = agent.act.state_dict()
    assert any(not torch.equal(before[k], after[k]) for k in before if k != "priorK")
    assert torch.equal(before["priorK"], after["priorK"])                 # fix_K: the prior never trains
    # the mean critic loss goes down when the same buffer is fitted again
    c0 = R.logger.values["train/critic_loss"]
    agent.update_net(buf, steps, batch_size=4096, repeat_times=8)
    assert R.logger.values["train/critic_loss"] < c0
    agent.save_load_model(str(tmp_path), if_save=True)
    assert os.path.exists(tmp_path / "actor.pth") and os.path.exists(tmp_path / "critic.pth")
    sd = torch.load(tmp_path / "actor.pth")
    assert sorted(sd) == sorted(["a_std_log", "priorK"] + [f"{m}.{i}.{p}" for m in ("other_net", "integrator_net", "net")
                                                          for i in (0, 2) for p in ("weight", "bias")])
    other = R.AgentResidualIntegratorModularPPO()
    other.init(64, env.state_dim, env.action_dim, env.n_integrator)
    other.save_load_model(str(tmp_path), if_save=False)
    assert all(torch.equal(other.act.state_dict()[k].cpu(), after[k].cpu()) for k in after)


def test_zero_initialised_agent_evaluates_like_the_prior():
    """init_actor_zero (agent_residual.py:45-50): the deterministic episodes of a fresh agent are the prior controller's."""
    import pime_b200.rl as R
    import pime_b200.vec as V
    n = 512
    env = _make(WT, n, dtype=torch.float64, noise_scale=0.0)
    agent = R.AgentResidualIntegratorModularPPO()
    agent.init(32, 4, 1, 1)
    agent.init_residual({"init_K": env.K.reshape(-1, 1)})
    env.seed(3)
    eps = R.evaluate_batched(env, agent)
    ref = V.WaterTankVec(n, dtype=torch.float64, noise_scale=0.0, seed=3)
    ref.reset()
    ref.rollout(200, -env.K, actor=None, deterministic=True)
    got = np.array([e[0] for e in eps])
    np.testing.assert_allclose(got, ref.ep_return.cpu().numpy(), rtol=1e-9, atol=1e-9)
    r_avg, r_std, s_avg, _ = R.Evaluator.get_r_avg_std_s_avg_std(eps)
    assert s_avg == 200 and r_avg < 0 and r_std > 0


def test_train_and_evaluate_smoke(tmp_path):
    """run.py:99-225 end to end on the pH plant (config 2 shrunk): explore -> update -> evaluate, files on disk."""
    import pime_b200.rl as R
    env = _make(PH, 128)
    args = R.Arguments(if_on_policy=True)
    args.agent = R.MODELS["residualintegratormodularppo"]()
    args.agent.lambda_gae_adv, args.agent.ratio_clip = 0.99, 0.2
    args.env, args.env_eval = env, _make(PH, 64)
    args.cwd = str(tmp_path / "run")
    args.net_dim, args.batch_size, args.repeat_times, args.target_step = 32, 1024, 2, 128 * 50
    args.max_memo = args.target_step
    args.break_step, args.eval_gap, args.eval_times1, args.eval_times2 = 3 * 128 * 50, 1, 64, 64
    args.gamma, args.fix_K = 0.98, True
    args.residual_kwargs = {"init_K": env.K.reshape(-1, 1)}
    args.Modular_kwargs = {"integrator_dim": env.n_integrator}
    env.target_return = 1e9
    args.env_eval.target_return = 1e9
    R.configure_logger(0, str(tmp_path / "tb"), "smoke")
    agent, buf = R.train_and_evaluate(args)
    assert buf.now_len == 128 * 50 and os.path.exists(os.path.join(args.cwd, "actor.pth"))
    hist = [h for h in R.logger.history if "training/total_step" in h]
    assert [h["training/total_step"] for h in hist][-1] == 3 * 128 * 50
    assert all(np.isfinite(h.get("train/critic_loss", 0.0)) for h in hist)


def test_train_and_evaluate_with_the_default_eval_env(tmp_path):
    """Arguments.env_eval = None is the default (run.py:127: `env_eval = deepcopy(env)`): the PreprocessEnv wrapper and the
    device env underneath must survive copy.deepcopy (advisor finding, round 1) and the copy must be independent."""
    import pime_b200.rl as R
    env = _make(WT, 16)
    args = R.Arguments(if_on_policy=True)
    args.agent = R.MODELS["residualppo"]()
    args.env, args.env_eval = env, None
    args.cwd = str(tmp_path / "run")
    args.net_dim, args.batch_size, args.repeat_times, args.target_step = 32, 256, 1, 16 * 200
    args.max_memo = args.target_step
    args.break_step, args.eval_gap, args.eval_times1, args.eval_times2 = 2 * 16 * 200, 1, 8, 8
    args.residual_kwargs = {"init_K": env.K.reshape(-1, 1)}
    env.target_return = 1e9
    R.configure_logger(0, None)
    test_dirs = []
    args.test_render = lambda agent, d: test_dirs.append(d)              # called at step 0 and every test_render_times steps
    args.test_render_times = 16 * 200
    agent, buf = R.train_and_evaluate(args)
    assert buf.now_len == 16 * 200 and os.path.exists(os.path.join(args.cwd, "actor.pth"))
    assert [os.path.basename(d) for d in test_dirs] == ["step_0", "step_3200", "step_6400"]
    import copy
    twin = copy.deepcopy(env)
    assert twin.env.vec is not env.env.vec and torch.equal(twin.env.vec.h1, env.env.vec.h1)
    twin.env.vec.h1.add_(1.0)
    assert not torch.equal(twin.env.vec.h1, env.env.vec.h1)


def test_cuda_graph_minibatch_step_is_transparent():
    """The recorded minibatch step (index draw + gather + forward + backward + Adam) leaves the training state untouched
    while it is being recorded, and trains like the eager step (same kernels, different index draws)."""
    import pime_b200.rl as R
    n = 64
    env = _make(WT, n)
    finals = {}
    for mode in (False, True):
        torch.manual_seed(0)
        env.seed(0)
        agent = R.AgentResidualIntegratorModularPPO()
        agent.learning_rate = 3e-4
        agent.use_cuda_graph = mode
        agent.use_fused_learner = False          # this test is about the autograd step (the path of frozen / distributed runs)
        agent.init(32, env.state_dim, env.action_dim, env.n_integrator)
        agent.init_residual({"init_K": env.K.reshape(-1, 1)})
        buf = R.ReplayBuffer(n * env.max_step, env.state_dim, 1, True, False, True, num_envs=n)
        steps = agent.explore_env(env, buf, n * env.max_step, 1.0, 0.99)
        if mode:   # recording alone must be a no-op on parameters and Adam state
            before = [p.detach().clone() for p in agent.act.parameters()] + [p.detach().clone() for p in agent.cri.parameters()]
            buf.update_now_len_before_sample()
            r, m, a, nz, s = buf.sample_all()
            data = (s, a, torch.zeros_like(r), torch.zeros_like(r), torch.zeros_like(r))

            def mb(src, out):
                idx = torch.randint(steps, size=(256,), device=agent.device)
                oa, oc, ou, oe = agent.ppo_objectives(*(t[idx] for t in src))
                agent.optimizer.zero_grad(set_to_none=False)
                ou.backward()
                agent.optimizer.step()
                out[:4].copy_(torch.stack([ou.detach(), oa.detach(), oc.detach(), oe.detach()]))
            agent._graphed_step(mb, data, steps, 256)
            after = list(agent.act.parameters()) + list(agent.cri.parameters())
            assert all(torch.equal(x, y) for x, y in zip(before, after))
            assert all(float(v.abs().max()) == 0.0 for st in agent.optimizer.state.values() for v in st.values() if torch.is_tensor(v))
            agent._graph = None
        agent.update_net(buf, steps, batch_size=256, repeat_times=1)
        c0 = R.logger.values["train/critic_loss"]
        agent.update_net(buf, steps, batch_size=256, repeat_times=4)
        finals[mode] = (c0, R.logger.values["train/critic_loss"])
        assert finals[mode][1] < finals[mode][0]
        assert (agent._graph is not None) == mode
    assert abs(finals[True][1] - finals[False][1]) <= 0.25 * abs(finals[False][1])


def test_examples_train_py_runs_the_reference_command_line(tmp_path):
    """examples/train.py = the reference's train.py command line on this stack (run_ph_changing.sh shrunk)."""
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    cmd = [sys.executable, os.path.join(root, "examples", "train.py"), "--fix_K", "--algo", "ResidualIntegratorModularPPO",
           "--env", PH, "--net_dim", "32", "--target_step", "1600", "--batch_size", "256", "--repeat_times", "2",
           "--lambda_gae_adv", "0.99", "--ratio_clip", "0.2", "--gamma", "0.98", "--break_step", "4800", "--eval_times1", "8",
           "--eval_times2", "8", "--eval_gap", "1", "--num_envs", "32", "--out", str(tmp_path)]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert res.returncode == 0, res.stdout[-2000:] + res.stderr[-2000:]
    found = [os.path.join(dp, f) for dp, _, fn in os.walk(tmp_path) for f in fn]
    assert any(f.endswith("final_model/actor.pth") for f in found) and any(f.endswith("final_model/staircase.npz") for f in found)
    z = np.load([f for f in found if f.endswith("final_model/staircase.npz")][0])
    assert z["agent.ys"].shape == (250, 32) and z["linear.ys"].shape == (250, 32) and np.isfinite(z["agent.totals"]).all()


# ------------------------------------------------------------------------------------------------ fused learner kernels
def _fused_setup(g, tag, lr=3e-4):
    import pime_b200.rl as R
    agent = _agent_from_fixture(g, tag)
    agent.optimizer = torch.optim.Adam([{"params": agent.act.parameters(), "lr": lr}, {"params": agent.cri.parameters(), "lr": lr}])
    dev = agent.device
    data = tuple(torch.as_tensor(g[f"{tag}.{k}"]).to(dev).reshape(len(g[f"{tag}.state"]), -1) for k in
                 ("state", "action", "r_sum", "logprob", "adv_gae"))
    data = (data[0].contiguous(),) + tuple(t.reshape(-1).contiguous() for t in data[1:])
    f = R.FusedLearner(agent.act, agent.cri, agent.state_dim, agent.net_dim, dev)
    f.load(agent.act, agent.cri)
    return agent, f, data, torch.as_tensor(g[f"{tag}.idx"]).to(dev)


def _split(f, agent, flat):
    names = [k for k in f._keys[0]] + ["cri." + k for k in f._keys[1]] + ["a_std_log"]
    return {name: flat[o:o + t.numel()].view_as(t).cpu().numpy() for name, (t, o) in zip(names, f._slices(agent.act, agent.cri))}


@pytest.mark.parametrize("tag", ["modular", "plain"])
def test_fused_ppo_kernels_match_the_reference_gradients_and_adam_step(golden, tag):
    """pime_ppo_step against the reference's own numbers (oracle/gen_golden.py:gen_ppo: agent.py:635-658 run on a fixed
    index set): the four objectives (2e-5), every gradient (1e-4 relative) and the parameters after ONE Adam step (1e-5)."""
    g = golden("ppo")
    agent, f, data, idx = _fused_setup(g, tag)
    grad = torch.zeros_like(f.theta)
    f.step(data, idx, agent, grad_out=grad)                                    # gradient-only mode: theta untouched
    np.testing.assert_allclose(f.losses(0, 1)[0, [1, 2, 0, 3]].cpu().numpy(), g[f"{tag}.losses"], rtol=2e-5, atol=1e-6)
    for name, got in _split(f, agent, grad).items():
        np.testing.assert_allclose(got, g[f"{tag}.grad.{name}"], rtol=1e-4, atol=1e-6, err_msg=name)
    before = f.theta.clone()
    f.store(agent.act, agent.cri)
    assert all(torch.equal(a, b) for a, b in zip(_split_t(f, agent, before), f._tensors(agent.act, agent.cri)))

    agent, f, data, idx = _fused_setup(g, tag)                                 # fresh moments: the fused Adam step
    f.step(data, idx, agent)
    f.store(agent.act, agent.cri)
    assert int(f.state[0]) == 1 and float(f.state.view(torch.float32)[2]) == 0.0 and int(f.state[1]) == 0
    for k in g.files:
        for net, pre in ((agent.act, f"{tag}.act1."), (agent.cri, f"{tag}.cri1.")):
            if k.startswith(pre):
                np.testing.assert_allclose(net.state_dict()[k[len(pre):]].cpu().numpy(), g[k], rtol=1e-5, atol=1e-6, err_msg=k)
    # the transposed copy the forward pass reads follows the update
    w = agent.cri.net[2].weight
    o = dict((id(t), o) for t, o in f._slices(agent.act, agent.cri))[id(w)]
    assert torch.equal(f.theta_t[o:o + w.numel()].view(w.shape[1], w.shape[0]).t(), w)


def _split_t(f, agent, flat):
    return [flat[o:o + t.numel()].view_as(t) for t, o in f._slices(agent.act, agent.cri)]


@pytest.mark.parametrize("kind,S,H,B", [("modular", 4, 256, 256), ("modular", 3, 128, 128), ("plain", 30, 256, 200),
                                        ("plain", 3, 64, 37), ("modular", 4, 32, 1000)])
def test_fused_ppo_steps_track_the_autograd_path(kind, S, H, B):
    """Five consecutive minibatch steps (ragged batches included) from the same start and the same index draws: the fused
    kernels and the torch autograd + torch.optim.Adam step stay together (fp32, different summation order only)."""
    import pime_b200.rl as R
    torch.manual_seed(3)
    agents = []
    for _ in range(2):
        agent = R.AgentResidualIntegratorModularPPO() if kind == "modular" else R.AgentResidualPPO()
        agent.init(H, S, 1, 1) if kind == "modular" else agent.init(H, S, 1)
        with torch.no_grad():
            agent.act.net[-1].weight.normal_(0, 0.1)
        agents.append(agent)
    a, b = agents
    b.act.load_state_dict(a.act.state_dict())
    b.cri.load_state_dict(a.cri.state_dict())
    L = 3000
    state = torch.randn(L, S, device="cuda") * 2
    action = torch.randn(L, device="cuda")
    r_sum = torch.randn(L, device="cuda") * 3 - 1
    logprob = -(torch.randn(L, device="cuda").pow(2) * 0.5 + a.act.a_std_log.item() + a.act.sqrt_2pi_log)
    adv = torch.randn(L, device="cuda")
    data = (state, action, r_sum, logprob, adv)
    f = R.FusedLearner(a.act, a.cri, S, H, a.device)
    f.load(a.act, a.cri)
    params = [p for grp in b.optimizer.param_groups for p in grp["params"]]
    for it in range(5):
        idx = torch.randint(L, size=(B,), device="cuda")
        f.step(data, idx, a)
        oa, oc, ou, oe = b.ppo_objectives(state[idx], action[idx].unsqueeze(1), r_sum[idx], logprob[idx], adv[idx])
        b.optimizer.zero_grad(set_to_none=False)
        ou.backward()
        b.optimizer.step()
        np.testing.assert_allclose(f.losses(it, 1)[0].cpu().numpy(), [ou.item(), oa.item(), oc.item(), oe.item()], rtol=1e-4, atol=1e-5)
    f.store(a.act, a.cri)
    lr = b.optimizer.param_groups[0]["lr"]
    for (n1, p1), (n2, p2) in zip(list(a.act.named_parameters()) + list(a.cri.named_parameters()),
                                  list(b.act.named_parameters()) + list(b.cri.named_parameters())):
        if n1 == "priorK":
            continue
        # an Adam step moves a weight by at most ~lr whatever the gradient's size: five steps agree to a fraction of one
        d = (p1 - p2).detach().abs()
        assert float(d.max()) <= 0.6 * lr and float(d.mean()) <= 0.02 * lr, n1


def test_update_net_takes_the_fused_path_and_matches_autograd():
    import pime_b200.rl as R
    res = []
    n = 256
    for fused in (True, False):
        torch.manual_seed(11)
        env = _make(WT, n)
        agent = R.AgentResidualIntegratorModularPPO()
        agent.init(64, env.state_dim, env.action_dim, env.n_integrator)
        agent.use_fused_learner = fused
        agent.use_cuda_graph = False             # eager autograd step: the same index draws as the fused loop
        agent.init_residual({"init_K": env.K.reshape(-1, 1)})
        buf = R.ReplayBuffer(n * env.max_step, env.state_dim, 1, True, False, True, num_envs=n)
        steps = agent.explore_env(env, buf, n * env.max_step, 1.0, 0.99)
        torch.manual_seed(12)
        out = agent.update_net(buf, steps, batch_size=256, repeat_times=1)     # 200 minibatch steps
        assert (agent._fused is not None) == fused
        res.append((out, {k: v.clone() for k, v in agent.act.state_dict().items()}, {k: v.clone() for k, v in agent.cri.state_dict().items()},
                    dict(R.logger.values)))
    (o1, a1, c1, l1), (o2, a2, c2, l2) = res
    for k in ("train/united_loss", "train/actor_loss", "train/critic_loss", "train/entropy_losses"):
        np.testing.assert_allclose(l1[k], l2[k], rtol=5e-3, atol=1e-4, err_msg=k)
    lr = 1e-4
    for d1, d2 in ((a1, a2), (c1, c2)):
        for k in d1:
            assert float((d1[k] - d2[k]).abs().max()) <= 3 * lr, k        # 200 Adam steps of 1e-4 each: the same trajectory
            assert float((d1[k] - d2[k]).abs().mean()) <= 0.05 * lr, k


def test_fused_learner_eligibility_and_plain_ppo_arm():
    """The frozen_* variants keep the autograd step (their frozen tensors must not move); the plain PPO baseline arm
    (agent.py:591-609, no prior) trains through the fused kernels like the residual agents."""
    import pime_b200.rl as R
    n = 64
    env = _make(WT, n)
    frozen = R.AgentResidualIntegratorModularPPO()
    frozen.init(32, env.state_dim, env.action_dim, env.n_integrator)
    frozen.init_residual({"init_K": env.K.reshape(-1, 1)})
    frozen.frozen_integrator()
    assert not R.FusedLearner.eligible(frozen, 256)
    buf = R.ReplayBuffer(n * env.max_step, env.state_dim, 1, True, False, True, num_envs=n)
    steps = frozen.explore_env(env, buf, n * env.max_step, 1.0, 0.99)
    held = {k: v.clone() for k, v in frozen.act.state_dict().items() if k.startswith("integrator_net")}
    frozen.update_net(buf, steps, 256, 1)
    assert frozen._fused is None and all(torch.equal(frozen.act.state_dict()[k], v) for k, v in held.items())

    plain = R.AgentPPO()
    plain.init(32, env.state_dim, env.action_dim)
    assert R.FusedLearner.eligible(plain, 256) and not R.FusedLearner.eligible(plain, 1 << 20)
    buf2 = R.ReplayBuffer(n * env.max_step, env.state_dim, 1, True, False, True, num_envs=n)
    steps = plain.explore_env(env, buf2, n * env.max_step, 1.0, 0.99)
    before = {k: v.clone() for k, v in plain.act.state_dict().items()}
    plain.update_net(buf2, steps, 256, 1)
    plain.update_net(buf2, steps, 256, 4)
    assert plain._fused is not None and plain._fused.steps == 5 * (steps // 256)
    assert all(np.isfinite(R.logger.values[k]) for k in ("train/critic_loss", "train/actor_loss", "train/entropy_losses"))
    assert all(torch.isfinite(v).all() for v in plain.act.state_dict().values())
    assert any(not torch.equal(before[k], v) for k, v in plain.act.state_dict().items())
    plain.init_actor_zero()                         # a new optimizer: the fused moments start over as well
    assert plain._fused is None


def test_split_adam_path_equals_the_fused_step(golden):
    """Data-parallel form of the step on one rank: pime_ppo_step(grad_out) -> all-reduce (world 1: identity) ->
    pime_ppo_apply_grad leaves the parameters, transposes and moments of the fused step: same arithmetic per element,
    bit-identical everywhere except the two Linear(H -> 1) output layers, whose gradients the rows kernel accumulates with
    floating-point atomics (order varies from launch to launch, last-bit differences)."""
    import torch.distributed as dist
    g = golden("ppo")
    if not dist.is_initialized():
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("MASTER_PORT", "29511")
        dist.init_process_group("nccl", rank=0, world_size=1, device_id=torch.device("cuda", 0))
    try:
        a1, f1, data, idx = _fused_setup(g, "modular")
        a2, f2, _, _ = _fused_setup(g, "modular")
        for s in range(3):
            ix = (idx + 7 * s) % data[0].shape[0]
            f1.step(data, ix, a1)
            f2.step(data, ix, a2, f2.dist_grad())
            for name in ("theta", "theta_t", "m", "v"):
                x, y = getattr(f1, name), getattr(f2, name)
                assert torch.allclose(x, y, rtol=2e-4, atol=1e-10), (s, name)
                if s == 0:   # first step: only the atomically-summed output layers may differ at all (later steps inherit it)
                    assert int((x != y).sum()) <= 2 * (a1.net_dim + 1), (s, name)
        assert int(f2.state[0]) == 3 and torch.allclose(f1.loss_ring, f2.loss_ring, rtol=1e-5, atol=1e-7)
    finally:
        dist.destroy_process_group()


_DIST_WORKER = r"""
import os, sys, numpy as np, torch, torch.distributed as dist
sys.path.insert(0, sys.argv[1])
rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
torch.cuda.set_device(rank)
dist.init_process_group("nccl", device_id=torch.device("cuda", rank))
import pime_b200.gym_api as G, pime_b200.rl as R
n, H = 64, 128
env = R.PreprocessEnv(G.make("NonLinearWaterTankChangingParamUniformGoalIntegrator-SquareDistance-v2", num_envs=n, dtype=torch.float32))
env.env.vec.env_offset = rank * n
torch.manual_seed(0)
agent = R.AgentResidualIntegratorModularPPO(); agent.learning_rate = 3e-4
agent.init(H, env.state_dim, 1, 1); agent.init_residual({"init_K": env.K.reshape(-1, 1)})
buf = R.ReplayBuffer(n * 200, env.state_dim, 1, True, False, True, num_envs=n)
torch.manual_seed(100 + rank)                      # different minibatch draws per rank
for it in range(2):
    steps = agent.explore_env(env, buf, n * 200, 1.0, 0.99)
    agent.update_net(buf, steps, 256, 2)
assert "all-reduce" in agent.learner_path, agent.learner_path
# large minibatches: the tensor-core step, one flat all-reduce of its gradient before the Adam kernel
agent.update_net(buf, steps, 2048, 2)
assert "pime_ppo_grad_tc" in agent.learner_path and "all-reduce" in agent.learner_path, agent.learner_path
flat = torch.cat([p.detach().reshape(-1) for p in list(agent.act.parameters()) + list(agent.cri.parameters())])
ref = flat.clone(); dist.broadcast(ref, 0)
assert torch.equal(flat, ref), "replicas diverged"
assert torch.isfinite(flat).all()
# single-learner mode: the NCCL all-gather of the sharded replay gives every rank the rows of all 2 n envs, time-major,
# rank 0's env range first -- and one rollout over the whole range on one GPU writes exactly those rows
full = buf.gather()
assert full.num_envs == 2 * n and full.now_len == 2 * buf.now_len
mine = full.buf_state.view(-1, 2 * n, env.state_dim)[:, rank * n:(rank + 1) * n]
assert torch.equal(mine.reshape(-1, env.state_dim), buf.buf_state[:buf.now_len])
chk = full.buf_other.double().sum(); ref2 = chk.clone(); dist.broadcast(ref2, 0)
assert torch.equal(chk, ref2)
if rank == 0: print("DIST_OK", agent.learner_path)
dist.destroy_process_group()
"""


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs (NCCL refuses two ranks on one device)")
def test_two_rank_nccl_training_keeps_replicas_identical(tmp_path):
    """configs[4] in miniature on 2 GPUs: sharded envs, different minibatches per rank, gradients averaged by NCCL inside the
    hand-written learner step -> bit-identical replicas after two iterations."""
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    script = tmp_path / "w.py"
    script.write_text(_DIST_WORKER)
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
           "--master-port", "29533", str(script), root]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert res.returncode == 0 and "DIST_OK" in res.stdout, res.stdout[-2000:] + res.stderr[-3000:]
