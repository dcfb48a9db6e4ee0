"""GPU parity: the tcgen05 actor / critic forward vs the reference modules' outputs (fixtures) and the fp32 oracle.

Operands are fp16 (activations in [-1,1], weights), accumulation fp32 in TMEM, tanh = MUFU tanh.approx.
Stated tolerance on a_avg = net(obs): 4e-3 absolute + 1e-2 relative."""
import numpy as np
import pytest
import torch

from gpu_util import dev, host

pytestmark = pytest.mark.gpu
ATOL, RTOL = 4e-3, 1e-2


@pytest.fixture(scope="module")
def V():
    import pime_b200.vec as vec
    return vec


def _fixture_sd(g, tag):
    return {k[len(tag) + 4:]: g[k] for k in g.files if k.startswith(tag + ".sd.")}


@pytest.mark.parametrize("kind,H,S,D", [("modular", 32, 4, 1), ("modular", 64, 3, 1), ("plain", 32, 30, 0), ("plain", 32, 3, 0)])
def test_actor_forward_matches_reference_module_outputs(V, golden, kind, H, S, D):
    g = golden("actor")
    tag = f"{kind}.H{H}.S{S}"
    pack = V.ActorPack(kind, S, H, D).update(_fixture_sd(g, tag))
    got = host(pack.forward(dev(g[tag + ".obs"])))
    err = np.max(np.abs(got - g[tag + ".a_avg"]))
    print(f"{tag}: max |a_avg err| = {err:.3e}")
    np.testing.assert_allclose(got, g[tag + ".a_avg"], atol=ATOL, rtol=RTOL)


def _torch_default_params(kind, H, S, D, seed, scale_last=0.1):
    """Random parameters at torch.nn.Linear's default init scale, in state_dict form."""
    rng = np.random.default_rng(seed)

    def lin(o, i):
        b = 1.0 / np.sqrt(i)
        return rng.uniform(-b, b, (o, i)).astype(np.float32), rng.uniform(-b, b, o).astype(np.float32)
    sd = {}
    if kind == "modular":
        shapes = [("other_net.0", H, S - D), ("other_net.2", H // 2, H), ("integrator_net.0", H, D), ("integrator_net.2", H // 2, H),
                  ("net.0", H, H), ("net.2", 1, H)]
    else:
        shapes = [("net.0", H, S), ("net.2", H, H), ("net.4", H, H), ("net.6", 1, H)]
    for name, o, i in shapes:
        w, b = lin(o, i)
        sd[name + ".weight"], sd[name + ".bias"] = w, b
    last = shapes[-1][0]
    sd[last + ".weight"] = (rng.normal(0, scale_last, (1, H))).astype(np.float32)
    return sd


def _torch_forward(kind, sd, obs, relu=False):
    act = torch.relu if relu else torch.tanh
    t = {k: torch.as_tensor(v).cuda() for k, v in sd.items()}
    x = obs
    if kind == "modular":
        So = t["other_net.0.weight"].shape[1]
        a = act(x[:, :So] @ t["other_net.0.weight"].T + t["other_net.0.bias"])
        a = act(a @ t["other_net.2.weight"].T + t["other_net.2.bias"])
        b = act(x[:, So:] @ t["integrator_net.0.weight"].T + t["integrator_net.0.bias"])
        b = act(b @ t["integrator_net.2.weight"].T + t["integrator_net.2.bias"])
        c = act(torch.cat([a, b], 1) @ t["net.0.weight"].T + t["net.0.bias"])
        return (c @ t["net.2.weight"].T + t["net.2.bias"])[:, 0]
    h = act(x @ t["net.0.weight"].T + t["net.0.bias"])
    h = act(h @ t["net.2.weight"].T + t["net.2.bias"])
    h = act(h @ t["net.4.weight"].T + t["net.4.bias"])
    return (h @ t["net.6.weight"].T + t["net.6.bias"])[:, 0]


# Bounds on (a_avg - fp32 torch) per compiled (kind, H): (RMS over n = 1 / 129 / 40000, |mean| at n = 40000), set from one
# B200 run (NVIDIA B200, 1000 W power limit) at 1.5x the measured value; the comment gives the measured max |error|, RMS and
# |mean|.  The fused rollout's network is pinned bit for bit to this kernel (test_gpu_08), so these bounds carry over to it.
FWD_BOUNDS = {  # (kind)(H)-S(S): (rms, |mean|),  measured: max      rms      |mean|
    "modular256-S4": (2.6e-04, 1.4e-04),  # 5.8e-04  1.7e-04  9.2e-05
    "modular128-S3": (3.6e-04, 4.2e-05),  # 4.5e-04  2.4e-04  2.8e-05
    "modular64-S3": (1.1e-04, 2.7e-05),  # 2.5e-04  7.2e-05  1.8e-05
    "modular32-S4": (6.8e-05, 8.3e-06),  # 1.4e-04  4.5e-05  5.5e-06
    "plain256-S30": (2.5e-04, 4.9e-05),  # 6.9e-04  1.6e-04  3.2e-05
    "plain256-S3": (3.0e-04, 1.4e-04),  # 4.8e-04  2.0e-04  8.7e-05
    "plain128-S12": (1.9e-04, 7.4e-05),  # 5.1e-04  1.2e-04  4.9e-05
    "plain64-S4": (1.8e-04, 6.2e-05), # 2.1e-04  1.1e-04  4.1e-05
    "plain32-S3": (1.6e-04, 6.1e-05), # 1.7e-04  1.0e-04  4.0e-05
    "critic256-S4": (4.6e-04, 3.8e-05),  # 1.5e-03  3.0e-04  2.5e-05
    "critic128-S3": (2.3e-04, 1.6e-05),  # 8.2e-04  1.5e-04  1.0e-05
    "critic64-S4": (7.6e-04, 1.1e-04),  # 9.4e-04  5.0e-04  6.9e-05
    "critic32-S3": (2.2e-04, 1.4e-06),  # 3.8e-04  1.4e-04  9.0e-07
}


@pytest.mark.parametrize("kind,H,S,D", [("modular", 256, 4, 1), ("modular", 128, 3, 1), ("modular", 64, 3, 1), ("modular", 32, 4, 1),
                                        ("plain", 256, 30, 0), ("plain", 256, 3, 0), ("plain", 128, 12, 0), ("plain", 64, 4, 0),
                                        ("plain", 32, 3, 0), ("critic", 256, 4, 0), ("critic", 128, 3, 0), ("critic", 64, 4, 0),
                                        ("critic", 32, 3, 0)])
@pytest.mark.parametrize("n", [1, 129, 40000])
def test_forward_vs_torch_fp32(V, oracle, kind, H, S, D, n):
    torch.backends.cuda.matmul.allow_tf32 = False
    sd = _torch_default_params("modular" if kind == "modular" else "plain", H, S, D, seed=H + S)
    pack = V.ActorPack(kind, S, H, D).update(sd)
    rng = np.random.default_rng(n)
    obs = rng.uniform(-2, 12, (n, S)).astype(np.float32)
    if kind == "modular":
        obs[:, -1] = rng.uniform(-25, 25, n)
    got = host(pack.forward(dev(obs)))
    want = host(_torch_forward("modular" if kind == "modular" else "plain", sd, dev(obs), relu=(kind == "critic")))
    e = got.astype(np.float64) - want
    err, rms, mean = np.max(np.abs(e)), np.sqrt(np.mean(e ** 2)), np.mean(e)
    print(f"{kind} H{H} S{S} n{n}: max err {err:.3e}, rms {rms:.3e}, mean {mean:+.3e}, |want| max {np.abs(want).max():.3f}")
    np.testing.assert_allclose(got, want, atol=ATOL, rtol=RTOL)
    rb, mb = FWD_BOUNDS[f"{kind}{H}-S{S}"]
    assert rms <= rb, (rms, rb)
    if n == 40000:
        assert abs(mean) <= mb, (mean, mb)
    if kind != "critic" and n <= 129:  # the C oracle restates the same fp32 forward
        acfg = oracle.ActorCfg(kind=1 if kind == "modular" else 0, state_dim=S, mid_dim=H, integrator_dim=D)
        o = oracle.actor_forward(acfg, oracle.pack_actor_params(sd, acfg.kind), obs)
        np.testing.assert_allclose(o, want, atol=2e-5, rtol=1e-4)


def test_zero_last_layer_gives_exact_zero(V):
    """init_actor_zero (agent_residual.py:45-50): the residual starts at exactly 0."""
    sd = _torch_default_params("modular", 256, 4, 1, seed=1)
    sd["net.2.weight"][:] = 0.0
    sd["net.2.bias"][:] = 0.0
    pack = V.ActorPack("modular", 4, 256, 1).update(sd)
    obs = torch.rand((1000, 4), device="cuda") * 10
    assert float(pack.forward(obs).abs().max()) == 0.0


def test_repack_after_update_changes_output(V):
    sd = _torch_default_params("plain", 64, 3, 0, seed=2)
    pack = V.ActorPack("plain", 3, 64).update(sd)
    obs = torch.rand((256, 3), device="cuda")
    a = pack.forward(obs).clone()
    sd["net.6.bias"] = sd["net.6.bias"] + 1.0
    b = pack.update(sd).forward(obs)
    np.testing.assert_allclose(host(b - a), 1.0, atol=1e-6)


@pytest.mark.parametrize("kind,H,S,D", [("modular", 256, 4, 1), ("modular", 128, 3, 1), ("plain", 256, 30, 0), ("critic", 256, 4, 0),
                                        ("plain", 32, 3, 0)])
@pytest.mark.parametrize("n", [1, 33, 40000])
def test_fidelity_mode_forward_vs_torch_fp32(V, kind, H, S, D, n):
    """PIME_PRECISION_FP32 (fp32 CUDA cores, tanhf): |a_avg - fp32 torch| <= 2e-5 at every size, ragged row counts included."""
    sd = _torch_default_params(kind, H, S, D, seed=H + S)
    obs = torch.as_tensor(np.random.default_rng(n).uniform(-1, 10, (n, S)).astype(np.float32)).cuda()
    if S == 4:
        obs[:, 3] = torch.as_tensor(np.random.default_rng(1).uniform(-25, 25, n).astype(np.float32)).cuda()
    pack = V.ActorPack(kind, S, H, D, precision="fp32").update(sd)
    got = host(pack.forward(obs))
    prev = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = False
    try:
        want = host(_torch_forward(kind, sd, obs, relu=kind == "critic"))
    finally:
        torch.backends.cuda.matmul.allow_tf32 = prev
    err = np.abs(got - want.reshape(-1)).max()
    print(f"fidelity {kind}-{H} S={S} n={n}: max |a_avg err| = {err:.2e}")
    assert err <= 2e-5
    # the same packed image still serves the throughput engine
    tc = host(pack.set_precision("tc").forward(obs))
    np.testing.assert_allclose(tc, want.reshape(-1), atol=ATOL, rtol=RTOL)
