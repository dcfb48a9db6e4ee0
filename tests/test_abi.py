"""CPU tests: the C-ABI library loads without a GPU, exports every symbol include/pime_b200.h declares, its structs
match the ctypes mirrors, and compute entry points fail loudly (no CPU fallback)."""
import ctypes as C
import os
import re
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "pime_b200.h")


@pytest.fixture(scope="module")
def L():
    sys.path.insert(0, ROOT)
    import pime_b200.build as build
    build.build()
    import pime_b200._lib as lib
    return lib


def _header_functions():
    src = open(HEADER).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(pime_[a-z0-9_]+)\s*\(", src)))


def test_every_declared_symbol_is_exported(L):
    declared = _header_functions()
    assert len(declared) >= 30
    out = subprocess.run(["nm", "-D", "--defined-only", L.LIB_PATH], capture_output=True, text=True, check=True).stdout
    exported = set(re.findall(r" T (pime_[a-z0-9_]+)", out))
    missing = [s for s in declared if s not in exported]
    assert not missing, f"declared in the header but not exported: {missing}"
    assert sorted(L.SYMBOLS) == declared, "pime_b200._lib.SYMBOLS must list exactly the header's functions"
    lib = L.lib()
    assert lib.pime_abi_version() == 5


def test_struct_layouts_match_header(L, tmp_path):
    prog = tmp_path / "sizes.c"
    prog.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "pime_b200.h"\nint main(){'
                    'printf("%zu %zu %zu %zu %zu %zu\\n", sizeof(pime_wt_config), sizeof(pime_wt_state), sizeof(pime_ph_config),'
                    'sizeof(pime_ph_state), sizeof(pime_actor_config), sizeof(pime_rollout_args));'
                    'printf("%zu %zu %zu %zu\\n", offsetof(pime_wt_config, z1), offsetof(pime_wt_config, r_hi),'
                    'offsetof(pime_rollout_args, eps), offsetof(pime_rollout_args, status));return 0;}')
    exe = tmp_path / "sizes"
    subprocess.run(["gcc", "-I", os.path.join(ROOT, "include"), str(prog), "-o", str(exe)], check=True)
    out = subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split()
    got = [int(v) for v in out]
    want = [C.sizeof(L.WtConfig), C.sizeof(L.WtState), C.sizeof(L.PhConfig), C.sizeof(L.PhState), C.sizeof(L.ActorConfig),
            C.sizeof(L.RolloutArgs), L.WtConfig.z1.offset, L.WtConfig.r_hi.offset, L.RolloutArgs.eps.offset,
            L.RolloutArgs.status.offset]
    assert got == want


def test_default_configs_are_the_registered_values(L):
    w = L.wt_config()
    assert (w.A1, w.A2, w.G, w.sample_t, w.n_discrete, w.max_step, w.P_max_action) == (1, 1, 980, 2.0, 20, 200, 10.0)
    assert (w.a1_lo, w.a1_hi, w.Kp_lo, w.Kp_hi) == (0.0015, 0.0024, 0.07, 0.17)
    assert w.reward_type == L.REWARD["square_distance"] and w.integral_max == 25.0 and w.noise_scale == 0.01
    p = L.ph_config()
    assert (p.max_episode_steps, p.table_len, p.act_high, p.sample_t) == (50, 100000, 1.5, 20.0)
    assert (p.qww_lo, p.qww_hi, p.qc_lo, p.qc_hi, p.x_hi, p.r_lo, p.r_hi) == (0.005, 0.015, 0.0015, 0.0025, 50.0, 3.0, 11.0)
    assert (p.kw, p.kchem, p.ka, p.MNaOH, p.MHA, p.MNH3) == (1e-14, 5.6e-10, 0.5e-5, 0.01, 0.005, 0.01)


@pytest.mark.parametrize("kind,S,H,D,count", [(1, 4, 256, 1, 133382 - 1 - 4), (1, 3, 128, 1, 33797 - 1 - 3),
                                              (0, 30, 256, 0, 30 * 256 + 256 + 2 * (256 * 256 + 256) + 257),
                                              (2, 4, 256, 0, 133121)])
def test_actor_parameter_counts(L, kind, S, H, D, count):
    """SURVEY 8a d4/d5/f1: parameter counts of the reference modules (minus a_std_log and priorK, which are scalars
    of the rollout call, not of the packed image)."""
    cfg = L.ActorConfig(kind=kind, state_dim=S, mid_dim=H, integrator_dim=D)
    assert L.lib().pime_actor_param_count(C.byref(cfg)) == count
    assert L.lib().pime_actor_pack_bytes(C.byref(cfg)) > 2 * (count - 3 * H - S * H)
    bad = L.ActorConfig(kind=kind, state_dim=S, mid_dim=100, integrator_dim=D)
    assert L.lib().pime_actor_param_count(C.byref(bad)) == -1


def test_compute_entry_points_fail_loudly_without_gpu(L):
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    lib = L.lib()
    assert lib.pime_device_info(None, None, None) == L.ENODEV
    cfg = L.wt_config()
    buf = (C.c_float * 8)()
    ibuf = (C.c_int32 * 8)()
    st = L.WtState(**{k: C.cast(buf, C.c_void_p) for k in ("h1", "h2", "r", "I", "a1", "a2", "Kp", "ep_return")},
                   t=C.cast(ibuf, C.c_void_p), episode=C.cast(ibuf, C.c_void_p))
    rc = lib.pime_wt_step_f32(C.byref(cfg), C.c_int64(8), C.byref(st), buf, None, None, C.c_uint64(0), C.c_uint64(0),
                              C.c_uint32(0), None, buf, C.cast(ibuf, C.c_void_p), None)
    assert rc == L.ENODEV
    assert b"no CPU fallback" in lib.pime_last_error()
    with pytest.raises(L.PimeError):
        L.check(rc)
    import pime_b200.vec as V
    with pytest.raises(L.PimeError):
        V.WaterTankVec(4)
    # argument validation happens before the device check
    rc = lib.pime_wt_step_f32(C.byref(cfg), C.c_int64(8), C.byref(st), None, None, None, C.c_uint64(0), C.c_uint64(0),
                              C.c_uint32(0), None, buf, C.cast(ibuf, C.c_void_p), None)
    assert rc == L.EINVAL
    with pytest.raises(ValueError):
        L.check(rc)


def test_rollout_entries_reject_out_of_range_configs(L):
    """The device and host-buffer rollout entries check the config as the step entries do: n_discrete < 1, reward_type
    outside 0..2 and table_len <= 1 (with which the fused pH kernel would read before the start of its table) are
    PIME_EINVAL, with or without a GPU.  n = 0 and a prior-only argument block: nothing would be launched if the check
    were missing, and every pointer is non-null, so only the config can be what the call rejects."""
    lib = L.lib()
    buf = (C.c_double * 8)()
    p = C.cast(buf, C.c_void_p)
    ep_host = (C.c_float * 8)()
    args = L.RolloutArgs(actor=None, priorK_host=(C.c_double * 4)(), T=1)
    wst = L.WtState(**{f: p for f, _ in L.WtState._fields_})
    pst = L.PhState(**{f: p for f, _ in L.PhState._fields_})
    n0 = C.c_int64(0)
    for bad in ({"n_discrete": 0}, {"reward_type": 3}):
        cfg = L.wt_config(**bad)
        for fn in (lib.pime_wt_rollout_f32, lib.pime_wt_rollout_f64):
            assert fn(C.byref(cfg), n0, C.byref(wst), C.byref(args), None) == L.EINVAL, bad
        rc = lib.pime_wt_rollout_host_f32(C.byref(cfg), n0, C.byref(wst), C.byref(wst), C.byref(args), ep_host, None)
        assert rc == L.EINVAL, bad
    cfg = L.ph_config(table_len=0)
    for fn in (lib.pime_ph_rollout_f32, lib.pime_ph_rollout_f64):
        assert fn(C.byref(cfg), p, n0, C.byref(pst), C.byref(args), None) == L.EINVAL
    rc = lib.pime_ph_rollout_host_f32(C.byref(cfg), p, n0, C.byref(pst), C.byref(pst), C.byref(args), ep_host, None)
    assert rc == L.EINVAL


def test_product_never_touches_the_oracle():
    """The oracle is test infrastructure: nothing under the package or include/ may import, link or mention it."""
    pkg = os.path.join(ROOT, "pime-robust-non-linear-set-point-control-with-reinforcement-learning_b200")
    offenders = []
    for base in (pkg, os.path.join(ROOT, "include"), os.path.join(ROOT, "pime_b200")):
        for dp, dn, fn in os.walk(base):
            if os.path.basename(dp) in ("build", "__pycache__"):
                continue
            for f in fn:
                if f.endswith((".py", ".cu", ".cuh", ".h", ".c", ".cpp")):
                    txt = open(os.path.join(dp, f), errors="replace").read()
                    if re.search(r"pime_oracle|ref_loader|oracle/|/root/reference", txt):
                        offenders.append(os.path.join(dp, f))
    assert not offenders, offenders
    out = subprocess.run(["ldd", os.path.join(pkg, "libpime_b200.so")], capture_output=True, text=True).stdout
    assert "oracle" not in out


def _device_program(kind, H, S):
    """Python restatement of Engine::mma_loop (csrc/tc_mlp.cuh): the (N, k16s, d_col) sequence the MMA warp issues per pass."""
    MAXB = 16384
    Hh, K16, Da, Db = H // 2, H // 16, 0, H

    def blk_k16(N, K):
        return min(MAXB // (N * 32), K)

    def layer(N, d, k_lo=0, k_hi=None, bias=True):
        out = [(N, 1, d)] if bias else []
        kpb = blk_k16(N, K16)
        k_hi = K16 if k_hi is None else k_hi
        out += [(N, kpb, d) for _ in range(k_lo, k_hi, kpb)]
        return out

    if kind == 1:   # modular
        return [(H, 1, Db)] + layer(Hh, Da) + layer(Hh, Da + Hh) + layer(H, Db)
    nin = 16 if S <= 16 else 32
    KP = ((((3 if S <= 10 else 2) * nin + 2) + 15) // 16) * 16
    kpb = blk_k16(H, 5)
    p0 = [(H, min(kpb, KP // 16 - k), Da) for k in range(0, KP // 16, kpb)]
    return p0 + layer(H, Db) + layer(H, Da)     # even pass: X = Da, Y = Db (the pack lists the even pass)


@pytest.mark.parametrize("kind,S", [(1, 4), (1, 3), (1, 2), (0, 3), (0, 4), (0, 12), (0, 16), (0, 17), (0, 30), (0, 31), (2, 3), (2, 4), (2, 30)])
@pytest.mark.parametrize("H", [32, 64, 128, 256])
def test_pack_block_list_matches_the_kernels_static_mma_program(L, kind, S, H):
    """The TMA producer streams the pack's block list; the MMA warp runs a static program.  They must agree block for
    block (a mismatch deadlocks the kernel): checked here without a GPU for every supported shape."""
    cfg = L.ActorConfig(kind=kind, state_dim=S, mid_dim=H, integrator_dim=1 if kind == 1 else 0)
    buf = (C.c_int32 * (4 * 64))()
    n = L.lib().pime_actor_block_list(C.byref(cfg), buf, 64)
    assert 0 < n <= 24
    got = [(buf[4 * b], buf[4 * b + 1], buf[4 * b + 2]) for b in range(n)]
    assert got == _device_program(kind, H, S)
    sizes = [buf[4 * b + 3] for b in range(n)]
    assert all(0 < s <= 16384 and s == N * k * 32 for s, (N, k, _) in zip(sizes, got))
    # header + fp16 blocks, then the fp32 copy of the parameters (the fidelity-mode forward reads it), both 16-byte aligned
    f32_off = (sum(sizes) + 4096 + 15) & ~15
    assert ((f32_off + 4 * L.lib().pime_actor_param_count(C.byref(cfg)) + 15) & ~15) == L.lib().pime_actor_pack_bytes(C.byref(cfg))
    assert all(d + N <= 2 * H for N, _, d in got)              # accumulators stay inside the two TMEM buffers


@pytest.mark.parametrize("kind,S,H", [(1, 4, 256), (1, 3, 128), (1, 2, 32), (0, 3, 64), (0, 30, 256), (0, 12, 128)])
def test_ppo_learner_layout_is_host_computable(L, kind, S, H):
    """pime_ppo_theta_layout / pime_ppo_work_floats need no GPU: theta = [actor | pad | critic | a_std_log] with the critic
    on a 16-byte boundary (its hidden-layer matrices are streamed with cp.async.bulk), scratch = per-row activations and
    pre-activation gradients of both nets + the gathered state row + the two output gradients."""
    cfg = L.ActorConfig(kind=kind, state_dim=S, mid_dim=H, integrator_dim=1 if kind == 1 else 0)
    cri = L.ActorConfig(kind=2, state_dim=S, mid_dim=H, integrator_dim=0)
    pa, pc = L.lib().pime_actor_param_count(C.byref(cfg)), L.lib().pime_actor_param_count(C.byref(cri))
    if kind == 1:
        assert pa == H * (S - 1) + H + (H // 2) * H + H // 2 + H + H + (H // 2) * H + H // 2 + H * H + H + H + 1
    else:
        assert pa == H * S + H + 2 * (H * H + H) + H + 1
    assert pc == H * S + H + 2 * (H * H + H) + H + 1
    lay = (C.c_int64 * 3)()
    assert L.lib().pime_ppo_theta_layout(C.byref(cfg), lay) == 0
    assert lay[0] % 4 == 0 and pa <= lay[0] < pa + 4 and lay[1] == lay[0] + pc and lay[2] == lay[1] + 1
    assert L.lib().pime_ppo_theta_count(C.byref(cfg)) == lay[2]
    la = (4 if kind == 1 else 3) * H + 3 * H
    for B in (2, 37, 256, 4096):
        assert L.lib().pime_ppo_work_floats(C.byref(cfg), C.c_int32(B)) == B * (32 + 2 * la + 2)
    bad = L.ActorConfig(kind=kind, state_dim=S, mid_dim=48, integrator_dim=1 if kind == 1 else 0)
    assert L.lib().pime_ppo_theta_count(C.byref(bad)) == -1


def test_host_entry_slice_plan(L):
    """csrc/host_pipe.cuh: the host-buffer entries cut large env ranges into <= 8 slices of whole waves (148 SMs x 256 envs);
    small ranges, stacking frames (single = 1) and n = 0 stay in one piece; a forced count slices by whole 256-env tiles."""
    lib = L.lib()
    wave = 148 * 256

    def plan(n, single=0):
        out = (C.c_int64 * 2)()
        assert lib.pime_host_slice_plan(C.c_int64(n), C.c_int32(single), out) == 0
        return int(out[0]), int(out[1])

    assert plan(0) == (1, 0) and plan(1000) == (1, 1000) and plan(8 * wave - 1) == (1, 8 * wave - 1)
    assert plan(8 * wave) == (2, 4 * wave)
    assert plan(1 << 20) == (6, 5 * wave)                       # BASELINE configs[2]: 5 x 5 waves + 2.7 waves
    s, ln = plan(1 << 23)                                       # configs[3] on one GPU
    assert s == 8 and ln % wave == 0 and (s - 1) * ln < (1 << 23) <= s * ln
    assert plan(1 << 23, single=1) == (1, 1 << 23)
    for n in (wave * 9 + 5, 3 * (1 << 20) + 17, 1 << 25):
        s, ln = plan(n)
        assert 1 <= s <= 8 and ln % wave == 0 and (s - 1) * ln < n <= s * ln and ln >= 4 * wave
    assert lib.pime_set_host_slices(3) == 0
    try:
        assert plan(1000) == (3, 512) and plan(300) == (2, 256) and plan(100) == (1, 100)
    finally:
        assert lib.pime_set_host_slices(0) == 0
    assert lib.pime_set_host_slices(9) != 0
