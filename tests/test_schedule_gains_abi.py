"""CPU tests of the scheduled rollout entries with per-env controller gains (pime_*_rollout_schedule_gains_*): the
pime_schedule_gains layout matches its ctypes mirror, every bad argument is PIME_EINVAL before any device check, the
Tracked kernels compile as they did before the Gained kernels existed, and the Gained tcgen05 kernels of the fp32 plants
keep every value in registers."""
import ctypes as C
import json
import os
import subprocess
import sys

import pytest

from test_schedule_abi import PKG, ROOT, _cuobjdump, kernel_table, nvcc_release

ENTRIES = ("pime_wt_rollout_schedule_gains_f32", "pime_wt_rollout_schedule_gains_f64",
           "pime_ph_rollout_schedule_gains_f32", "pime_ph_rollout_schedule_gains_f64")
GOLDEN = os.path.join(ROOT, "tests", "golden", "track_kernels.json")


@pytest.fixture(scope="module")
def L():
    sys.path.insert(0, ROOT)
    import pime_b200.build as build
    build.build()
    import pime_b200._lib as lib
    return lib


def test_schedule_gains_layout_matches_header(L, tmp_path):
    prog = tmp_path / "gains.c"
    prog.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "pime_b200.h"\nint main(){'
                    'printf("%zu %zu %d\\n", sizeof(pime_schedule_gains), offsetof(pime_schedule_gains, priorK_dev),'
                    'PIME_B200_ABI_VERSION);return 0;}')
    exe = tmp_path / "gains"
    subprocess.run(["gcc", "-I", os.path.join(ROOT, "include"), str(prog), "-o", str(exe)], check=True)
    got = [int(v) for v in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split()]
    G = L.ScheduleGains
    assert got == [C.sizeof(G), G.priorK_dev.offset, 5]


def test_bad_arguments_are_rejected_before_the_device_check(L):
    """n = 0, valid config and state: each of the four entries rejects a sample of what the _response entries reject, a
    missing gain block or matrix, a priorK_host given besides the matrix and the stacking observation with PIME_EINVAL,
    with or without a GPU; a good call is PIME_OK with a device and PIME_ENODEV without, with and without an extension."""
    lib = L.lib()
    buf = (C.c_double * 8)()
    p = C.cast(buf, C.c_void_p)
    sp = (C.c_double * 32)(*range(32))
    wst = L.WtState(**{f: p for f, _ in L.WtState._fields_})
    pst = L.PhState(**{f: p for f, _ in L.PhState._fields_})
    pcfg = L.ph_config()
    actor = L.ActorConfig(kind=L.ACTOR_PLAIN, state_dim=4, mid_dim=64)
    n0 = C.c_int64(0)

    def call(fn, sched, args, ext, resp, gains, wcfg=None):
        refs = [C.byref(v) if v is not None else None for v in (args, sched, ext, resp, gains)]
        if "_wt_" in fn:
            return getattr(lib, fn)(C.byref(wcfg or L.wt_config()), n0, C.byref(wst), *refs, None)
        return getattr(lib, fn)(C.byref(pcfg), p, n0, C.byref(pst), *refs, None)

    def good(policy=L.POLICY_ACTOR, per_env=False, with_ext=True):
        s = L.Schedule(num_segments=5, segment_steps=3, resample_params=0, setpoints_host=None if per_env else sp, metrics=p)
        a = L.RolloutArgs(actor=None, priorK_host=None, T=15, deterministic=1)
        x = L.ScheduleExt(setpoints_dev=p if per_env else None, policy=policy) if with_ext else None
        return s, a, x, L.StepResponse(response=p, settle_band=0.02), L.ScheduleGains(priorK_dev=p)

    bad = []
    # a sample of what the _response entries reject
    s, a, x, r, g = good()
    a.auto_reset = 1
    bad.append(("auto_reset", s, a, x, r, g))
    s, a, x, r, g = good()
    a.T = 16
    bad.append(("T != K L", s, a, x, r, g))
    s, a, x, r, g = good()
    r.settle_band = 1.0
    bad.append(("settle_band=1", s, a, x, r, g))
    s, a, x, r, g = good()
    r.settle_band = float("nan")
    bad.append(("settle_band=nan", s, a, x, r, g))
    s, a, x, r, g = good()
    bad.append(("null response block", s, a, x, None, g))
    s, a, x, r, g = good(L.POLICY_LINEAR)
    a.actor = C.pointer(actor)
    a.actor_pack = p
    bad.append(("linear with an actor", s, a, x, r, g))
    s, a, x, r, g = good()
    bad.append(("null schedule", None, a, x, r, g))
    # the gains' own rules
    for with_ext in (True, False):
        s, a, x, r, g = good(with_ext=with_ext)
        bad.append((f"null gain block, ext={with_ext}", s, a, x, r, None))
        s, a, x, r, g = good(with_ext=with_ext)
        g.priorK_dev = None
        bad.append((f"null priorK_dev, ext={with_ext}", s, a, x, r, g))
        s, a, x, r, g = good(with_ext=with_ext)
        a.priorK_host = (C.c_double * 4)()
        bad.append((f"priorK_host given, ext={with_ext}", s, a, x, r, g))
    for fn in ENTRIES:
        for what, s, a, x, r, g in bad:
            assert call(fn, s, a, x, r, g) == L.EINVAL, (fn, what)
    stack = L.wt_config(obs_mode=L.WT_OBS_STACKING, num_stack=4)
    for fn in ENTRIES[:2]:
        for with_ext in (True, False):
            s, a, x, r, g = good(with_ext=with_ext)
            assert call(fn, s, a, x, r, g, wcfg=stack) == L.EINVAL, (fn, "stacking")
    import torch
    want = L.OK if torch.cuda.is_available() else L.ENODEV
    for fn in ENTRIES:
        for policy in (L.POLICY_ACTOR, L.POLICY_LINEAR):
            for per_env in (False, True):
                s, a, x, r, g = good(policy, per_env)
                assert call(fn, s, a, x, r, g) == want, (fn, policy, per_env, lib.pime_last_error())
        s, a, x, r, g = good(with_ext=False)
        a.deterministic = 0
        assert call(fn, s, a, x, r, g) == want, fn
    for obs in (L.WT_OBS_GOAL, L.WT_OBS_INTEGRATOR):
        for fn in ENTRIES[:2]:
            s, a, x, r, g = good()
            assert call(fn, s, a, x, r, g, wcfg=L.wt_config(obs_mode=obs)) == want, (fn, obs)


def test_tracked_kernels_compile_as_before(L):
    """Per-env gains are a separate instantiation (Gained<Glue>) in objects of their own, and their reads are behind
    kGained, which every other glue sets to false.  Every Tracked kernel keeps the figures recorded in
    tests/golden/track_kernels.json (taken from the build before the Gained kernels existed, same nvcc)."""
    golden = json.load(open(GOLDEN))
    if _cuobjdump() is None:
        pytest.skip("cuobjdump not found")
    if nvcc_release() != golden["nvcc"]:
        pytest.skip(f"figures recorded with nvcc {golden['nvcc']}, this is {nvcc_release()}")
    build_dir = os.path.join(PKG, "build")
    assert len(golden["objects"]) == 4
    for obj, want in golden["objects"].items():
        got = kernel_table(build_dir, obj)
        assert got == want, obj
        assert not any("Gained" in k for k in got), obj


def test_gained_f32_tcgen05_kernels_do_not_spill(L):
    """ptxas -v of the four Gained objects: each holds the 10 kernels (tcgen05 plain / modular at four H, fidelity, prior)
    of a non-stacking glue on Gained<...>; no Gained tcgen05 kernel of the fp32 water tank spills, and no fp32 pH one
    spills more than its Tracked twin."""
    if _cuobjdump() is None:
        pytest.skip("cuobjdump not found")
    build_dir = os.path.join(PKG, "build")
    checked = 0
    for plant in ("wt", "ph"):
        for dt in ("f32", "f64"):
            got = kernel_table(build_dir, f"rollout_gain_{plant}_{dt}.o")
            tracked = kernel_table(build_dir, f"rollout_track_{plant}_{dt}.o")
            assert len(got) == 10 and all("Gained" in k for k in got), (plant, dt, sorted(got)[:4])
            assert not any("Lb1E" in k for k in got), (plant, dt)   # no stacking glue
            for name in got:
                assert name.replace("NS_6GainedINS_6", "NS_7TrackedINS_6") in tracked, name
            if dt != "f32":
                continue
            for name, fig in got.items():
                if not name.startswith("_ZN4pime14rollout_kernel"):
                    continue
                twin = tracked[name.replace("NS_6GainedINS_6", "NS_7TrackedINS_6")]
                if plant == "wt":
                    assert fig[2] == fig[3] == 0, (name, fig)
                else:
                    assert fig[2] <= twin[2] and fig[3] <= twin[3], (name, fig, twin)
                checked += 1
    assert checked == 16, checked   # water tank 8, pH 8
