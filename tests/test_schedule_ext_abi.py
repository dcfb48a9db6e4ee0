"""CPU tests of the scheduled rollout entries with an extension block (pime_*_rollout_schedule_ext_*): the
pime_schedule_ext layout matches its ctypes mirror, every bad extension is PIME_EINVAL before any device check, and the
scheduled tcgen05 kernels of the fp32 plants still keep every value in registers."""
import ctypes as C
import os
import subprocess
import sys

import pytest

from test_schedule_abi import PKG, ROOT, kernel_table, _cuobjdump

ENTRIES = ("pime_wt_rollout_schedule_ext_f32", "pime_wt_rollout_schedule_ext_f64", "pime_ph_rollout_schedule_ext_f32",
           "pime_ph_rollout_schedule_ext_f64")


@pytest.fixture(scope="module")
def L():
    sys.path.insert(0, ROOT)
    import pime_b200.build as build
    build.build()
    import pime_b200._lib as lib
    return lib


def test_schedule_ext_layout_matches_header(L, tmp_path):
    prog = tmp_path / "ext.c"
    prog.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "pime_b200.h"\nint main(){'
                    'printf("%zu %zu %zu %zu %d %d %d\\n", sizeof(pime_schedule_ext), offsetof(pime_schedule_ext, setpoints_dev),'
                    'offsetof(pime_schedule_ext, policy), offsetof(pime_schedule_ext, reserved0), PIME_POLICY_ACTOR,'
                    'PIME_POLICY_LINEAR, PIME_B200_ABI_VERSION);return 0;}')
    exe = tmp_path / "ext"
    subprocess.run(["gcc", "-I", os.path.join(ROOT, "include"), str(prog), "-o", str(exe)], check=True)
    got = [int(v) for v in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split()]
    X = L.ScheduleExt
    assert got == [C.sizeof(X), X.setpoints_dev.offset, X.policy.offset, X.reserved0.offset, L.POLICY_ACTOR, L.POLICY_LINEAR, 5]


def test_bad_extensions_are_rejected_before_the_device_check(L):
    """n = 0, valid config and state: each of the four entries rejects every bad schedule / extension / argument combination
    with PIME_EINVAL, with or without a GPU; a good one is PIME_OK with a device and PIME_ENODEV without."""
    lib = L.lib()
    buf = (C.c_double * 8)()
    p = C.cast(buf, C.c_void_p)
    sp = (C.c_double * 32)(*range(32))
    wst = L.WtState(**{f: p for f, _ in L.WtState._fields_})
    pst = L.PhState(**{f: p for f, _ in L.PhState._fields_})
    wcfg, pcfg = L.wt_config(), L.ph_config()
    actor = L.ActorConfig(kind=L.ACTOR_PLAIN, state_dim=4, mid_dim=64)
    n0 = C.c_int64(0)

    def call(fn, sched, args, ext):
        refs = [C.byref(v) if v is not None else None for v in (args, sched, ext)]
        if "_wt_" in fn:
            return getattr(lib, fn)(C.byref(wcfg), n0, C.byref(wst), *refs, None)
        return getattr(lib, fn)(C.byref(pcfg), p, n0, C.byref(pst), *refs, None)

    def good(policy=L.POLICY_ACTOR, per_env=False):
        s = L.Schedule(num_segments=5, segment_steps=3, resample_params=0, setpoints_host=None if per_env else sp, metrics=p)
        a = L.RolloutArgs(actor=None, priorK_host=(C.c_double * 4)(), T=15, deterministic=1)
        x = L.ScheduleExt(setpoints_dev=p if per_env else None, policy=policy)
        return s, a, x

    bad = []
    # what the entries without an extension reject
    for field, value in (("num_segments", 0), ("num_segments", 17), ("segment_steps", 0)):
        s, a, x = good()
        setattr(s, field, value)
        bad.append((f"{field}={value}", s, a, x))
    s, a, x = good()
    a.T = 16
    bad.append(("T != K L", s, a, x))
    s, a, x = good()
    a.auto_reset = 1
    bad.append(("auto_reset", s, a, x))
    s, a, x = good()
    a.priorK_host = None
    bad.append(("priorK_host", s, a, x))
    s, a, x = good()
    bad.append(("null schedule", None, a, x))
    # the extension's own rules
    s, a, x = good()
    bad.append(("null ext", s, a, None))
    for policy in (-1, 2, 7):
        s, a, x = good()
        x.policy = policy
        bad.append((f"policy={policy}", s, a, x))
    for policy in (L.POLICY_ACTOR, L.POLICY_LINEAR):
        s, a, x = good(policy)
        x.reserved0 = 1
        bad.append((f"reserved0, policy={policy}", s, a, x))
        s, a, x = good(policy)
        s.setpoints_host = None
        bad.append((f"no set-points, policy={policy}", s, a, x))
        s, a, x = good(policy)
        x.setpoints_dev = p
        bad.append((f"both set-points, policy={policy}", s, a, x))
    s, a, x = good(L.POLICY_LINEAR)
    a.actor = C.pointer(actor)
    a.actor_pack = p
    bad.append(("linear with an actor", s, a, x))
    s, a, x = good(L.POLICY_LINEAR, per_env=True)
    a.deterministic = 0
    bad.append(("linear, stochastic", s, a, x))
    for fn in ENTRIES:
        for what, s, a, x in bad:
            assert call(fn, s, a, x) == L.EINVAL, (fn, what)
    import torch
    want = L.OK if torch.cuda.is_available() else L.ENODEV
    for fn in ENTRIES:
        for policy in (L.POLICY_ACTOR, L.POLICY_LINEAR):
            for per_env in (False, True):
                s, a, x = good(policy, per_env)
                assert call(fn, s, a, x) == want, (fn, policy, per_env, lib.pime_last_error())
        s, a, x = good()
        a.deterministic = 0     # the actor policy may be stochastic
        assert call(fn, s, a, x) == want, fn


def test_scheduled_f32_tcgen05_kernels_do_not_spill(L):
    """ptxas -v of the four rollout objects: no scheduled (Segmented) tcgen05 kernel of an fp32 plant spills more than its
    plain twin -- 0 bytes for each but the pH plain-actor H = 256 kernel, whose plain instantiation spills 12 bytes too."""
    if _cuobjdump() is None:
        pytest.skip("cuobjdump not found")
    build_dir = os.path.join(PKG, "build")
    checked = 0
    for obj in ("rollout_wt_f32.o", "rollout_wt_f64.o", "rollout_ph_f32.o", "rollout_ph_f64.o"):
        got = kernel_table(build_dir, obj)
        for name, fig in got.items():
            if "Segmented" not in name or not name.startswith("_ZN4pime14rollout_kernel"):
                continue
            if "GlueIf" not in name:   # WtGlue<float, ...> / PhGlue<float>
                continue
            twin = name.replace("NS_9SegmentedINS_6", "NS_6").replace("EEEEELi", "EEELi").replace("EEEELi", "EELi")
            assert twin in got, (name, twin)
            assert fig[2] <= got[twin][2] and fig[3] <= got[twin][3], (obj, name, fig, got[twin])
            if "WtGlue" in name:
                assert fig[2] == fig[3] == 0, (obj, name, fig)
            checked += 1
    assert checked == 20, checked   # water tank 8 + 4 stacking, pH 8
