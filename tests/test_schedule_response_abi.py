"""CPU tests of the scheduled rollout entries with the step response (pime_*_rollout_schedule_response_*): the
pime_step_response layout matches its ctypes mirror, every bad argument is PIME_EINVAL before any device check, the
Segmented kernels compile as they did before the Tracked kernels existed, and the Tracked tcgen05 kernels of the fp32
plants keep every value in registers."""
import ctypes as C
import json
import os
import subprocess
import sys

import pytest

from test_schedule_abi import PKG, ROOT, _cuobjdump, kernel_table, nvcc_release

ENTRIES = ("pime_wt_rollout_schedule_response_f32", "pime_wt_rollout_schedule_response_f64",
           "pime_ph_rollout_schedule_response_f32", "pime_ph_rollout_schedule_response_f64")
GOLDEN = os.path.join(ROOT, "tests", "golden", "schedule_kernels.json")


@pytest.fixture(scope="module")
def L():
    sys.path.insert(0, ROOT)
    import pime_b200.build as build
    build.build()
    import pime_b200._lib as lib
    return lib


def test_step_response_layout_matches_header(L, tmp_path):
    prog = tmp_path / "resp.c"
    prog.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "pime_b200.h"\nint main(){'
                    'printf("%zu %zu %zu %d\\n", sizeof(pime_step_response), offsetof(pime_step_response, response),'
                    'offsetof(pime_step_response, settle_band), PIME_B200_ABI_VERSION);return 0;}')
    exe = tmp_path / "resp"
    subprocess.run(["gcc", "-I", os.path.join(ROOT, "include"), str(prog), "-o", str(exe)], check=True)
    got = [int(v) for v in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split()]
    R = L.StepResponse
    assert got == [C.sizeof(R), R.response.offset, R.settle_band.offset, 5]


def test_bad_arguments_are_rejected_before_the_device_check(L):
    """n = 0, valid config and state: each of the four entries rejects what the _ext entries reject, a missing response
    block or buffer, a settle band outside (0, 1) and segments longer than 65535 steps with PIME_EINVAL, with or without a
    GPU; a good call is PIME_OK with a device and PIME_ENODEV without, with and without an extension block."""
    lib = L.lib()
    buf = (C.c_double * 8)()
    p = C.cast(buf, C.c_void_p)
    sp = (C.c_double * 32)(*range(32))
    wst = L.WtState(**{f: p for f, _ in L.WtState._fields_})
    pst = L.PhState(**{f: p for f, _ in L.PhState._fields_})
    wcfg, pcfg = L.wt_config(), L.ph_config()
    actor = L.ActorConfig(kind=L.ACTOR_PLAIN, state_dim=4, mid_dim=64)
    n0 = C.c_int64(0)

    def call(fn, sched, args, ext, resp):
        refs = [C.byref(v) if v is not None else None for v in (args, sched, ext, resp)]
        if "_wt_" in fn:
            return getattr(lib, fn)(C.byref(wcfg), n0, C.byref(wst), *refs, None)
        return getattr(lib, fn)(C.byref(pcfg), p, n0, C.byref(pst), *refs, None)

    def good(policy=L.POLICY_ACTOR, per_env=False, with_ext=True):
        s = L.Schedule(num_segments=5, segment_steps=3, resample_params=0, setpoints_host=None if per_env else sp, metrics=p)
        a = L.RolloutArgs(actor=None, priorK_host=(C.c_double * 4)(), T=15, deterministic=1)
        x = L.ScheduleExt(setpoints_dev=p if per_env else None, policy=policy) if with_ext else None
        return s, a, x, L.StepResponse(response=p, settle_band=0.02)

    bad = []
    # what the _ext entries reject
    for field, value in (("num_segments", 0), ("num_segments", 17), ("segment_steps", 0)):
        s, a, x, r = good()
        setattr(s, field, value)
        bad.append((f"{field}={value}", s, a, x, r))
    s, a, x, r = good()
    a.T = 16
    bad.append(("T != K L", s, a, x, r))
    s, a, x, r = good()
    a.auto_reset = 1
    bad.append(("auto_reset", s, a, x, r))
    s, a, x, r = good()
    a.priorK_host = None
    bad.append(("priorK_host", s, a, x, r))
    s, a, x, r = good()
    bad.append(("null schedule", None, a, x, r))
    s, a, x, r = good(with_ext=False)
    s.setpoints_host = None
    bad.append(("no ext, no set-points", s, a, x, r))
    for policy in (-1, 2):
        s, a, x, r = good()
        x.policy = policy
        bad.append((f"policy={policy}", s, a, x, r))
    s, a, x, r = good()
    x.reserved0 = 1
    bad.append(("reserved0", s, a, x, r))
    s, a, x, r = good()
    x.setpoints_dev = p
    bad.append(("both set-points", s, a, x, r))
    s, a, x, r = good(L.POLICY_LINEAR)
    a.actor = C.pointer(actor)
    a.actor_pack = p
    bad.append(("linear with an actor", s, a, x, r))
    s, a, x, r = good(L.POLICY_LINEAR, per_env=True)
    a.deterministic = 0
    bad.append(("linear, stochastic", s, a, x, r))
    # the step response's own rules
    for with_ext in (True, False):
        s, a, x, r = good(with_ext=with_ext)
        bad.append((f"null response block, ext={with_ext}", s, a, x, None))
        s, a, x, r = good(with_ext=with_ext)
        r.response = None
        bad.append((f"null response, ext={with_ext}", s, a, x, r))
        for band in (0.0, 1.0, -0.02, 1.5, float("nan"), float("inf"), -float("inf")):
            s, a, x, r = good(with_ext=with_ext)
            r.settle_band = band
            bad.append((f"settle_band={band}, ext={with_ext}", s, a, x, r))
        s, a, x, r = good(with_ext=with_ext)
        s.num_segments, s.segment_steps, a.T = 1, 65536, 65536
        bad.append((f"segment_steps=65536, ext={with_ext}", s, a, x, r))
    for fn in ENTRIES:
        for what, s, a, x, r in bad:
            assert call(fn, s, a, x, r) == L.EINVAL, (fn, what)
    import torch
    want = L.OK if torch.cuda.is_available() else L.ENODEV
    for fn in ENTRIES:
        for policy in (L.POLICY_ACTOR, L.POLICY_LINEAR):
            for per_env in (False, True):
                s, a, x, r = good(policy, per_env)
                assert call(fn, s, a, x, r) == want, (fn, policy, per_env, lib.pime_last_error())
        s, a, x, r = good(with_ext=False)
        a.deterministic = 0
        assert call(fn, s, a, x, r) == want, fn
        s, a, x, r = good(with_ext=False)
        s.num_segments, s.segment_steps, a.T = 1, 65535, 65535   # the longest segment the packed step counts hold
        r.settle_band = 0.999
        assert call(fn, s, a, x, r) == want, fn


def test_segmented_kernels_compile_as_before(L):
    """The step response is a separate instantiation (Tracked<Glue>) in objects of its own, and its code is behind
    kTracked, which a Segmented glue sets to false.  Every Segmented kernel keeps the figures recorded in
    tests/golden/schedule_kernels.json (taken from the build before the Tracked kernels existed, same nvcc)."""
    golden = json.load(open(GOLDEN))
    if _cuobjdump() is None:
        pytest.skip("cuobjdump not found")
    if nvcc_release() != golden["nvcc"]:
        pytest.skip(f"figures recorded with nvcc {golden['nvcc']}, this is {nvcc_release()}")
    build_dir = os.path.join(PKG, "build")
    for obj, want in golden["objects"].items():
        got = kernel_table(build_dir, obj)
        assert {k: v for k, v in got.items() if "Segmented" in k} == want, obj
        assert not any("Tracked" in k for k in got), obj


def test_tracked_f32_tcgen05_kernels_do_not_spill(L):
    """ptxas -v of the four Tracked objects: each holds the 16 / 10 kernels of its Segmented counterpart on Tracked<...>;
    no Tracked tcgen05 kernel of the fp32 water tank spills, and no pH one spills more than its plain twin."""
    if _cuobjdump() is None:
        pytest.skip("cuobjdump not found")
    build_dir = os.path.join(PKG, "build")
    checked = 0
    for plant, count in (("wt", 16), ("ph", 10)):
        for dt in ("f32", "f64"):
            got = kernel_table(build_dir, f"rollout_track_{plant}_{dt}.o")
            plain = kernel_table(build_dir, f"rollout_{plant}_{dt}.o")
            assert len(got) == count and all("Tracked" in k for k in got), (plant, dt, sorted(got)[:4])
            if dt != "f32":
                continue
            for name, fig in got.items():
                if not name.startswith("_ZN4pime14rollout_kernel"):
                    continue
                twin = name.replace("NS_7TrackedINS_6", "NS_6").replace("EEEEELi", "EEELi").replace("EEEELi", "EELi")
                assert twin in plain, (name, twin)
                if plant == "wt":
                    assert fig[2] == fig[3] == 0, (name, fig)
                else:
                    assert fig[2] <= plain[twin][2] and fig[3] <= plain[twin][3], (name, fig, plain[twin])
                checked += 1
    assert checked == 20, checked   # water tank 8 + 4 stacking, pH 8
