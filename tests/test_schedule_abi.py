"""CPU tests of the scheduled rollout entries (pime_*_rollout_schedule_*): the pime_schedule layout matches its ctypes
mirror, every bad schedule is PIME_EINVAL before any device check, and the scheduled kernels left the compiled code of
every pre-existing rollout kernel as it was (registers, stack, spills, shared memory, SASS instruction count)."""
import ctypes as C
import json
import os
import re
import shutil
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "pime-robust-non-linear-set-point-control-with-reinforcement-learning_b200")
GOLDEN = os.path.join(ROOT, "tests", "golden", "rollout_kernels.json")


@pytest.fixture(scope="module")
def L():
    sys.path.insert(0, ROOT)
    import pime_b200.build as build
    build.build()
    import pime_b200._lib as lib
    return lib


def test_schedule_layout_matches_header(L, tmp_path):
    prog = tmp_path / "sched.c"
    prog.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "pime_b200.h"\nint main(){'
                    'printf("%zu %zu %zu %zu %zu %zu %d\\n", sizeof(pime_schedule), offsetof(pime_schedule, segment_steps),'
                    'offsetof(pime_schedule, resample_params), offsetof(pime_schedule, reserved0),'
                    'offsetof(pime_schedule, setpoints_host), offsetof(pime_schedule, metrics), PIME_MAX_SEGMENTS);return 0;}')
    exe = tmp_path / "sched"
    subprocess.run(["gcc", "-I", os.path.join(ROOT, "include"), str(prog), "-o", str(exe)], check=True)
    got = [int(v) for v in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split()]
    S = L.Schedule
    assert got == [C.sizeof(S), S.segment_steps.offset, S.resample_params.offset, S.reserved0.offset,
                   S.setpoints_host.offset, S.metrics.offset, L.MAX_SEGMENTS]


def test_bad_schedules_are_rejected_before_the_device_check(L):
    """n = 0, valid config / state / prior-only argument block: nothing would be launched, so only the schedule (or the
    argument block it is checked against) can be what each of the four entries rejects -- with or without a GPU."""
    lib = L.lib()
    buf = (C.c_double * 8)()
    p = C.cast(buf, C.c_void_p)
    sp = (C.c_double * 32)(*range(32))
    wst = L.WtState(**{f: p for f, _ in L.WtState._fields_})
    pst = L.PhState(**{f: p for f, _ in L.PhState._fields_})
    wcfg, pcfg = L.wt_config(), L.ph_config()
    n0 = C.c_int64(0)

    def call(fn, sched, args):
        sched_ref = C.byref(sched) if sched is not None else None
        if "_wt_" in fn:
            return getattr(lib, fn)(C.byref(wcfg), n0, C.byref(wst), C.byref(args), sched_ref, None)
        return getattr(lib, fn)(C.byref(pcfg), p, n0, C.byref(pst), C.byref(args), sched_ref, None)

    def good():
        return (L.Schedule(num_segments=5, segment_steps=3, resample_params=0, setpoints_host=sp, metrics=p),
                L.RolloutArgs(actor=None, priorK_host=(C.c_double * 4)(), T=15))

    bad = []
    for field, value in (("num_segments", 0), ("num_segments", 17), ("num_segments", -1), ("segment_steps", 0),
                         ("segment_steps", -3), ("setpoints_host", None)):
        s, a = good()
        setattr(s, field, value)
        bad.append((f"{field}={value}", s, a))
    s, a = good()
    a.T = 16
    bad.append(("T != K L", s, a))
    s, a = good()
    a.auto_reset = 1
    bad.append(("auto_reset", s, a))
    s, a = good()
    bad.append(("null schedule", None, a))
    entries = ("pime_wt_rollout_schedule_f32", "pime_wt_rollout_schedule_f64", "pime_ph_rollout_schedule_f32",
               "pime_ph_rollout_schedule_f64")
    for fn in entries:
        for what, s, a in bad:
            assert call(fn, s, a) == L.EINVAL, (fn, what)
        # what the plain entries reject, the scheduled ones reject too
        s, a = good()
        a.priorK_host = None
        assert call(fn, s, a) == L.EINVAL, (fn, "priorK_host")
    for bad_cfg in ({"n_discrete": 0}, {"reward_type": 3}, {"obs_mode": 5}):
        cfg = L.wt_config(**bad_cfg)
        s, a = good()
        for fn in entries[:2]:
            assert getattr(lib, fn)(C.byref(cfg), n0, C.byref(wst), C.byref(a), C.byref(s), None) == L.EINVAL, bad_cfg
    cfg = L.ph_config(table_len=0)
    s, a = good()
    for fn in entries[2:]:
        assert getattr(lib, fn)(C.byref(cfg), p, n0, C.byref(pst), C.byref(a), C.byref(s), None) == L.EINVAL
        assert getattr(lib, fn)(C.byref(pcfg), None, n0, C.byref(pst), C.byref(a), C.byref(s), None) == L.EINVAL
    # a good schedule at n = 0 is accepted wherever a device is present, and fails only the device check otherwise
    import torch
    s, a = good()
    want = L.OK if torch.cuda.is_available() else L.ENODEV
    for fn in entries:
        assert call(fn, s, a) == want, fn


# ------------------------------------------------------------------------------------------------ compiled code
def nvcc_release():
    exe = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    out = subprocess.run([exe, "--version"], capture_output=True, text=True).stdout
    m = re.search(r"release (\S+), V(\S+)", out)
    return m.group(2) if m else None


def _cuobjdump():
    exe = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    return exe if os.path.exists(exe) else None


def kernel_table(build_dir, obj):
    """{mangled kernel name: [registers, stack, spill stores, spill loads, shared memory, SASS instructions]} of one object
    of build.py (its ptxas -v log is written beside it)."""
    res, cur = {}, None
    for line in open(os.path.join(build_dir, obj + ".log")):
        m = re.search(r"Compiling entry function '(\S+)'", line) or re.search(r"Function properties for (\S+)", line)
        if m:
            cur = m.group(1)
            res.setdefault(cur, [None] * 6)
        m = re.search(r"(\d+) bytes stack frame, (\d+) bytes spill stores, (\d+) bytes spill loads", line)
        if m and cur:
            res[cur][1:4] = [int(v) for v in m.groups()]
        m = re.search(r"Used (\d+) registers", line)
        if m and cur:
            res[cur][0] = int(m.group(1))
            m2 = re.search(r"(\d+) bytes smem", line)
            res[cur][4] = int(m2.group(1)) if m2 else 0
    out = subprocess.run([_cuobjdump(), "-sass", os.path.join(build_dir, obj)], capture_output=True, text=True, check=True).stdout
    cur = None
    for line in out.splitlines():
        m = re.match(r"\s+Function : (\S+)", line)
        if m:
            cur = m.group(1)
            res.setdefault(cur, [None] * 6)[5] = 0
        elif cur and re.match(r"\s+/\*[0-9a-f]{4,}\*/\s+\S", line):
            res[cur][5] += 1
    return {k: v for k, v in res.items() if v[5] is not None}


def test_plain_rollout_kernels_compile_as_before(L):
    """The scheduled launch is a separate instantiation (Segmented<Glue>) whose segment logic compiles to nothing for a
    plain glue.  Every rollout kernel that existed before it keeps the figures recorded in tests/golden/rollout_kernels.json
    (taken from the build without the scheduled kernels, same nvcc); the scheduled twins exist beside them."""
    golden = json.load(open(GOLDEN))
    if _cuobjdump() is None:
        pytest.skip("cuobjdump not found")
    if nvcc_release() != golden["nvcc"]:
        pytest.skip(f"figures recorded with nvcc {golden['nvcc']}, this is {nvcc_release()}")
    build_dir = os.path.join(PKG, "build")
    for obj, want in golden["objects"].items():
        got = kernel_table(build_dir, obj)
        for name, fig in want.items():
            assert got.get(name) == fig, (obj, name, fig, got.get(name))
        new = set(got) - set(want)
        assert new and all("Segmented" in k for k in new), (obj, sorted(new)[:4])
        assert len(new) == len(want), obj
