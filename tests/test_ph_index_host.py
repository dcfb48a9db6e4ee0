"""CPU tests (no GPU needed) of the pH titration-table index and of the configurations the library refuses.

The reference looks pH up as ``pH[np.argwhere(MHCl >= np.around(C*x, 5))[0]]`` (ph.py:187-189).  The oracle's
pime_oracle_ph_index restates that search for any uniform grid; the kernels' ph_lookup computes rint(C*x*1e5), which
is the same index on the grid i * 1e-5 only.  So every pH entry point and the gym front end reject any other step.
"""
import ctypes as C
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def L():
    sys.path.insert(0, ROOT)
    import pime_b200.build as build
    build.build()
    import pime_b200._lib as lib
    return lib


def _argwhere_index(MHCl, Cx):
    """ph.py:188 as written: first index with MHCl >= around(C x, 5); -1 where the reference raises IndexError"""
    hit = np.argwhere(MHCl >= np.around(Cx, 5))
    return int(hit[0][0]) if hit.size else -1


def _cx_samples(rng, stop):
    """C x products: random (C, x) of the registered ranges, values of C x 1e5 within a few ulp of a half-integer (where
    the rounding of around() decides the entry), 0, negatives, and values past the end of the grid"""
    C_ = rng.uniform(0.0015, 0.0025, 600)
    x = rng.uniform(0.0, stop / 0.0015, 600)
    cx = list(C_ * x)
    for k in rng.integers(0, int(stop * 1e5) - 1, 300):
        v = (k + 0.5) / 1e5
        cx += [v, np.nextafter(v, 0.0), np.nextafter(v, 1.0), np.nextafter(np.nextafter(v, 1.0), 1.0)]
    cx += [0.0, 4e-6, 6e-6, -3e-6, stop * 0.999, stop, stop * 1.001, 2 * stop]
    return np.array(cx)


@pytest.mark.parametrize("step,stop", [(1e-5, 0.2), (1e-5, 1.0), (2e-5, 0.2), (5e-6, 0.2), (1e-4, 1.0)])
def test_oracle_index_is_the_reference_argwhere(oracle, step, stop):
    MHCl = np.arange(0.0, stop, step)   # the grids gym_api accepts: np.arange(0, stop, step)
    cfg = oracle.ph_cfg(table_len=MHCl.shape[0], mhcl_step=step)
    assert np.array_equal(MHCl, np.arange(MHCl.shape[0]) * step)
    rng = np.random.default_rng(int(step * 1e7) + int(stop))
    cx = _cx_samples(rng, stop)
    want = np.array([_argwhere_index(MHCl, v) for v in cx])
    got = np.array([oracle.ph_index(cfg, float(v)) for v in cx])
    np.testing.assert_array_equal(got, want)
    assert (want == -1).any() and (want > 0).any()
    # the kernels' index rint(C x 1e5): the reference's entry on the 1e-5 grid, a different one on any other
    k = np.rint(cx * 1e5)
    live = want >= 0
    if step == 1e-5:
        np.testing.assert_array_equal(np.maximum(k[live], 0), want[live])
    else:
        assert (np.maximum(k[live], 0) != want[live]).mean() > 0.5


def test_kernel_index_of_the_product_is_the_reference_entry(oracle):
    """ph_lookup forms C*x and then *1e5 as two rounded products (not C*(x*1e5)): on the default grid that is the oracle's
    entry for random (C, x) of the registered ranges, including the products that land within an ulp of a half-integer"""
    rng = np.random.default_rng(3)
    MHCl = np.arange(0.0, 1, 0.00001)
    cfg = oracle.ph_cfg()
    C_ = rng.uniform(0.0015, 0.0025, 4000)
    x = rng.uniform(0.0, 300.0, 4000)
    k = np.rint(C_ * x * 1e5).astype(np.int64)
    # x nudged so that C x 1e5 sits on a half-integer up to rounding
    x2 = (np.floor(C_ * x * 1e5) + 0.5) / 1e5 / C_
    k2 = np.rint(C_ * x2 * 1e5).astype(np.int64)
    for kk, cx in ((k, C_ * x), (k2, C_ * x2)):
        want = np.array([oracle.ph_index(cfg, float(v)) for v in cx])
        np.testing.assert_array_equal(np.where(kk >= MHCl.shape[0], -1, kk), want)


BAD_STEPS = (2e-5, 5e-6, 1e-4, 1e-5 * (1 + 1e-15))


def test_every_ph_entry_rejects_another_grid_step(L):
    """mhcl_step != 1e-5 is PIME_EINVAL at every pH entry, before the device check and at n = 0 (nothing would run): with
    or without a GPU.  With the registered step the stand-alone entries are not rejected for their arguments (the table
    build with an accepted config writes the device; test_gpu_14 runs it on device tensors)."""
    lib = L.lib()
    buf = (C.c_double * 64)()
    p = C.cast(buf, C.c_void_p)
    ep_host = (C.c_float * 8)()
    sp = (C.c_double * 1)(7.0)
    args = L.RolloutArgs(actor=None, priorK_host=(C.c_double * 3)(), T=1)
    pst = L.PhState(**{f: p for f, _ in L.PhState._fields_})
    sc = L.Schedule(num_segments=1, segment_steps=1, setpoints_host=sp)
    resp = L.StepResponse(response=p, settle_band=0.02)
    gains = L.ScheduleGains(priorK_dev=p)
    n0 = C.c_int64(0)
    u64 = C.c_uint64(0)

    def stand_alone(cfg):
        """the step / reset / update_system entries: at n = 0 they return before touching any pointer, whatever the
        config, so they are also called with the accepted one"""
        c = C.byref(cfg)
        out = {}
        for dt in ("f32", "f64"):
            f = lambda name: getattr(lib, f"pime_ph_{name}_{dt}")   # noqa: E731
            out[f"update_system_{dt}"] = f("update_system")(c, n0, C.byref(pst), None)
            out[f"reset_{dt}"] = f("reset")(c, p, n0, C.byref(pst), u64, u64, 1, None, None, p, None)
            out[f"step_{dt}"] = f("step")(c, p, n0, C.byref(pst), p, None, p, p, p, None)
        return out

    def calls(cfg):
        """every pH entry; only ever called with a rejected config (the host buffers here are not device memory)"""
        c = C.byref(cfg)
        out = stand_alone(cfg)
        out["table_build"] = lib.pime_ph_table_build(c, p, p, None)
        out["rollout_host_f32"] = lib.pime_ph_rollout_host_f32(c, p, n0, C.byref(pst), C.byref(pst), C.byref(args), ep_host, None)
        for dt in ("f32", "f64"):
            f = lambda name: getattr(lib, f"pime_ph_{name}_{dt}")   # noqa: E731
            out[f"rollout_{dt}"] = f("rollout")(c, p, n0, C.byref(pst), C.byref(args), None)
            out[f"schedule_{dt}"] = f("rollout_schedule")(c, p, n0, C.byref(pst), C.byref(args), C.byref(sc), None)
            out[f"schedule_ext_{dt}"] = f("rollout_schedule_ext")(c, p, n0, C.byref(pst), C.byref(args), C.byref(sc),
                                                                  C.byref(L.ScheduleExt()), None)
            out[f"schedule_response_{dt}"] = f("rollout_schedule_response")(c, p, n0, C.byref(pst), C.byref(args), C.byref(sc),
                                                                            None, C.byref(resp), None)
            out[f"schedule_gains_{dt}"] = f("rollout_schedule_gains")(c, p, n0, C.byref(pst), C.byref(args), C.byref(sc), None,
                                                                      C.byref(resp), C.byref(gains), None)
        return out

    for step in BAD_STEPS:
        got = calls(L.ph_config(mhcl_step=step))
        assert all(rc == L.EINVAL for rc in got.values()), (step, got)
        assert b"mhcl_step" in lib.pime_last_error()
    ok = stand_alone(L.ph_config())
    assert all(rc != L.EINVAL for rc in ok.values()), ok


def test_table_build_rejects_before_the_device_check(L):
    import torch
    lib = L.lib()
    host = (C.c_double * 4)()
    for step in BAD_STEPS:
        assert lib.pime_ph_table_build(C.byref(L.ph_config(mhcl_step=step, table_len=4)), host, None, None) == L.EINVAL
    if not torch.cuda.is_available():
        assert lib.pime_ph_table_build(C.byref(L.ph_config(table_len=4)), host, None, None) == L.ENODEV


@pytest.mark.parametrize("stop,step", [(0.2, 0.00002), (1.0, 0.000005), (1.0, 0.0001)])
def test_gym_env_rejects_another_grid_step(L, stop, step):
    """The reference accepts any MHCl; the gym classes raise for a grid they would look up differently, before any
    device work (so also without a GPU)"""
    import pime_b200.gym_api as G
    for cls in (G.PH1DChangingParamUniformGoalIntegrator, G.PH1DChangingParamUniformGoal,
                G.PH1DChangingParamUniformGoalIntegrator_NoBound):
        with pytest.raises(NotImplementedError, match="1e-5"):
            cls(MHCl=np.arange(0.0, stop, step))
