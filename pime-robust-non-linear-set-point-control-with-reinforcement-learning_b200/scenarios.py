"""Batched evaluation scenarios: the reference's staircase set-point tests and robust-test parameter sweeps, every env
of a vec object at once, returning the arrays the reference's plot scripts consume (no plotting here), or per-env
tracking metrics only.

  utils/test.py:70-207        test_policy_uniform            water tank, set-points 2, 6, 9, 4, 1
  utils/test.py:209-347       test_policy_uniform_integrator water tank + integrator, set-points 3, 6, 9, 4, 2
  utils/test.py:1369-1407     test_ph_policy_uniform_integrator   pH, set-points 10, 6, 3, 8, 5
  utils/test.py:1056-1067     test_watertank: agent (deterministic) vs env.get_linear_action (the CLIPPED prior)
  utils/robust_test.py:4-47   robust_test_nonlinear_watertank: off-nominal (a1, a2, Kp), max_step = 500, if_reset_all = False
  utils/test.py:1225-1240     the pH robust sets: off-nominal (qww_V, qc_V)

The whole staircase of the agent policy is ONE fused launch (vec.rollout_schedule): between segments the kernel does
what the reference does -- reset() (new ensemble member unless if_reset_all is False, t = 0, I = 0), restore the plant
state, set the next set-point -- and it keeps per env and segment the return, the integral of |r - y|, the final |r - y|
and the overshoot.  ``staircase`` returns the trajectories of that launch; ``staircase_metrics`` and ``robust_map``
return the metrics alone ([K, n] per metric, no trajectory buffers), which is what a robustness map over millions of
ensemble members needs.  ``staircase_metrics`` and ``robust_map`` run either policy in that one launch -- the clipped
linear baseline (get_linear_action, computed in the plant dtype) as well as the agent -- and take either one staircase for
every env or a [K, n] matrix of per-env set-points (e.g. random staircases in [r_lo, r_hi], or a map over set-point
sequence x ensemble parameters).  With ``response=True`` the same launch also returns each segment's step response --
settling time, rise time, control effort (total variation of the action) and peak action -- without any trajectory, so a
map can show where a policy commands more than the actuator takes.  Both also take the controller gains K per env ([S, n],
column i for env i), which is what a gain x plant map -- the fairness of the linear baseline, or the sensitivity of the
residual agent to the prior it runs over (fix_K) -- needs, in the same one launch.  ``staircase(policy='linear')`` keeps the per-step
loop of the prior kernel + the step kernel, which returns the same trajectories in fp64 and is what the fused linear
policy is tested against.
"""
from __future__ import annotations

import contextlib
from typing import Optional, Sequence

import numpy as np
import torch

from . import vec as V

WT_SETPOINTS = (2.0, 6.0, 9.0, 4.0, 1.0)
WT_INTEGRATOR_SETPOINTS = (3.0, 6.0, 9.0, 4.0, 2.0)
PH_SETPOINTS = (10.0, 6.0, 3.0, 8.0, 5.0)


def _is_wt(vec):
    return isinstance(vec, V.WaterTankVec)


@contextlib.contextmanager
def _staircase_setup(vec, setpoints, steps):
    """(set-points, steps per segment) with the reference's defaults, episodes never terminating inside a segment (the
    reference ignores `done` here: the step limit is lifted while the staircase runs)."""
    wt = _is_wt(vec)
    if setpoints is None:
        setpoints = (WT_INTEGRATOR_SETPOINTS if vec.obs_mode == "integrator" else WT_SETPOINTS) if wt else PH_SETPOINTS
    limit_field = "max_step" if wt else "max_episode_steps"
    saved_limit = getattr(vec.cfg, limit_field)
    steps = int(steps or saved_limit)
    setattr(vec.cfg, limit_field, 2 ** 30)
    try:
        yield setpoints, steps
    finally:
        setattr(vec.cfg, limit_field, saved_limit)


def _scheduled(vec, K, actor, setpoints, steps, resample_params, start, trajectories, policy="agent", response=False,
               settle_band=0.02):
    """The deterministic agent (or linear) policy over the whole staircase in one scheduled launch; the first segment
    restores ``start`` after its reset (utils/test.py:102-104)."""
    if policy not in ("agent", "linear"):
        raise ValueError("policy must be 'agent' or 'linear'")
    if policy == "linear" and actor is not None:
        raise ValueError("the linear policy takes no actor")
    if np.ndim(K) > 2:
        raise ValueError("K must be [S] or [S, n]")
    if np.ndim(K) == 2:   # per-env gains: column i is env i's K
        priorK = -torch.as_tensor(K, dtype=torch.float64)
    else:
        priorK = -np.asarray(K, dtype=np.float64).reshape(-1)[:vec.state_dim]
    with _staircase_setup(vec, setpoints, steps) as (setpoints, steps):
        if _is_wt(vec):
            vec.set_state(*start)
        else:
            vec.x.fill_(float(start[0]))
        return vec.rollout_schedule(setpoints, steps, priorK, actor=actor, deterministic=True,
                                    replay=trajectories, want_actions=trajectories, resample_params=resample_params,
                                    policy="actor" if policy == "agent" else "linear", response=response,
                                    settle_band=settle_band)


def _begin_segment(vec, r, resample, first, start):
    """reset(); set_state(previous plant state); set_r(r)  (utils/test.py:102-106, :1386-1388)."""
    if _is_wt(vec):
        keep = (vec.h1.clone(), vec.h2.clone())
        vec.reset(resample_params=resample)
        if first:
            vec.set_state(*start)
        else:
            vec.set_state(*keep)
        vec.set_r(r)
    else:
        keep = vec.x.clone()
        vec.reset(resample_params=resample)
        vec.x.copy_(torch.full_like(keep, float(start[0])) if first else keep)
        idx = torch.round(vec.C * vec.x * 1e5).long().clamp_(0, vec.table.numel() - 1)
        vec.y.copy_(vec.table[idx])                       # observe_state (ph.py:187-189) of the restored state
        vec.r.fill_(float(r))


def staircase(vec, policy: str, K, actor: Optional[V.ActorPack] = None, setpoints: Optional[Sequence[float]] = None,
              steps: Optional[int] = None, resample_params: bool = False, start=(0.0, 0.0)):
    """Run the staircase on every env of ``vec``.

    policy = 'agent': deterministic ``tanh(net(obs)) + obs @ (-K)`` (``actor`` = the agent's ActorPack; None = prior only);
    policy = 'linear': ``clip(-obs @ K, -1, 1)`` for the water tank (get_P_action), ``-obs @ K`` for pH (ph.py:227-231).
    K: [S], or [S, n] with column i for env i (policy='agent' only: the linear policy's per-step loop takes one K).
    Returns time-major arrays over all segments: obs [T, n, S] (the states the policy saw), xs [T, n, 2] (levels) or
    ys [T, n] (pH), refs [T, n], actions [T, n], rewards [T, n], totals [T, n] (running sum), integrators [T, n] or None.
    """
    wt = _is_wt(vec)
    # stacking observation: set_state / set_r do not touch the frame history (nonlinear_watertank.py:205-212 are inherited
    # unchanged), so the first num_stack observations of a segment still show the frames of the reset -- reproduced
    if np.ndim(K) == 2:
        if policy == "linear":
            raise ValueError("staircase(policy='linear') takes one K ([S]); per-env gains go through staircase_metrics")
    else:
        K = np.asarray(K, dtype=np.float64).reshape(-1)
    S = vec.state_dim
    if policy == "agent":
        out = _scheduled(vec, K, actor, setpoints, steps, resample_params, start, True)
        obs, actions, rewards = out["buf_state"], out["env_action"].float(), out["buf_other"][..., 0]
    elif policy == "linear":
        obs_l, act_l, rew_l = [], [], []
        with _staircase_setup(vec, setpoints, steps) as (setpoints, steps):
            for k, r in enumerate(setpoints):
                _begin_segment(vec, r, resample_params, k == 0, start)
                o_seg = torch.empty((steps, vec.n, S), dtype=torch.float32, device=vec.device)
                a_seg = torch.empty((steps, vec.n), dtype=torch.float32, device=vec.device)
                r_seg = torch.empty((steps, vec.n), dtype=torch.float32, device=vec.device)
                obs = vec.observe()
                for t in range(steps):
                    a = vec.prior_action(obs, K[:S], clip=wt)
                    o_seg[t] = obs.t()
                    a_seg[t] = a
                    obs, rew, _ = vec.step(a)
                    r_seg[t] = rew
                obs_l.append(o_seg); act_l.append(a_seg); rew_l.append(r_seg)
        obs, actions, rewards = torch.cat(obs_l), torch.cat(act_l), torch.cat(rew_l)
    else:
        raise ValueError("policy must be 'agent' or 'linear'")
    res = {"obs": obs, "actions": actions, "rewards": rewards, "totals": torch.cumsum(rewards.double(), 0)}
    if wt and vec.obs_mode == "stacking":   # env.state = the newest frame (update_state_P :1151-1153)
        res.update(xs=obs[..., -3:-1], refs=obs[..., -1], integrators=None)
    elif wt:
        res.update(xs=obs[..., :2], refs=obs[..., 2], integrators=obs[..., 3] if vec.obs_mode == "integrator" else None)
    else:
        res.update(ys=obs[..., 0], refs=obs[..., 1], integrators=obs[..., 2] if S == 3 else None)
    return res


METRICS = ("ret", "iae", "final_err", "overshoot")
RESPONSE = ("settle", "rise", "effort", "peak_action")


def staircase_metrics(vec, K, actor: Optional[V.ActorPack] = None, setpoints=None, steps: Optional[int] = None,
                      resample_params: bool = False, start=(0.0, 0.0), policy: str = "agent", response: bool = False,
                      settle_band: float = 0.02):
    """The staircase of ``staircase`` as one launch without trajectories: {"ret", "iae", "final_err", "overshoot"}, each
    [K, n] float64 (segment k, env i).  With y the controlled output (h2 / pH) and e = r - y: ret = sum of rewards, iae =
    sum of |e| over the segment's steps, final_err = |e| after its last step, overshoot = max(0, max of d (y - r)) with
    d = +1 when the segment starts below its set-point, -1 when above.
    policy: 'agent' or 'linear' as in ``staircase`` (K is the reference's K; 'linear' takes no actor).  K: [S] for every
    env, or a [S, n] array / tensor (column i: env i's K; not with the stacking observation).  setpoints: K floats for
    every env, or a [K, n] array / tensor (column i: env i's staircase).
    response=True adds the step response of each segment, [K, n] float64 each, computed in the same launch (L steps per
    segment, j = 0 .. L-1, u_j the action fed to the plant, y_b the output at the segment begin, D = |r - y_b|):
    settle = 1 + the last j with |e_j| > settle_band D (0: always inside the band, L: not settled); rise = 1 + the first j
    at which y has covered 90 % of D (-1: never, 0: D = 0); effort = sum of |u_j - u_{j-1}|; peak_action = max |u_j|."""
    out = _scheduled(vec, K, actor, setpoints, steps, resample_params, start, False, policy, response, settle_band)
    res = dict(zip(METRICS, out["metrics"].unbind(0)))
    if response:
        res.update(zip(RESPONSE, out["response"].unbind(0)))
    return res


def robust_map(K, params, actor: Optional[V.ActorPack] = None, plant: str = "wt", setpoints=None, steps=None,
               dtype=torch.float32, device="cuda", obs_mode="integrator", integrator="integrator", policy="agent",
               response: bool = False, settle_band: float = 0.02, **cfg):
    """Tracking metrics of the agent (or, policy='linear', the clipped linear baseline) policy over any number of off-nominal
    parameter sets, one env per set, in one launch.  setpoints: K floats, or [K, n] with column i for parameter row i.
    plant = 'wt': rows (a1, a2, Kp) as in robust_sweep (utils/robust_test.py), steps default 500; plant = 'ph': rows
    (qww_V, qc_V) with the discretised system refreshed (set_params(update_system=True)), steps default
    max_episode_steps.  The ensemble parameters are kept between segments (if_reset_all = False).  A grid over the axes
    is one np.meshgrid (or parameter_grid) in the caller.  response / settle_band: the step response, as in
    staircase_metrics.  Returns (metrics dict as staircase_metrics, params array).

    K: the reference's K (= -priorK), [S] for every row, or [S, n] with column i for parameter row i.  A gain x plant map
    is one np.repeat / np.tile in the caller; e.g. the water-tank integrator loop u = kp (r - h2) + ki I, i.e.
    K = [0, kp, -kp, -ki], over a (kp, ki) grid times a plant grid P ([m, 3]):

        kp, ki = np.meshgrid(kps, kis, indexing="ij")                        # G = kp.size gains
        Kg = np.stack([0 * kp, kp, -kp, -ki]).reshape(4, -1)                  # [4, G]
        K = np.repeat(Kg, len(P), axis=1)                                     # gain g for rows g m .. g m + m - 1
        metrics, p = robust_map(K, np.tile(P, (Kg.shape[1], 1)), policy="linear", response=True)

    (metrics[...][k].reshape(G, m) is then the map of segment k).  The ensemble parameter Kp in ``params`` is the pump
    constant of the plant (nonlinear_watertank.py), not a controller gain."""
    if plant == "wt":
        p = np.asarray(params, dtype=np.float64).reshape(-1, 3)
        steps = int(steps or 500)
        env = V.WaterTankVec(p.shape[0], dtype=dtype, device=device, obs_mode=obs_mode, max_step=steps, **cfg)
        env.reset()
        env.reset_changable_parameters(torch.as_tensor(p[:, 0]), torch.as_tensor(p[:, 1]), torch.as_tensor(p[:, 2]))
    elif plant == "ph":
        p = np.asarray(params, dtype=np.float64).reshape(-1, 2)
        env = V.PHVec(p.shape[0], dtype=dtype, device=device, integrator=integrator, **cfg)
        env.reset()
        env.set_params(torch.as_tensor(p[:, 0]), torch.as_tensor(p[:, 1]), update_system=True)
    else:
        raise ValueError("plant must be 'wt' or 'ph'")
    return staircase_metrics(env, K, actor=actor, setpoints=setpoints, steps=steps, resample_params=False, policy=policy,
                             response=response, settle_band=settle_band), p


ROBUST_TESTS = ((0.0024, 0.0019, 0.12), (0.0024, 0.0015, 0.12), (0.0024, 0.0015, 0.07))   # utils/robust_test.py:12-37


def robust_sweep(K, actor: Optional[V.ActorPack] = None, params=ROBUST_TESTS, obs_mode="integrator", max_step=500,
                 dtype=torch.float32, device="cuda", policy="agent", setpoints=None, **cfg):
    """robust_test_nonlinear_watertank for any list / grid of (a1, a2, Kp): one env per parameter set, all sets in the
    same launches.  Returns (staircase result dict, params array [n, 3])."""
    p = np.asarray(params, dtype=np.float64).reshape(-1, 3)
    env = V.WaterTankVec(p.shape[0], dtype=dtype, device=device, obs_mode=obs_mode, max_step=max_step, **cfg)
    env.reset()
    env.reset_changable_parameters(torch.as_tensor(p[:, 0]), torch.as_tensor(p[:, 1]), torch.as_tensor(p[:, 2]))
    res = staircase(env, policy, K, actor=actor, steps=max_step, resample_params=False, setpoints=setpoints)
    return res, p


def parameter_grid(a1, a2, Kp):
    """Cartesian product of the three ensemble-parameter axes -> [n, 3] (for robust_sweep)."""
    g = np.stack(np.meshgrid(np.asarray(a1, float), np.asarray(a2, float), np.asarray(Kp, float), indexing="ij"), -1)
    return g.reshape(-1, 3)
