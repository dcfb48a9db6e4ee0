"""gym-style drop-in envs: the reference's env ids, constructor kwargs, attributes and test API, executed by the
CUDA kernels (N = 1 per object by default, ``num_envs`` > 1 gives the batched form of the same object).

Mirrors (interface only -- the arithmetic lives in csrc/):
  gym_control/__init__.py:3-142          the 7 registered ids and their kwargs          -> REGISTRY / make()
  gym_control/envs/nonlinear_watertank.py NonLinearWaterTankChangingParamUniformGoal{,Integrator,Stacking}
  gym_control/envs/ph.py                  PH1DChangingParamUniformGoal{,Integrator,Integrator_NoBound}

N = 1 is launch-latency bound (one kernel + one small D2H copy per step); it exists so that train.py-style code
and the plot scripts' test API (set_state / set_r / set_params / get_linear_action ...) run unmodified.  Throughput
lives in pime_b200.vec (millions of envs per launch).

If the real ``gym`` package is importable the classes derive from gym.Env and are registered with it; otherwise a
minimal built-in Env / Box is used (gym==0.18.0 is not installed in the build image).
"""
from __future__ import annotations

import copy
from typing import Optional

import numpy as np
import torch

from . import _lib as L
from .vec import PHVec, WaterTankVec

try:  # pragma: no cover - gym is absent in the build image
    import gym as _gym
    _EnvBase = _gym.Env
    from gym.spaces import Box
except Exception:  # noqa: BLE001
    _gym = None

    class _EnvBase:  # minimal gym.Env surface used by elegantrl/env.py:194-245
        metadata = {"render.modes": ["human"]}
        reward_range = (-float("inf"), float("inf"))
        spec = None

        @property
        def unwrapped(self):
            return self

        def close(self):
            pass

    class Box:
        def __init__(self, low, high, shape=None, dtype=np.float32):
            low, high = np.asarray(low, dtype=dtype), np.asarray(high, dtype=dtype)
            self.shape = tuple(low.shape if shape is None else shape)
            self.low, self.high, self.dtype = np.broadcast_to(low, self.shape).copy(), np.broadcast_to(high, self.shape).copy(), np.dtype(dtype)

        def sample(self):
            return np.random.uniform(np.maximum(self.low, -1e6), np.minimum(self.high, 1e6)).astype(self.dtype)


class EnvSpec:
    def __init__(self, id, max_episode_steps=None, reward_threshold=None):
        self.id, self.max_episode_steps, self.reward_threshold = id, max_episode_steps, reward_threshold


def _f(x):
    return float(np.asarray(x, dtype=np.float64).reshape(-1)[0])


def _mirror(name):
    """Host-side view of one per-env device array: read -> python scalar (num_envs = 1) or numpy array; write -> broadcast."""
    def get(self):
        return self._scalar(getattr(self.vec, name))

    def put(self, v):
        t = getattr(self.vec, name)
        t.copy_(torch.as_tensor(v, dtype=t.dtype, device=t.device).expand_as(t))
    return property(get, put)


class _DeviceEnv(_EnvBase):
    """Shared plumbing: a *Vec object of num_envs envs plus host-side mirrors of the reference attributes."""

    n_integrator = 0

    def _obs_out(self, obs: torch.Tensor):
        o = obs.detach().cpu().numpy().astype(np.float64)
        return o[:, 0].copy() if self.num_envs == 1 else o.T.copy()

    def _scalar(self, t: torch.Tensor):
        v = t.detach().cpu().numpy()
        return v[0].item() if self.num_envs == 1 else v.copy()

    def _last(self, name):
        t = getattr(self.vec, name)
        if t is None:
            return None
        v = self._scalar(t)
        if self.num_envs == 1:
            return None if np.isnan(v) else v
        return v

    def seed(self, seed=None):
        """gym seeding API.  The device streams are Philox keyed by (seed, env id, tick); None keeps the current seed."""
        if seed is not None:
            self.vec.seed = int(seed)
        return [self.vec.seed]

    def set_reset_all(self, if_reset_all):
        self.if_reset_all = bool(if_reset_all)

    def __deepcopy__(self, memo):
        # utils/test.py:1058-1059 and utils/robust_test.py:5 deep-copy the env; device tensors are cloned.
        cls = self.__class__
        new = cls.__new__(cls)
        memo[id(self)] = new
        for k, v in self.__dict__.items():
            if k == "vec":
                continue
            setattr(new, k, copy.deepcopy(v, memo))
        new.vec = self._clone_vec()
        return new


# ====================================================================================================== water tank
class NonLinearWaterTankChangingParamUniformGoal(_DeviceEnv):
    """Reference nonlinear_watertank.py:942-1053 (obs [h1,h2,r]); base of the Integrator / Stacking variants."""

    _obs_mode = "goal"
    dim = 2

    def __init__(self, a1=(1, 2), a2=(1, 2), A1=2, A2=2, Kp=(1, 2), G=9.8, z1=1, z2=0.1, max_step=500, noise_scale=0.01,
                 gamma=0.99, seed=None, r=9.0, N=100, overflow_cost=-10, n_discrete=1, sample_t=0.02, reward_type="distance",
                 controller_type="P", distance_threshold=0.05, linearize_r=9.0, reset_from_last_state=True,
                 P_control_K=np.array([0.0, 0.4]), P_control_L=np.array([-0.4]), P_max_action=10.0, num_stack=0,
                 num_envs=1, device="cuda", dtype=torch.float64):
        if controller_type != "P":
            raise NotImplementedError("only controller_type='P' (the registered configuration) is implemented")
        self.num_envs = int(num_envs)
        self._dtype = dtype   # float64 = the reference's arithmetic (default); float32 = the throughput kernels
        self.a1_range, self.a2_range, self.Kp_range = list(a1), list(a2), list(Kp)
        self.A1, self.A2, self.G, self.z1, self.z2 = A1, A2, G, z1, z2
        self.max_step, self.noise_scale, self.gamma = max_step, noise_scale, gamma
        self.n_discrete, self.sample_t, self.delta_t = n_discrete, sample_t, sample_t / n_discrete
        self.reward_type, self.distance_threshold = reward_type, distance_threshold
        self.P_max_action = P_max_action
        self.K, self.L = np.asarray(P_control_K, dtype=np.float64), None
        self.num_stack = int(num_stack)
        self.if_reset_all = True
        self.reset_from_last_state = bool(reset_from_last_state)   # nonlinear_watertank.py:152, :904-910
        self.m = {"goal": 3, "integrator": 3, "stacking": 3 * self.num_stack}[self._obs_mode]
        self.n = 1
        self._device = device
        self._make_vec(0 if seed is None else int(seed))
        S = self.vec.state_dim
        low, high = np.zeros(S), np.full(S, np.inf)
        if self._obs_mode == "integrator":
            low[-1], high[-1] = -self.integral_max, self.integral_max
        self.observation_space = Box(low=low, high=high, dtype=np.float32)
        self.action_space = Box(low=-np.ones(1), high=np.ones(1), dtype=np.float32)
        self._reset_done = False

    def _cfg_kwargs(self):
        kw = dict(A1=self.A1, A2=self.A2, G=self.G, sample_t=self.sample_t, n_discrete=self.n_discrete, max_step=self.max_step,
                  P_max_action=self.P_max_action, reward_type=self.reward_type, z1=self.z1,
                  distance_threshold=self.distance_threshold, noise_scale=self.noise_scale,
                  a1_lo=self.a1_range[0], a1_hi=self.a1_range[1], a2_lo=self.a2_range[0], a2_hi=self.a2_range[1],
                  Kp_lo=self.Kp_range[0], Kp_hi=self.Kp_range[1])
        if self._obs_mode == "integrator":
            kw.update(integral_max=self.integral_max, integral_punish=self.integral_punish)
        return kw

    def _make_vec(self, seed):
        self.vec = WaterTankVec(self.num_envs, dtype=self._dtype, device=self._device, obs_mode=self._obs_mode,
                                num_stack=self.num_stack, seed=seed, reset_from_last_state=self.reset_from_last_state,
                                **self._cfg_kwargs())

    def _clone_vec(self):
        v = WaterTankVec(self.num_envs, dtype=self._dtype, device=self._device, obs_mode=self._obs_mode,
                         num_stack=self.num_stack, seed=self.vec.seed, env_offset=self.vec.env_offset,
                         reset_from_last_state=self.reset_from_last_state, **self._cfg_kwargs())
        for k in ("h1", "h2", "r", "I", "a1", "a2", "Kp", "t", "episode", "ep_return") + (
                ("last_h1", "last_h2") if self.reset_from_last_state else ()):
            getattr(v, k).copy_(getattr(self.vec, k))
        if v.frames is not None:
            v.frames.copy_(self.vec.frames)
        v.tick = self.vec.tick
        return v

    # ---- gym API
    def reset(self):
        self._reset_done = True
        return self._obs_out(self.vec.reset(resample_params=self.if_reset_all))

    def reset_all(self):
        self._reset_done = True
        return self._obs_out(self.vec.reset(resample_params=True))

    def reset_r(self):
        self._reset_done = True
        return self._obs_out(self.vec.reset(resample_params=False))

    def step(self, action):
        assert self._reset_done, "Please reset the env first"
        a = torch.as_tensor(np.asarray(action, dtype=np.float64).reshape(-1), device=self.vec.device)
        if a.numel() == 1 and self.num_envs > 1:
            a = a.expand(self.num_envs).contiguous()
        obs, rew, done = self.vec.step(a)
        if self.num_envs == 1:
            return self._obs_out(obs), float(rew[0]), bool(done[0]), {}
        return self._obs_out(obs), rew.cpu().numpy(), done.cpu().numpy().astype(bool), {}

    def _get_observe(self):
        assert self._reset_done, "Please reset the env first"
        return self._obs_out(self.vec.observe())

    # ---- ensemble API (nonlinear_watertank.py:890-900)
    def sample_parameters(self):
        return (np.random.uniform(*self.a1_range), np.random.uniform(*self.a2_range), np.random.uniform(*self.Kp_range))

    def get_changable_parameters(self):
        return self._scalar(self.vec.a1), self._scalar(self.vec.a2), self._scalar(self.vec.Kp)

    def reset_changable_parameters(self, a1, a2, Kp):
        self.vec.reset_changable_parameters(a1, a2, Kp)

    # ---- test / inspection API (nonlinear_watertank.py:205-212, :755-759)
    def set_state(self, h1, h2):
        """nonlinear_watertank.py:205-208.  The stacking variant inherits it unchanged: the frame history is NOT touched
        (frames change only in reset() and step(), :1145-1146,:1183-1184), so the returned observation is the old history."""
        self._reset_done = True
        self.vec.set_state(h1, h2)
        return self._get_observe()

    def set_r(self, r):
        self.vec.set_r(r)
        return self._get_observe()

    def get_P_action(self, state):
        """clip(-state[:m+n_int] . K, -1, 1) on the device (nonlinear_watertank.py:755-759)."""
        s = np.asarray(state, dtype=np.float64)
        S = self.K.shape[0]
        obs = torch.as_tensor(s.reshape(-1, s.shape[-1])[:, :S].T.copy(), device=self.vec.device)
        n = obs.shape[1]
        out = torch.empty(n, dtype=torch.float64, device=self.vec.device)
        import ctypes as C
        L.check(L.lib().pime_prior_action_f64(C.c_int64(n), C.c_int32(S), L.ptr(obs.contiguous()),
                                              self.K.ctypes.data_as(C.POINTER(C.c_double)), C.c_int(1), L.ptr(out), L.stream_ptr()))
        return out.cpu().numpy()

    get_linear_action = get_P_action

    def close(self):
        self._reset_done = False

    # host mirrors of the reference attributes; assignable like the plain attributes they mirror (utils/robust_test.py:12-37
    # writes test_env.a1 / a2 / Kp / max_step / if_reset_all directly)
    h1, h2, r = _mirror("h1"), _mirror("h2"), _mirror("r")
    a1, a2, Kp = _mirror("a1"), _mirror("a2"), _mirror("Kp")

    @property
    def max_step(self):
        return self._max_step

    @max_step.setter
    def max_step(self, v):
        self._max_step = int(v)
        if "vec" in self.__dict__:
            self.vec.cfg.max_step = int(v)

    state = property(lambda self: self._get_observe())
    _episode_steps = property(lambda self: self._scalar(self.vec.t))

    last_h1 = property(lambda self: self._last("last_h1"))   # None until the first episode ends (:185-186)
    last_h2 = property(lambda self: self._last("last_h2"))


class NonLinearWaterTankChangingParamUniformGoalIntegrator(NonLinearWaterTankChangingParamUniformGoal):
    """Reference nonlinear_watertank.py:828-939 (obs [h1,h2,r,I])."""

    _obs_mode = "integrator"
    n_integrator = 1
    integral_max = 25.0
    integral_punish = 0.0

    @property
    def integrator(self):
        return self._scalar(self.vec.I)

    @integrator.setter
    def integrator(self, v):
        self.vec.I.copy_(torch.as_tensor(v, dtype=torch.float64, device=self.vec.device).expand_as(self.vec.I))


class NonLinearWaterTankChangingParamUniformGoalStacking(NonLinearWaterTankChangingParamUniformGoal):
    """Reference nonlinear_watertank.py:1056-1208 (obs = last num_stack frames of [h1,h2,r], oldest first)."""

    _obs_mode = "stacking"

    def __init__(self, *args, num_stack=4, **kw):
        super().__init__(*args, num_stack=num_stack, **kw)


# ====================================================================================================== pH
class PH1DChangingParamUniformGoalIntegrator(_DeviceEnv):
    """Reference ph.py:350-445 (obs [y, r, I], clipped integrator)."""

    _integrator = "integrator"
    dim = 1
    n_integrator = 1
    integral_max = 25.0
    integral_punish = 0.0

    def __init__(self, qww_V=(0.005, 0.015), qc_V=(0.0015, 0.0025), kw=1e-14, kchem=5.6e-10, ka=0.5e-5, MNaOH=0.01, MHA=0.005,
                 MNH3=0.01, MHCl=None, r=7.0, n_discrete=200, sample_t=20, reset_from_last_state=False, reward_type="distance",
                 distance_threshold=0.05, P_control_K=np.array([1, 1]), P_control_L=np.array([-0.4]), action_punishment=0.0,
                 action_change_punishment=0.0, max_episode_steps=200, seed=None, time_limit=None, num_envs=1, device="cuda",
                 dtype=torch.float64):
        if action_change_punishment:
            raise NotImplementedError("action_change_punishment != 0 is not implemented (0 at every registered config)")
        self.num_envs = int(num_envs)
        self._dtype = dtype
        MHCl = np.arange(0.0, 0.2, step=0.00001) if MHCl is None else np.asarray(MHCl, dtype=np.float64)
        step = float(MHCl[1] - MHCl[0])
        if not np.array_equal(MHCl, np.arange(MHCl.shape[0]) * MHCl[1]):
            raise NotImplementedError("MHCl must be a uniform grid starting at 0 (np.arange(0, stop, step))")
        if step != 1e-5:   # the kernels' table index is rint(C x 1e5), the reference's argwhere only on this grid
            raise NotImplementedError("MHCl must have the step 1e-5 of every registered config")
        self.MHCl = MHCl
        self.qww_Vrange, self.qc_Vrange = list(qww_V), list(qc_V)
        self.sample_t, self.n_discrete, self.delta_t = sample_t, n_discrete, sample_t / n_discrete
        self.kw, self.kchem, self.ka, self.MNaOH, self.MHA, self.MNH3 = kw, kchem, ka, MNaOH, MHA, MNH3
        self.reward_type, self.distance_threshold = reward_type, distance_threshold
        self.max_episode_steps = max_episode_steps
        # gym's TimeLimit wrapper (registered max_episode_steps=50) is folded into the kernel's done flag
        self._max_episode_steps = time_limit if time_limit is not None else max_episode_steps
        self.K, self.L = np.asarray(P_control_K, dtype=np.float64), P_control_L
        self.action_punishment, self.action_change_punishment = action_punishment, action_change_punishment
        self.low, self.high, self.min_action, self.max_action = 0.0, 1.5, -1, 1
        self.if_reset_all = True
        self.reset_from_last_state = bool(reset_from_last_state)   # ph.py:101-102, :417-420
        self.m = 3 if self._integrator != "none" else 2
        self.n = 1
        self._device = device
        self._cfg = dict(reward_type=reward_type, max_episode_steps=int(self._max_episode_steps), table_len=int(MHCl.shape[0]),
                         mhcl_step=step, sample_t=float(sample_t), distance_threshold=distance_threshold,
                         integral_max=self.integral_max, integral_punish=self.integral_punish, action_punishment=action_punishment,
                         kw=kw, kchem=kchem, ka=ka, MNaOH=MNaOH, MHA=MHA, MNH3=MNH3, qww_lo=self.qww_Vrange[0],
                         qww_hi=self.qww_Vrange[1], qc_lo=self.qc_Vrange[0], qc_hi=self.qc_Vrange[1])
        self.vec = PHVec(self.num_envs, dtype=dtype, device=device, integrator=self._integrator,
                         seed=0 if seed is None else int(seed), reset_from_last_state=self.reset_from_last_state, **self._cfg)
        self.observation_space = Box(low=-np.full(self.m, np.inf), high=np.full(self.m, np.inf), dtype=np.float32)
        self.action_space = Box(low=-np.ones(1), high=np.ones(1), dtype=np.float32)
        self._reset_done = False

    def _clone_vec(self):
        v = PHVec(self.num_envs, dtype=self._dtype, device=self._device, integrator=self._integrator, seed=self.vec.seed,
                  env_offset=self.vec.env_offset, reset_from_last_state=self.reset_from_last_state, **self._cfg)
        for k in ("x", "y", "r", "I", "A", "B", "C", "qww_V", "qc_V", "t", "episode", "ep_return") + (
                ("last_x",) if self.reset_from_last_state else ()):
            getattr(v, k).copy_(getattr(self.vec, k))
        v.tick = self.vec.tick
        return v

    @property
    def pH(self):
        """The titration table (ph.py:72-84), built on the device."""
        return self.vec.table.cpu().numpy()

    def reset(self):
        self._reset_done = True
        obs = self.vec.reset(resample_params=self.if_reset_all)
        self.vec.check_status()
        return self._obs_out(obs)

    def reset_all(self):
        self._reset_done = True
        return self._obs_out(self.vec.reset(resample_params=True))

    def reset_r(self):
        self._reset_done = True
        return self._obs_out(self.vec.reset(resample_params=False))

    def step(self, action):
        assert self._reset_done, "Please reset the env first"
        a = torch.as_tensor(np.asarray(action, dtype=np.float64).reshape(-1), device=self.vec.device)
        if a.numel() == 1 and self.num_envs > 1:
            a = a.expand(self.num_envs).contiguous()
        obs, rew, done = self.vec.step(a, check=True)  # IndexError past the table, like ph.py:188
        if self.num_envs == 1:
            return self._obs_out(obs), float(rew[0]), bool(done[0]), {}
        return self._obs_out(obs), rew.cpu().numpy(), done.cpu().numpy().astype(bool), {}

    def _get_observe(self):
        return self._obs_out(self.vec.observe())

    def update_system(self):
        self.vec.update_system()

    def sample_parameters(self):
        return np.random.uniform(*self.qww_Vrange), np.random.uniform(*self.qc_Vrange)

    def get_changable_parameters(self):
        return self._scalar(self.vec.qww_V), self._scalar(self.vec.qc_V)

    def set_params(self, qww_V, qc_V):
        """ph.py:263-265 sets the parameters WITHOUT refreshing dsys (SURVEY T4); reproduced: call update_system()
        explicitly, as utils/test.py does not."""
        self.vec.set_params(qww_V, qc_V, update_system=False)

    def set_qww_V(self, qww_V):
        self.vec.qww_V.fill_(float(qww_V))

    def set_qc_V(self, qc_V):
        self.vec.qc_V.fill_(float(qc_V))

    def set_state(self, state):
        self._reset_done = True
        self.vec.x.copy_(torch.as_tensor(state, dtype=torch.float64, device=self.vec.device).expand_as(self.vec.x))
        idx = torch.round(self.vec.C * self.vec.x * 1e5).long()
        if int(idx.max()) >= self.vec.table.numel():
            raise IndexError("index out of the titration table (ph.py:188)")
        self.vec.y.copy_(self.vec.table[idx.clamp_min(0)])
        return self._get_observe()

    def set_r(self, r):
        self.vec.r.copy_(torch.as_tensor(r, dtype=torch.float64, device=self.vec.device).expand_as(self.vec.r))
        return self._get_observe()

    def get_linear_action(self, state=None):
        s = self._get_observe() if state is None else np.asarray(state, dtype=np.float64)
        return -s @ self.K.T

    y = property(lambda self: self._scalar(self.vec.y))
    r = property(lambda self: self._scalar(self.vec.r))
    state = property(lambda self: self._scalar(self.vec.x))
    last_state = property(lambda self: self._last("last_x"))   # None until an episode reaches the step limit (ph.py:102)
    qww_V = property(lambda self: self._scalar(self.vec.qww_V))
    qc_V = property(lambda self: self._scalar(self.vec.qc_V))
    _episode_steps = property(lambda self: self._scalar(self.vec.t))

    @property
    def integrator(self):
        return self._scalar(self.vec.I)

    @integrator.setter
    def integrator(self, v):
        self.vec.I.copy_(torch.as_tensor(v, dtype=torch.float64, device=self.vec.device).expand_as(self.vec.I))


class PH1DChangingParamUniformGoalIntegrator_NoBound(PH1DChangingParamUniformGoalIntegrator):
    """Reference ph.py:448-478 (integrator not clipped)."""
    _integrator = "nobound"


class PH1DChangingParamUniformGoal(PH1DChangingParamUniformGoalIntegrator):
    """Reference ph.py:479-485 (obs [y, r])."""
    _integrator = "none"
    n_integrator = 0


# ====================================================================================================== registry
def _wt_kwargs(P_control_K, **extra):
    kw = dict(reset_from_last_state=False, max_step=200, a1=[0.0015, 0.0024], a2=[0.0015, 0.0024], A1=1, A2=1, Kp=[0.07, 0.17],
              G=980, sample_t=2, n_discrete=20, controller_type="P", reward_type="square_distance", gamma=0.99,
              P_control_K=P_control_K)
    kw.update(extra)
    return kw


def _stack_K(k):
    K = np.zeros(3 * k)
    K[-3:] = [0.0, 0.4, -0.4]
    return K


_PH_KW = dict(P_control_K=np.array([-0.02, 0.02, 0.035]), P_control_L=None, reward_type="square_distance", max_episode_steps=50,
              MHCl=np.arange(0.0, 1, step=0.00001), time_limit=50)

# id -> (class, kwargs, TimeLimit steps)   (reference gym_control/__init__.py:3-142)
REGISTRY = {
    "PH1DChangingParamUniformGoalIntegrator-SqaureDistance-v35": (PH1DChangingParamUniformGoalIntegrator, _PH_KW, 50),
    "PH1DChangingParamUniformGoalIntegrator-SqaureDistance-NoIB-v35": (PH1DChangingParamUniformGoalIntegrator_NoBound, _PH_KW, 50),
    "NonLinearWaterTankChangingParamUniformGoal-SquareDistance-v2":
        (NonLinearWaterTankChangingParamUniformGoal, _wt_kwargs(np.array([0.0, 0.4, -0.4, 0.0])), None),
    "NonLinearWaterTankChangingParamUniformGoalIntegrator-SquareDistance-v2":
        (NonLinearWaterTankChangingParamUniformGoalIntegrator, _wt_kwargs(np.array([0.0, 0.4, -0.4, 0.0])), None),
    "NonLinearWaterTankChangingParamUniformGoalStacking4-SquareDistance-v2":
        (NonLinearWaterTankChangingParamUniformGoalStacking, _wt_kwargs(_stack_K(4), num_stack=4), None),
    "NonLinearWaterTankChangingParamUniformGoalStacking10-SquareDistance-v2":
        (NonLinearWaterTankChangingParamUniformGoalStacking, _wt_kwargs(_stack_K(10), num_stack=10), None),
    "NonLinearWaterTankChangingParamUniformGoalStacking1-SquareDistance-v2":
        (NonLinearWaterTankChangingParamUniformGoalStacking, _wt_kwargs(_stack_K(1), num_stack=1), None),
}


def make(env_id: str, **overrides):
    """gym.make(id, **overrides): kwargs merge like gym 0.18 (train.py:87-103 passes noise_scale / reward_type / r)."""
    cls, kwargs, limit = REGISTRY[env_id]
    kw = dict(kwargs)
    kw.update(overrides)
    if issubclass(cls, PH1DChangingParamUniformGoalIntegrator):
        for k in ("noise_scale",):
            kw.pop(k, None)
    env = cls(**kw)
    env.spec = EnvSpec(env_id, max_episode_steps=limit)
    return env
