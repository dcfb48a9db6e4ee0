"""Batched (vector) front end over the C ABI: millions of env instances, each with its own ensemble parameters.

State lives in torch CUDA tensors laid out structure-of-arrays (one tensor per field); every method is one
libpime_b200 call on the current CUDA stream.  torch is plumbing here (device memory, streams); all arithmetic
is in the CUDA library.
"""
from __future__ import annotations

import ctypes as C
import math
from typing import Optional

import numpy as np
import torch

from . import _lib as L

_SUFFIX = {torch.float32: "f32", torch.float64: "f64"}


def _fn(name: str, dtype):
    return getattr(L.lib(), f"{name}_{_SUFFIX[dtype]}")


def _require_cuda(device):
    if not torch.cuda.is_available():
        raise L.PimeError("no CUDA device: pime_b200 has no CPU fallback (the plants run only as sm_100a kernels)")
    return torch.device(device)


# ------------------------------------------------------------------------------------------------------ actor pack
class ActorPack:
    """Device image of one actor / critic: fp32 vectors + fp16 weight tiles in tcgen05 operand layout.

    ``kind``: 'plain' (ActorResidualPPO, net_residual.py:6-66), 'modular' (ActorResidualIntegratorModularPPO,
    :138-205) or 'critic' (CriticAdv, net.py:274-277).  ``update(state_dict)`` re-packs after a learner step.
    ``precision``: 'tc' (default) = throughput mode, |a_avg - fp32 torch| <= 4e-3; 'fp32' = fidelity mode, <= 2e-5.
    """

    KEYS = {
        "modular": ["other_net.0.weight", "other_net.0.bias", "other_net.2.weight", "other_net.2.bias",
                    "integrator_net.0.weight", "integrator_net.0.bias", "integrator_net.2.weight", "integrator_net.2.bias",
                    "net.0.weight", "net.0.bias", "net.2.weight", "net.2.bias"],
        "plain": ["net.0.weight", "net.0.bias", "net.2.weight", "net.2.bias", "net.4.weight", "net.4.bias",
                  "net.6.weight", "net.6.bias"],
    }
    KEYS["critic"] = KEYS["plain"]
    KIND = {"plain": L.ACTOR_PLAIN, "modular": L.ACTOR_MODULAR, "critic": L.CRITIC_ADV}

    PRECISION = {"tc": L.PRECISION_TC, "fp32": L.PRECISION_FP32}

    def __init__(self, kind: str, state_dim: int, mid_dim: int, integrator_dim: int = 0, device="cuda", precision="tc"):
        self.kind = kind
        self.device = _require_cuda(device)
        self.cfg = L.ActorConfig(kind=self.KIND[kind], state_dim=state_dim, mid_dim=mid_dim,
                                 integrator_dim=integrator_dim if kind == "modular" else 0, precision=self.PRECISION[precision])
        self.param_count = int(L.lib().pime_actor_param_count(C.byref(self.cfg)))
        nbytes = int(L.lib().pime_actor_pack_bytes(C.byref(self.cfg)))
        if self.param_count < 0 or nbytes < 0:
            raise ValueError(f"unsupported actor dimensions: kind={kind} S={state_dim} H={mid_dim} D={integrator_dim}")
        self.pack = torch.zeros(nbytes, dtype=torch.uint8, device=self.device)
        self.flat = torch.zeros(self.param_count, dtype=torch.float32, device=self.device)
        self.a_std_log = -0.5

    def update(self, state_dict) -> "ActorPack":
        parts = []
        for k in self.KEYS[self.kind]:
            v = state_dict[k]
            v = v if isinstance(v, torch.Tensor) else torch.as_tensor(np.asarray(v))
            parts.append(v.detach().to(device=self.device, dtype=torch.float32).reshape(-1))
        flat = torch.cat(parts)
        if flat.numel() != self.param_count:
            raise ValueError(f"state_dict has {flat.numel()} parameters, the kernel image expects {self.param_count}")
        self.flat.copy_(flat)
        if "a_std_log" in state_dict:
            v = state_dict["a_std_log"]
            self.a_std_log = float(v.reshape(-1)[0]) if hasattr(v, "reshape") else float(v)
        return self.update_from_flat()

    def set_precision(self, precision: str) -> "ActorPack":
        """'tc': tcgen05 throughput engine (fp16 hidden operands); 'fp32': fidelity mode (fp32 CUDA cores, tanhf).  The packed
        image holds both forms, so switching needs no re-pack."""
        self.cfg.precision = self.PRECISION[precision]
        return self

    def update_from_flat(self) -> "ActorPack":
        """Re-pack from ``self.flat`` (fp32 parameters in state_dict order, already on the device)."""
        L.check(L.lib().pime_actor_pack(C.byref(self.cfg), L.ptr(self.flat), L.ptr(self.pack), L.stream_ptr()))
        return self

    def forward(self, obs: torch.Tensor) -> torch.Tensor:
        """a_avg = net(obs) for row-major obs [n, S] (float32, CUDA)."""
        obs = obs.to(device=self.device, dtype=torch.float32).contiguous()
        assert obs.dim() == 2 and obs.shape[1] == self.cfg.state_dim
        out = torch.empty(obs.shape[0], dtype=torch.float32, device=self.device)
        L.check(L.lib().pime_actor_forward(C.byref(self.cfg), L.ptr(self.pack), C.c_int64(obs.shape[0]), L.ptr(obs),
                                           L.ptr(out), L.stream_ptr()))
        return out


# ------------------------------------------------------------------------------------------------------ shared rollout glue
def _rollout_args(env, T, actor, priorK, deterministic, auto_reset, reward_scale, gamma, eps, pnoise, replay, want_actions,
                  stats, keep, a_std_log=None, keep_params=False):
    n, S = env.n, env.state_dim
    a = L.RolloutArgs()
    a.a_std_log = -0.5 if a_std_log is None else float(a_std_log)   # net_residual.py:162 initial value
    if actor is not None:
        a.actor = C.pointer(actor.cfg)
        a.actor_pack = L.ptr(actor.pack)
        if a_std_log is None:
            a.a_std_log = float(actor.a_std_log)
    pk = np.ascontiguousarray(np.asarray(priorK, dtype=np.float64).reshape(-1))
    assert pk.shape[0] == S, f"priorK must have {S} entries"
    keep.append(pk)
    a.priorK_host = pk.ctypes.data_as(C.POINTER(C.c_double))
    a.deterministic = int(deterministic)
    a.T = int(T)
    a.auto_reset = int(auto_reset)
    a.reward_scale, a.gamma = float(reward_scale), float(gamma)
    a.seed, a.env_offset, a.tick0 = int(env.seed), int(env.env_offset), int(env.tick) & 0xFFFFFFFF
    out = {}
    if eps is not None:
        assert eps.shape == (T, n) and eps.dtype == torch.float32 and eps.is_cuda
        a.eps = L.ptr(eps)
    if pnoise is not None:
        p1, p2 = pnoise
        assert p1.shape == (T, n) and p1.dtype == env.dtype and p2.shape == (T, n)
        a.pnoise1, a.pnoise2 = L.ptr(p1), L.ptr(p2)
    if replay is True:
        replay = (torch.empty((T, n, S), dtype=torch.float32, device=env.device),
                  torch.empty((T, n, 4), dtype=torch.float32, device=env.device))
    if replay:
        bs, bo = replay
        assert bs.shape == (T, n, S) and bo.shape == (T, n, 4) and bs.dtype == torch.float32 and bo.dtype == torch.float32
        a.buf_state, a.buf_other = L.ptr(bs), L.ptr(bo)
        out["buf_state"], out["buf_other"] = bs, bo
    if want_actions:
        out["env_action"] = torch.empty((T, n), dtype=env.dtype, device=env.device)
        a.env_action = L.ptr(out["env_action"])
    if stats is None:
        stats = torch.zeros(8, dtype=torch.float64, device=env.device)
    out["stats"] = stats
    a.stats = L.ptr(stats)
    a.status = L.ptr(env.status)   # device fault flag: accumulated (atomicMin) until check_status() reads and clears it
    a.keep_params = int(keep_params)
    return a, out


def _schedule(env, setpoints, segment_steps, resample_params, metrics, keep):
    """pime_schedule of K = len(setpoints) segments of segment_steps steps; metrics: True (allocated [4, K, n] float64),
    a tensor of that shape (or wider in n), or None."""
    sp = np.ascontiguousarray(np.asarray(setpoints, dtype=np.float64).reshape(-1))
    keep.append(sp)
    K = sp.shape[0]
    if metrics is True:
        metrics = torch.empty((4, K, env.n), dtype=torch.float64, device=env.device)
    if metrics is not None:
        assert metrics.shape == (4, K, env.n) and metrics.dtype == torch.float64 and metrics.is_cuda
    sc = L.Schedule(num_segments=K, segment_steps=int(segment_steps), resample_params=int(bool(resample_params)),
                    setpoints_host=sp.ctypes.data_as(C.POINTER(C.c_double)), metrics=L.ptr(metrics))
    return sc, metrics


class _VecBase:
    def _alloc(self, names, n, f64=()):
        for k in names:
            setattr(self, k, torch.zeros(n, dtype=torch.float64 if k in f64 else self.dtype, device=self.device))
        self.t = torch.full((n,), -1, dtype=torch.int32, device=self.device)   # -1: "Please reset the env first"
        self.episode = torch.zeros(n, dtype=torch.int32, device=self.device)
        self.ep_return = torch.zeros(n, dtype=self.dtype, device=self.device)
        self.status = torch.zeros(1, dtype=torch.int32, device=self.device)
        self.tick = 0

    def check_status(self):
        code = int(self.status.item())
        if code != 0:
            self.status.zero_()
            L.check(code)

    def episode_stats(self, stats: Optional[torch.Tensor] = None) -> torch.Tensor:
        """(sum, sum of squares, count) of ep_return accumulated into a double[8] tensor (run.py:593-597)."""
        if stats is None:
            stats = torch.zeros(8, dtype=torch.float64, device=self.device)
        L.check(_fn("pime_reduce_episode_stats", self.dtype)(C.c_int64(self.n), L.ptr(self.ep_return), L.ptr(stats), L.stream_ptr()))
        return stats


# ------------------------------------------------------------------------------------------------------ water tank
class WaterTankVec(_VecBase):
    """n two-tank plants (reference gym_control/envs/nonlinear_watertank.py), one ensemble member each."""

    OBS = {"goal": L.WT_OBS_GOAL, "integrator": L.WT_OBS_INTEGRATOR, "stacking": L.WT_OBS_STACKING}

    def __init__(self, n: int, dtype=torch.float32, device="cuda", obs_mode="integrator", num_stack=0, seed=0, env_offset=0,
                 reset_from_last_state=False, **cfg):
        self.device = _require_cuda(device)
        self.n, self.dtype, self.seed, self.env_offset = int(n), dtype, int(seed), int(env_offset)
        self.cfg = L.wt_config(obs_mode=self.OBS[obs_mode], num_stack=int(num_stack),
                               reset_from_last_state=int(bool(reset_from_last_state)), **cfg)
        self.obs_mode = obs_mode
        self.num_stack = int(num_stack)
        self.state_dim = {"goal": 3, "integrator": 4}.get(obs_mode, 3 * self.num_stack)
        self._alloc(["h1", "h2", "r", "I", "a1", "a2", "Kp"], self.n)
        self.frames = (torch.zeros((3 * self.num_stack, self.n), dtype=dtype, device=self.device)
                       if obs_mode == "stacking" else None)
        # levels at the last `done` (nonlinear_watertank.py:185-186, :819-821); NaN = None
        self.last_h1 = self.last_h2 = None
        if reset_from_last_state:
            self.last_h1 = torch.full((self.n,), float("nan"), dtype=dtype, device=self.device)
            self.last_h2 = torch.full((self.n,), float("nan"), dtype=dtype, device=self.device)
        self._st = L.WtState(h1=L.ptr(self.h1), h2=L.ptr(self.h2), r=L.ptr(self.r), I=L.ptr(self.I), a1=L.ptr(self.a1),
                             a2=L.ptr(self.a2), Kp=L.ptr(self.Kp), t=L.ptr(self.t), episode=L.ptr(self.episode),
                             ep_return=L.ptr(self.ep_return), frames=L.ptr(self.frames), last_h1=L.ptr(self.last_h1),
                             last_h2=L.ptr(self.last_h2))

    def _obs_buf(self):
        return torch.empty((self.state_dim, self.n), dtype=self.dtype, device=self.device)

    def reset(self, mask: Optional[torch.Tensor] = None, resample_params: bool = True) -> torch.Tensor:
        """reset() of every (masked) env -> observation [S, n] (component-major)."""
        obs = self._obs_buf()
        if mask is not None:
            mask = mask.to(device=self.device, dtype=torch.uint8).contiguous()
            obs.copy_(self.observe())
        L.check(_fn("pime_wt_reset", self.dtype)(C.byref(self.cfg), C.c_int64(self.n), C.byref(self._st), C.c_uint64(self.seed),
                                                 C.c_uint64(self.env_offset), C.c_int(int(resample_params)), L.ptr(mask),
                                                 L.ptr(obs), L.stream_ptr()))
        return obs

    def observe(self) -> torch.Tensor:
        if self.obs_mode == "stacking":
            return self.frames.clone()
        rows = [self.h1, self.h2, self.r] + ([self.I] if self.obs_mode == "integrator" else [])
        return torch.stack(rows, 0)

    def step(self, action: torch.Tensor, noise1: Optional[torch.Tensor] = None, noise2: Optional[torch.Tensor] = None):
        """env.step for all n envs -> (obs [S,n], reward [n], done [n] uint8)."""
        action = action.to(device=self.device, dtype=self.dtype).contiguous().reshape(-1)
        assert action.numel() == self.n
        obs = self._obs_buf()
        reward = torch.empty(self.n, dtype=self.dtype, device=self.device)
        done = torch.empty(self.n, dtype=torch.uint8, device=self.device)
        L.check(_fn("pime_wt_step", self.dtype)(C.byref(self.cfg), C.c_int64(self.n), C.byref(self._st), L.ptr(action),
                                                L.ptr(noise1), L.ptr(noise2), C.c_uint64(self.seed), C.c_uint64(self.env_offset),
                                                C.c_uint32(self.tick & 0xFFFFFFFF), L.ptr(obs), L.ptr(reward), L.ptr(done),
                                                L.stream_ptr()))
        self.tick += 1
        return obs, reward, done

    def prior_action(self, obs: torch.Tensor, K, clip: bool = True) -> torch.Tensor:
        """get_P_action (nonlinear_watertank.py:755-759): clip(-obs . K, -1, 1)."""
        K = np.ascontiguousarray(np.asarray(K, np.float64).reshape(-1))
        out = torch.empty(self.n, dtype=self.dtype, device=self.device)
        obs = obs.contiguous()
        L.check(_fn("pime_prior_action", self.dtype)(C.c_int64(self.n), C.c_int32(K.shape[0]), L.ptr(obs),
                                                     K.ctypes.data_as(C.POINTER(C.c_double)), C.c_int(int(clip)), L.ptr(out),
                                                     L.stream_ptr()))
        return out

    def rollout(self, T: int, priorK, actor: Optional[ActorPack] = None, deterministic=False, auto_reset=False,
                reward_scale=1.0, gamma=0.99, eps=None, pnoise=None, replay=None, want_actions=False, stats=None,
                a_std_log=None, resample_params=True):
        """T fused steps (plant + prior + obs + actor) in one launch; see pime_wt_rollout_* in the header.
        eps=None draws the exploration noise in the kernel (Philox); pass a zero tensor for a noise-free policy.
        resample_params=False: the in-kernel auto-reset keeps (a1, a2, Kp) like reset_r() (if_reset_all=False)."""
        keep = []
        a, out = _rollout_args(self, T, actor, priorK, deterministic, auto_reset, reward_scale, gamma, eps, pnoise, replay,
                               want_actions, stats, keep, a_std_log, keep_params=not resample_params)
        L.check(_fn("pime_wt_rollout", self.dtype)(C.byref(self.cfg), C.c_int64(self.n), C.byref(self._st), C.byref(a),
                                                   L.stream_ptr()))
        self.tick += T
        return out

    def rollout_schedule(self, setpoints, segment_steps: int, priorK, actor: Optional[ActorPack] = None, deterministic=False,
                         reward_scale=1.0, gamma=0.99, eps=None, pnoise=None, replay=None, want_actions=False, stats=None,
                         a_std_log=None, resample_params=False, metrics=True):
        """The set-point staircase in one launch (pime_wt_rollout_schedule_*): T = K * segment_steps fused steps, segment k
        tracking setpoints[k] and beginning with reset(resample_params) -> set_state(levels before it) -> set_r(setpoints[k]).
        Returns rollout()'s dict plus metrics [4, K, n] float64 (ret, iae, final_err, overshoot per segment and env)."""
        keep = []
        sc, metrics = _schedule(self, setpoints, segment_steps, resample_params, metrics, keep)
        T = sc.num_segments * sc.segment_steps
        a, out = _rollout_args(self, T, actor, priorK, deterministic, False, reward_scale, gamma, eps, pnoise, replay,
                               want_actions, stats, keep, a_std_log)
        L.check(_fn("pime_wt_rollout_schedule", self.dtype)(C.byref(self.cfg), C.c_int64(self.n), C.byref(self._st), C.byref(a),
                                                            C.byref(sc), L.stream_ptr()))
        self.tick += T
        out["metrics"] = metrics
        return out

    def rollout_host(self, host_state: dict, T: int, priorK, actor: Optional[ActorPack] = None, deterministic=False,
                     ep_return_host: Optional[torch.Tensor] = None, **kw):
        """Host-buffer entry (fp32): host_state maps h1,h2,r,I,a1,a2,Kp (float32) and t, episode (int32) to HOST
        tensors (pinned for full-speed copies).  Copies them in, runs the fused rollout, copies ep_return (and the final
        h1,h2,r,I) back and synchronises -- every host<->device byte is inside this call."""
        assert self.dtype == torch.float32
        keep = []
        a, out = _rollout_args(self, T, actor, priorK, deterministic, kw.pop("auto_reset", False), kw.pop("reward_scale", 1.0),
                               kw.pop("gamma", 0.99), None, None, kw.pop("replay", None), False, kw.pop("stats", None), keep,
                               kw.pop("a_std_log", None), keep_params=not kw.pop("resample_params", True))
        assert not kw, f"unknown arguments {list(kw)}"
        hs = L.WtState(**{k: L.ptr(host_state.get(k)) for k in ("h1", "h2", "r", "I", "a1", "a2", "Kp", "t", "episode")})
        if ep_return_host is None:
            ep_return_host = torch.empty(self.n, dtype=torch.float32, pin_memory=True)
        L.check(L.lib().pime_wt_rollout_host_f32(C.byref(self.cfg), C.c_int64(self.n), C.byref(hs), C.byref(self._st), C.byref(a),
                                                 L.ptr(ep_return_host), L.stream_ptr()))
        self.tick += T
        out["ep_return_host"] = ep_return_host
        return out

    # ensemble API (nonlinear_watertank.py:896-900)
    def get_changable_parameters(self):
        return self.a1, self.a2, self.Kp

    def reset_changable_parameters(self, a1, a2, Kp):
        for dst, src in ((self.a1, a1), (self.a2, a2), (self.Kp, Kp)):
            dst.copy_(torch.as_tensor(src, dtype=self.dtype, device=self.device).expand_as(dst))

    def set_state(self, h1, h2):
        self.h1.copy_(torch.as_tensor(h1, dtype=self.dtype, device=self.device).expand_as(self.h1))
        self.h2.copy_(torch.as_tensor(h2, dtype=self.dtype, device=self.device).expand_as(self.h2))

    def set_r(self, r):
        self.r.copy_(torch.as_tensor(r, dtype=self.dtype, device=self.device).expand_as(self.r))


# ------------------------------------------------------------------------------------------------------ pH
_TABLES: dict = {}


def ph_table(cfg: L.PhConfig, device) -> tuple:
    """The titration table (ph.py:72-84) built once per device/config by the table kernel: (f64, f32) tensors."""
    key = (str(device), cfg.table_len, cfg.mhcl_step, cfg.kw, cfg.kchem, cfg.ka, cfg.MNaOH, cfg.MHA, cfg.MNH3)
    if key not in _TABLES:
        t64 = torch.empty(cfg.table_len, dtype=torch.float64, device=device)
        t32 = torch.empty(cfg.table_len, dtype=torch.float32, device=device)
        L.check(L.lib().pime_ph_table_build(C.byref(cfg), L.ptr(t64), L.ptr(t32), L.stream_ptr()))
        _TABLES[key] = (t64, t32)
    return _TABLES[key]


class PHVec(_VecBase):
    """n pH-neutralisation plants (reference gym_control/envs/ph.py), one (qww_V, qc_V) ensemble member each."""

    MODE = {"none": L.PH_NO_INTEGRATOR, "integrator": L.PH_INTEGRATOR, "nobound": L.PH_INTEGRATOR_NOBOUND}

    def __init__(self, n: int, dtype=torch.float32, device="cuda", integrator="integrator", seed=0, env_offset=0,
                 reset_from_last_state=False, **cfg):
        self.device = _require_cuda(device)
        self.n, self.dtype, self.seed, self.env_offset = int(n), dtype, int(seed), int(env_offset)
        self.cfg = L.ph_config(integrator_mode=self.MODE[integrator], reset_from_last_state=int(bool(reset_from_last_state)),
                               **cfg)
        self.state_dim = 2 if integrator == "none" else 3
        self.integrator = integrator
        # x, A, B (and last_x) are fp64 in both flavours: the titration index rint(C x 1e5) must not depend on the dtype
        self._alloc(["x", "y", "r", "I", "A", "B", "C", "qww_V", "qc_V"], self.n, f64=("x", "A", "B"))
        t64, t32 = ph_table(self.cfg, self.device)
        self.table = t64 if dtype == torch.float64 else t32
        # state at the last time-limit step (ph.py:102, :345-346); NaN = None
        self.last_x = (torch.full((self.n,), float("nan"), dtype=torch.float64, device=self.device) if reset_from_last_state else None)
        self._st = L.PhState(x=L.ptr(self.x), y=L.ptr(self.y), r=L.ptr(self.r), I=L.ptr(self.I), A=L.ptr(self.A),
                             B=L.ptr(self.B), C=L.ptr(self.C), qww_V=L.ptr(self.qww_V), qc_V=L.ptr(self.qc_V),
                             t=L.ptr(self.t), episode=L.ptr(self.episode), ep_return=L.ptr(self.ep_return),
                             last_x=L.ptr(self.last_x))

    def _obs_buf(self):
        return torch.empty((self.state_dim, self.n), dtype=self.dtype, device=self.device)

    def observe(self):
        rows = [self.y, self.r] + ([self.I] if self.integrator != "none" else [])
        return torch.stack(rows, 0)

    def reset(self, mask: Optional[torch.Tensor] = None, resample_params: bool = True) -> torch.Tensor:
        obs = self._obs_buf()
        if mask is not None:
            mask = mask.to(device=self.device, dtype=torch.uint8).contiguous()
            obs.copy_(self.observe())
        L.check(_fn("pime_ph_reset", self.dtype)(C.byref(self.cfg), L.ptr(self.table), C.c_int64(self.n), C.byref(self._st),
                                                 C.c_uint64(self.seed), C.c_uint64(self.env_offset),
                                                 C.c_int(int(resample_params)), L.ptr(mask), L.ptr(obs), L.ptr(self.status),
                                                 L.stream_ptr()))
        return obs

    def update_system(self):
        """update_system (ph.py:114-121) for every env from its (qww_V, qc_V)."""
        L.check(_fn("pime_ph_update_system", self.dtype)(C.byref(self.cfg), C.c_int64(self.n), C.byref(self._st), L.stream_ptr()))

    def step(self, action: torch.Tensor, check: bool = False):
        action = action.to(device=self.device, dtype=self.dtype).contiguous().reshape(-1)
        assert action.numel() == self.n
        obs = self._obs_buf()
        reward = torch.empty(self.n, dtype=self.dtype, device=self.device)
        done = torch.empty(self.n, dtype=torch.uint8, device=self.device)
        L.check(_fn("pime_ph_step", self.dtype)(C.byref(self.cfg), L.ptr(self.table), C.c_int64(self.n), C.byref(self._st),
                                                L.ptr(action), L.ptr(obs), L.ptr(reward), L.ptr(done), L.ptr(self.status),
                                                L.stream_ptr()))
        self.tick += 1
        if check:
            self.check_status()
        return obs, reward, done

    def prior_action(self, obs: torch.Tensor, K, clip: bool = False) -> torch.Tensor:
        K = np.ascontiguousarray(np.asarray(K, np.float64).reshape(-1))
        out = torch.empty(self.n, dtype=self.dtype, device=self.device)
        obs = obs.contiguous()
        L.check(_fn("pime_prior_action", self.dtype)(C.c_int64(self.n), C.c_int32(K.shape[0]), L.ptr(obs),
                                                     K.ctypes.data_as(C.POINTER(C.c_double)), C.c_int(int(clip)), L.ptr(out),
                                                     L.stream_ptr()))
        return out

    def rollout(self, T: int, priorK, actor: Optional[ActorPack] = None, deterministic=False, auto_reset=False,
                reward_scale=1.0, gamma=0.99, eps=None, replay=None, want_actions=False, stats=None, a_std_log=None,
                resample_params=True):
        keep = []
        a, out = _rollout_args(self, T, actor, priorK, deterministic, auto_reset, reward_scale, gamma, eps, None, replay,
                               want_actions, stats, keep, a_std_log, keep_params=not resample_params)
        L.check(_fn("pime_ph_rollout", self.dtype)(C.byref(self.cfg), L.ptr(self.table), C.c_int64(self.n), C.byref(self._st),
                                                   C.byref(a), L.stream_ptr()))
        self.tick += T
        return out

    def rollout_schedule(self, setpoints, segment_steps: int, priorK, actor: Optional[ActorPack] = None, deterministic=False,
                         reward_scale=1.0, gamma=0.99, eps=None, replay=None, want_actions=False, stats=None, a_std_log=None,
                         resample_params=False, metrics=True):
        """The set-point staircase in one launch (pime_ph_rollout_schedule_*): segment k begins with reset(resample_params),
        the state x before it restored (y looked up under the new C) and r = setpoints[k].  See WaterTankVec.rollout_schedule."""
        keep = []
        sc, metrics = _schedule(self, setpoints, segment_steps, resample_params, metrics, keep)
        T = sc.num_segments * sc.segment_steps
        a, out = _rollout_args(self, T, actor, priorK, deterministic, False, reward_scale, gamma, eps, None, replay,
                               want_actions, stats, keep, a_std_log)
        L.check(_fn("pime_ph_rollout_schedule", self.dtype)(C.byref(self.cfg), L.ptr(self.table), C.c_int64(self.n),
                                                            C.byref(self._st), C.byref(a), C.byref(sc), L.stream_ptr()))
        self.tick += T
        out["metrics"] = metrics
        return out

    HOST_FIELDS = ("x", "y", "r", "I", "A", "B", "C", "qww_V", "qc_V", "t", "episode")

    def rollout_host(self, host_state: dict, T: int, priorK, actor: Optional[ActorPack] = None, deterministic=False,
                     ep_return_host: Optional[torch.Tensor] = None, **kw):
        """Host-buffer entry (float flavour): host_state maps HOST_FIELDS to HOST tensors (x, A, B float64; y, r, I, C, qww_V,
        qc_V float32; t, episode int32; pinned for full-speed copies).  Copies them in, runs the fused rollout, copies
        ep_return and the final x, y, r, I back and synchronises -- every host<->device byte is inside this call."""
        assert self.dtype == torch.float32
        keep = []
        a, out = _rollout_args(self, T, actor, priorK, deterministic, kw.pop("auto_reset", False), kw.pop("reward_scale", 1.0),
                               kw.pop("gamma", 0.99), None, None, kw.pop("replay", None), False, kw.pop("stats", None), keep,
                               kw.pop("a_std_log", None), keep_params=not kw.pop("resample_params", True))
        assert not kw, f"unknown arguments {list(kw)}"
        hs = L.PhState(**{k: L.ptr(host_state.get(k)) for k in self.HOST_FIELDS})
        if ep_return_host is None:
            ep_return_host = torch.empty(self.n, dtype=torch.float32, pin_memory=True)
        L.check(L.lib().pime_ph_rollout_host_f32(C.byref(self.cfg), L.ptr(self.table), C.c_int64(self.n), C.byref(hs),
                                                 C.byref(self._st), C.byref(a), L.ptr(ep_return_host), L.stream_ptr()))
        self.tick += T
        out["ep_return_host"] = ep_return_host
        return out

    def get_changable_parameters(self):
        return self.qww_V, self.qc_V

    def set_params(self, qww_V, qc_V, update_system: bool = True):
        """set_params (ph.py:263-265).  The reference forgets to refresh dsys (SURVEY T4); here the discretised
        system is refreshed unless update_system=False is passed to mimic the stale behaviour."""
        self.qww_V.copy_(torch.as_tensor(qww_V, dtype=self.dtype, device=self.device).expand_as(self.qww_V))
        self.qc_V.copy_(torch.as_tensor(qc_V, dtype=self.dtype, device=self.device).expand_as(self.qc_V))
        if update_system:
            self.update_system()


def gae_scan(reward: torch.Tensor, mask: torch.Tensor, value: torch.Tensor, lambda_gae: float, stride: int = 1):
    """Per-env reverse scan of AgentPPO.compute_reward_gae (agent.py:685-708) on time-major [T, n] data.
    reward/mask may be strided views into buf_other (stride=4)."""
    T, n = value.shape
    r_sum = torch.empty((T, n), dtype=torch.float32, device=value.device)
    adv = torch.empty((T, n), dtype=torch.float32, device=value.device)
    L.check(L.lib().pime_gae_scan(C.c_int64(n), C.c_int32(T), C.c_void_p(reward.data_ptr()), C.c_void_p(mask.data_ptr()),
                                  C.c_int32(stride), L.ptr(value.contiguous()), C.c_float(lambda_gae), L.ptr(r_sum), L.ptr(adv),
                                  L.stream_ptr()))
    return r_sum, adv
