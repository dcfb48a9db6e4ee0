"""Agent / buffer / trainer surface of the reference's ElegantRL fork, driven by the CUDA library.

What train.py and the run_*_changing.sh scripts touch (SURVEY.md section 8b), with the same names, argument meaning and
state-dict keys, so that ``actor.pth`` / ``critic.pth`` files are interchangeable with the reference:

  elegantrl/net_residual.py:6-66,138-205      ActorResidualPPO, ActorResidualIntegratorModularPPO
  elegantrl/net.py:274-277 (+ ActorPPO)       CriticAdv, ActorPPO
  elegantrl/agent.py:536-708                  AgentPPO (select_action, explore_env, update_net, compute_reward_*)
  elegantrl/agent_residual.py:15-98           Residual mix-in, AgentResidualPPO, AgentResidualIntegratorModularPPO
  elegantrl/replay.py:238-379                 ReplayBuffer (on-policy part)
  elegantrl/env.py:10-72,194-245              PreprocessEnv
  elegantrl/run.py:14-225,478-619             Arguments, train_and_evaluate, Evaluator, get_episode_return
  utils/utils.py                              MODELS, IF_ONPOLICY

Where the work happens:
  * explore_env on a pime_b200 env (any ``num_envs``): ONE fused CUDA launch per episode batch
    (plant + prior + observation + tcgen05 actor + replay rows), the replay stays in HBM, time-major [T, n, .];
  * update_net: critic values of the whole buffer by the tcgen05 forward kernel, GAE / reward-to-go by the per-env
    scan kernel; the minibatch surrogate / SmoothL1 / Adam step is pime_ppo_step (csrc/learner.cu, two hand-written
    launches) whenever every parameter is trained; the frozen_* variants keep the torch autograd step;
  * torch.distributed (NCCL): replay stays sharded by env, gradients are averaged with one flat all-reduce per
    minibatch, the advantage normalisation uses global moments.
Foreign gym envs (anything without a ``vec``) run the reference's sequential loop through select_action.
"""
from __future__ import annotations

import math
import os
import time
from copy import deepcopy
from typing import Optional

import numpy as np
import torch
import torch.nn as nn

from . import vec as V


# ====================================================================================================== logger
from . import logger  # noqa: E402  (SB3-style module-level logger: the reference's elegantrl/logger.py is missing, SURVEY T1)


def get_latest_run_id(log_path: Optional[str] = None, log_name: str = "") -> int:
    """Greatest N among the directories ``{log_path}/{log_name}_N`` (elegantrl/utils.py:10-24)."""
    import glob
    best = 0
    for path in glob.glob(f"{log_path}/{log_name}_[0-9]*"):
        head, _, ext = os.path.basename(path).rpartition("_")
        if head == log_name and ext.isdigit():
            best = max(best, int(ext))
    return best


def configure_logger(verbose=0, tensorboard_log=None, tb_log_name="", reset_num_timesteps=True):
    """elegantrl/utils.py:26-47: outputs go to ``{tensorboard_log}/{tb_log_name}_{run id}`` as tensorboard events + csv
    (+ stdout when verbose >= 1).  The reference only writes files when tensorboard is importable; the csv is written here
    either way."""
    if tensorboard_log is not None:
        run = get_latest_run_id(tensorboard_log, tb_log_name)
        if not reset_num_timesteps:
            run -= 1
        save_path = os.path.join(tensorboard_log, f"{tb_log_name}_{run + 1}")
        logger.configure(save_path, (["stdout"] if verbose >= 1 else []) + ["tensorboard", "csv"])
    elif verbose == 0:
        logger.configure(format_strings=[""])
    else:
        logger.configure(format_strings=["stdout"])
    return logger


# ====================================================================================================== networks
def layer_norm(layer, std=1.0, bias_const=1e-6):
    """net.py:617-619."""
    torch.nn.init.orthogonal_(layer.weight, std)
    torch.nn.init.constant_(layer.bias, bias_const)


def _mlp(sizes, act):
    layers = []
    for i in range(len(sizes) - 1):
        layers.append(nn.Linear(sizes[i], sizes[i + 1]))
        if i < len(sizes) - 2:
            layers.append(act())
    return nn.Sequential(*layers)


class _GaussianHead:
    """get_action_noise / compute_logprob shared by the PPO actors (net_residual.py:51-66)."""

    def a_avg(self, state):
        raise NotImplementedError

    def get_action_noise(self, state):
        a_avg = self.a_avg(state)
        noise = torch.randn_like(a_avg)
        return a_avg + noise * self.a_std_log.exp(), noise

    def compute_logprob(self, state, action):
        delta = ((self.a_avg(state) - action) / self.a_std_log.exp()).pow(2) * 0.5
        return -(self.a_std_log + self.sqrt_2pi_log + delta).sum(1)


class ActorPPO(nn.Module, _GaussianHead):
    """Plain PPO baseline arm (reference elegantrl/net.py ActorPPO): action = tanh(net(s)), no prior."""
    kind = "plain"

    def __init__(self, mid_dim, state_dim, action_dim, if_use_dn=False):
        super().__init__()
        assert not if_use_dn and action_dim == 1, "only the configuration the scripts use is implemented"
        self.net = _mlp([state_dim, mid_dim, mid_dim, mid_dim, action_dim], nn.Tanh)
        self.a_std_log = nn.Parameter(torch.zeros((1, action_dim)) - 0.5, requires_grad=True)
        self.sqrt_2pi_log = np.log(np.sqrt(2 * np.pi))
        layer_norm(self.net[-1], std=0.1)

    def a_avg(self, state):
        return self.net(state)

    def forward(self, state):
        return self.net(state).tanh()

    def frozen_transfer(self):
        for p in self.net.parameters():
            p.requires_grad = False
        for p in self.net[-1].parameters():
            p.requires_grad = True


class ActorResidualPPO(ActorPPO):
    """net_residual.py:6-66: action = tanh(net(s)) + s @ priorK."""

    def __init__(self, mid_dim, state_dim, action_dim, if_use_dn=False):
        nn.Module.__init__(self)
        assert not if_use_dn and action_dim == 1, "only the configuration the scripts use is implemented"
        self.net = _mlp([state_dim, mid_dim, mid_dim, mid_dim, action_dim], nn.Tanh)
        self.a_std_log = nn.Parameter(torch.zeros((1, action_dim)) - 0.5, requires_grad=True)
        self.sqrt_2pi_log = np.log(np.sqrt(2 * np.pi))
        self.priorK = nn.Parameter(torch.randn(state_dim, action_dim) * 0.01, requires_grad=False)
        layer_norm(self.net[-1], std=0.1)

    def forward(self, state):
        return self.net(state).tanh() + state @ self.priorK


class ActorResidualIntegratorModularPPO(nn.Module, _GaussianHead):
    """net_residual.py:138-205: two branches (other observations / integrated error) joined by ``net``."""
    kind = "modular"

    def __init__(self, mid_dim, state_dim, action_dim, integrator_dim, if_use_dn=False):
        super().__init__()
        assert not if_use_dn and action_dim == 1, "only the configuration the scripts use is implemented"
        self.other_dim = state_dim - integrator_dim
        self.other_net = nn.Sequential(nn.Linear(self.other_dim, mid_dim), nn.Tanh(), nn.Linear(mid_dim, mid_dim // 2), nn.Tanh())
        self.integrator_net = nn.Sequential(nn.Linear(integrator_dim, mid_dim), nn.Tanh(), nn.Linear(mid_dim, mid_dim // 2), nn.Tanh())
        self.net = nn.Sequential(nn.Linear(mid_dim // 2 * 2, mid_dim), nn.Tanh(), nn.Linear(mid_dim, action_dim))
        self.a_std_log = nn.Parameter(torch.zeros((1, action_dim)) - 0.5, requires_grad=True)
        self.sqrt_2pi_log = np.log(np.sqrt(2 * np.pi))
        self.priorK = nn.Parameter(torch.randn(state_dim, action_dim) * 0.01, requires_grad=False)
        layer_norm(self.net[-1], std=0.1)

    def a_avg(self, state):
        return self.net(torch.cat([self.other_net(state[:, :self.other_dim]), self.integrator_net(state[:, self.other_dim:])], dim=-1))

    def forward(self, state):
        return self.a_avg(state).tanh() + state @ self.priorK

    def frozen_integrator(self):
        for p in self.integrator_net.parameters():
            p.requires_grad = False

    def frozen_transfer(self):
        for m in (self.integrator_net, self.other_net, self.net):
            for p in m.parameters():
                p.requires_grad = False
        for p in self.net[-1].parameters():
            p.requires_grad = True


class CriticAdv(nn.Module):
    """net.py:274-277 as constructed (ReLU MLP S -> H -> H -> H -> 1, output layer orthogonal std 0.5)."""
    kind = "critic"

    def __init__(self, state_dim, mid_dim, if_use_dn=False):
        super().__init__()
        assert not if_use_dn
        # the reference builds the net twice (the first Sequential is discarded); building it twice keeps torch's RNG
        # stream, hence the initial weights for a given seed, identical to the reference's
        for _ in range(2):
            self.net = _mlp([state_dim, mid_dim, mid_dim, mid_dim, 1], nn.ReLU)
        layer_norm(self.net[-1], std=0.5)

    def forward(self, state):
        return self.net(state)

    def frozen_transfer(self):
        for p in self.net.parameters():
            p.requires_grad = False


# ====================================================================================================== fused learner
class FusedLearner:
    """The two-launch PPO minibatch step of libpime_b200 (pime_ppo_step, csrc/learner.cu): flat fp32 copies of the actor,
    the critic and a_std_log (+ their transposes and the Adam moments), loaded from the torch modules before a round of
    minibatch steps and stored back after it.  The moments and the step count persist across update_net calls like the
    state of the torch optimizer they replace (agent.py:56-58)."""

    RING = 4096

    def __init__(self, act, cri, state_dim, net_dim, device):
        import ctypes as C
        self.C, self.L = C, V.L
        D = getattr(act, "other_dim", None)
        self.kind = act.kind
        self.cfg = V.L.ActorConfig(kind=V.ActorPack.KIND[act.kind], state_dim=state_dim, mid_dim=net_dim,
                                   integrator_dim=state_dim - D if D is not None else 0)
        lay = (C.c_int64 * 3)()
        V.L.check(V.L.lib().pime_ppo_theta_layout(C.byref(self.cfg), lay))
        self.cri_off, self.astd_off, n = int(lay[0]), int(lay[1]), int(lay[2])
        self.device = device
        self.theta, self.theta_t, self.m, self.v = (torch.zeros(n, dtype=torch.float32, device=device) for _ in range(4))
        self.state = torch.zeros(1024, dtype=torch.int32, device=device)
        self.loss_ring = torch.zeros((self.RING, 4), dtype=torch.float32, device=device)
        self.work = None
        self.grad = None        # distributed: flat gradient of this rank's minibatch, all-reduced before the Adam kernel
        self.work_tc = None     # scratch of the tensor-core step (activations / gradients of one minibatch in T-format)
        self.steps = 0          # host mirror of the device step count
        self._args = None
        self._step_fn = V.L.lib().pime_ppo_step
        self._keys = (V.ActorPack.KEYS[act.kind], V.ActorPack.KEYS["critic"])

    @staticmethod
    def use_tc(agent, batch_size):
        """Batches from ``tc_learner_min_batch`` rows on take the tcgen05 step (pime_ppo_grad_tc: 128-row tiles, hi / lo fp16
        GEMMs); it needs net_dim 128 or 256."""
        return batch_size >= agent.tc_learner_min_batch and agent.net_dim in (128, 256) and batch_size <= (1 << 20)

    @staticmethod
    def eligible(agent, batch_size):
        """Everything trainable (the frozen_* variants keep the autograd step), one action.  Under torch.distributed the
        step becomes gradient kernels -> flat all-reduce -> Adam kernel (pime_ppo_apply_grad)."""
        if agent.act.kind not in ("plain", "modular") or batch_size < 2:
            return False
        if not (batch_size <= agent.fused_max_batch or FusedLearner.use_tc(agent, batch_size)):
            return False
        named = list(agent.act.named_parameters()) + list(agent.cri.named_parameters())
        return all(p.requires_grad or n == "priorK" for n, p in named) and agent.act.a_std_log.numel() == 1

    def _tensors(self, act, cri):
        sa, sc = dict(act.named_parameters()), dict(cri.named_parameters())
        return [sa[k] for k in self._keys[0]] + [sc[k] for k in self._keys[1]] + [act.a_std_log]

    def _slices(self, act, cri):
        """(tensor, offset in theta) for every trained tensor: actor from 0, critic from cri_off, a_std_log last."""
        ts = self._tensors(act, cri)
        na = len(self._keys[0])
        out, o = [], 0
        for i, t in enumerate(ts):
            if i == na:
                o = self.cri_off
            if i == len(ts) - 1:
                o = self.astd_off
            out.append((t, o))
            o += t.numel()
        return out

    def load(self, act, cri):
        with torch.no_grad():
            for t, o in self._slices(act, cri):
                self.theta[o:o + t.numel()].copy_(t.detach().reshape(-1))
        self.L.check(self.L.lib().pime_ppo_transpose(self.C.byref(self.cfg), self.L.ptr(self.theta), self.L.ptr(self.theta_t),
                                                     self.L.stream_ptr()))

    def store(self, act, cri):
        with torch.no_grad():
            for t, o in self._slices(act, cri):
                t.copy_(self.theta[o:o + t.numel()].view_as(t))

    def _bind(self, data, idx, agent, tc, grad_out=None):
        """The argument block (by reference) for rows ``idx`` of data = (state, action, r_sum, logprob, advantage) on the
        SIMT step or, with ``tc``, the tensor-core step.  It is rebuilt, and its scratch grown, only when a data pointer, the
        batch size, the path or grad_out changes; the scalars follow the agent / optimizer on every call (a learning-rate
        change between two update_net calls must reach the kernels)."""
        C, L = self.C, self.L
        B = int(idx.numel())
        key = (tuple(t.data_ptr() for t in data), B, tc, None if grad_out is None else grad_out.data_ptr())
        if self._args is None or self._args[0] != key:
            state, action, r_sum, logprob, advantage = data
            if tc:
                need = int(L.lib().pime_ppo_tc_work_bytes(C.byref(self.cfg), C.c_int32(B)))
                if need < 0:
                    raise ValueError("the tensor-core learner needs net_dim 128 or 256")
                if self.work_tc is None or self.work_tc.numel() < need:
                    self.work_tc = torch.empty(need, dtype=torch.uint8, device=self.device)
            else:
                need = int(L.lib().pime_ppo_work_floats(C.byref(self.cfg), C.c_int32(B)))
                if self.work is None or self.work.numel() < need:
                    self.work = torch.empty(need, dtype=torch.float32, device=self.device)
            a = L.PpoArgs(actor=C.pointer(self.cfg), theta=L.ptr(self.theta), theta_t=L.ptr(self.theta_t), adam_m=L.ptr(self.m),
                          adam_v=L.ptr(self.v), grad_out=L.ptr(grad_out), buf_state=L.ptr(state), buf_action=L.ptr(action),
                          buf_r_sum=L.ptr(r_sum), buf_logprob=L.ptr(logprob), buf_advantage=L.ptr(advantage), batch=B,
                          state=L.ptr(self.state), work=None if tc else L.ptr(self.work), loss_ring=L.ptr(self.loss_ring),
                          ring_len=self.RING)
            self._args = (key, a, C.byref(a), data)
        a = self._args[1]
        a.idx = idx.data_ptr()
        grp = agent.optimizer.param_groups[0]
        a.ratio_clip, a.lambda_entropy = agent.ratio_clip, agent.lambda_entropy
        a.lr, a.beta1, a.beta2, a.eps = grp["lr"], grp["betas"][0], grp["betas"][1], grp["eps"]
        return self._args[2]

    def step(self, data, idx, agent, grad_out=None):
        """One minibatch step on rows ``idx`` of data = (state, action, r_sum, logprob, advantage)."""
        C, L = self.C, self.L
        args = self._bind(data, idx, agent, False, grad_out)
        stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
        L.check(self._step_fn(args, stream))
        if grad_out is not None and grad_out is self.grad:   # data parallel: mean gradient over the job, then Adam
            torch.distributed.all_reduce(grad_out)
            L.check(L.lib().pime_ppo_apply_grad(args, L.ptr(grad_out), C.c_float(1.0 / torch.distributed.get_world_size()), stream))
        self.steps += 1

    def dist_grad(self):
        if self.grad is None:
            self.grad = torch.zeros_like(self.theta)
        return self.grad

    def step_tc(self, data, idx, agent, distributed=False):
        """One minibatch step on the tensor cores: pime_ppo_grad_tc -> (all-reduce) -> pime_ppo_apply_grad -> close."""
        C, L = self.C, self.L
        args = self._bind(data, idx, agent, True)
        grad = self.dist_grad()
        stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
        lib = L.lib()
        L.check(lib.pime_ppo_grad_tc(args, L.ptr(self.work_tc), L.ptr(grad), stream))
        scale = 1.0
        if distributed:
            torch.distributed.all_reduce(grad)               # one flat 1.07-MB all-reduce between two of this library's kernels
            scale = 1.0 / torch.distributed.get_world_size()
        L.check(lib.pime_ppo_apply_grad(args, L.ptr(grad), C.c_float(scale), stream))
        L.check(lib.pime_ppo_close_step(args, stream))
        self.steps += 1

    def losses(self, first, count):
        """Rows [first, first + count) of the loss ring -> [count, 4] (united, actor, critic, entropy)."""
        rows = torch.arange(first, first + count, device=self.device) % self.RING
        return self.loss_ring[rows]


# ====================================================================================================== replay buffer
class ReplayBuffer:
    """On-policy part of replay.py:238-379 with the storage in HBM.

    Rows are (state[S]) and other = (reward*scale, mask, a_raw, noise) as in the reference.  ``num_envs`` > 1 makes the
    buffer time-major: row index = t * num_envs + env, which is how the fused rollout kernel writes it; the GAE scan
    then runs per env column.  With num_envs = 1 the order is the reference's.
    """

    def __init__(self, max_len, state_dim, action_dim, if_on_policy=True, if_per=False, if_gpu=True, num_envs=1, device="cuda"):
        assert if_on_policy and not if_per, "only the on-policy buffer is on the PIME path"
        assert action_dim == 1
        self.device = torch.device(device if torch.cuda.is_available() else "cpu")
        self.num_envs = int(num_envs)
        self.max_len = int(math.ceil(max_len / self.num_envs) * self.num_envs)
        self.state_dim, self.action_dim, self.other_dim = int(state_dim), 1, 4
        self.now_len = self.next_idx = 0
        self.if_full = False
        self.if_on_policy, self.if_per, self.if_gpu = True, False, True
        self.buf_state = torch.empty((self.max_len, self.state_dim), dtype=torch.float32, device=self.device)
        self.buf_other = torch.empty((self.max_len, self.other_dim), dtype=torch.float32, device=self.device)
        self._host_state, self._host_other, self._host_from = [], [], 0

    # ---- reference API
    def append_buffer(self, state, other):
        """One transition from a host loop (foreign gym env); staged on the host, uploaded before sampling."""
        if not self._host_state:
            self._host_from = self.next_idx
        self._host_state.append(np.asarray(state, dtype=np.float32).reshape(-1))
        self._host_other.append(np.asarray(other, dtype=np.float32).reshape(-1))
        self.next_idx += 1
        if self.next_idx >= self.max_len:
            self._flush()
            self.if_full, self.next_idx = True, 0

    def _flush(self):
        if self._host_state:
            k = len(self._host_state)
            self.buf_state[self._host_from:self._host_from + k] = torch.as_tensor(np.stack(self._host_state), device=self.device)
            self.buf_other[self._host_from:self._host_from + k] = torch.as_tensor(np.stack(self._host_other), device=self.device)
            self._host_state, self._host_other = [], []

    def rollout_views(self, T):
        """Time-major [T, n, S] / [T, n, 4] views of the next T*n rows (what pime_*_rollout_* writes)."""
        n = self.num_envs
        assert self.next_idx % n == 0 and self.next_idx + T * n <= self.max_len, "replay buffer too small for this rollout"
        lo = self.next_idx
        return (self.buf_state[lo:lo + T * n].view(T, n, self.state_dim), self.buf_other[lo:lo + T * n].view(T, n, 4))

    def commit_rollout(self, T):
        self.next_idx += T * self.num_envs

    def update_now_len_before_sample(self):
        self._flush()
        self.now_len = self.max_len if self.if_full else self.next_idx

    def empty_buffer_before_explore(self):
        self._host_state, self._host_other = [], []
        self.next_idx = self.now_len = 0
        self.if_full = False

    def gather(self):
        """Single-learner mode (SURVEY 8e): every rank receives the whole job's on-policy replay.  The local buffer holds
        time-major rows [T, n_rank, .] of this rank's contiguous env range (``shard_range``); the result is a time-major
        buffer over ALL envs, [T, sum(n_rank), .], ranks in order -- the rows one process would have written had it owned
        every env.  One all-gather (NCCL on GPUs) of the (S + 4)-float rows; ranks may own different numbers of envs (the
        shorter ones are padded for the collective).  Without torch.distributed it returns self."""
        if not _dist_on():
            return self
        dist = torch.distributed
        self._flush()
        world, n = dist.get_world_size(), self.num_envs
        rows = self.max_len if self.if_full else self.next_idx
        assert rows % n == 0, "the time-major buffer holds whole steps"
        T = rows // n
        meta = torch.tensor([n, T], dtype=torch.int64, device=self.device)
        metas = [torch.empty_like(meta) for _ in range(world)]
        dist.all_gather(metas, meta)
        ns = [int(m[0]) for m in metas]
        assert all(int(m[1]) == T for m in metas), "every rank must hold the same number of steps"
        n_max, W = max(ns), self.state_dim + self.other_dim
        mine = torch.zeros((T, n_max, W), dtype=torch.float32, device=self.device)
        mine[:, :n, :self.state_dim] = self.buf_state[:rows].view(T, n, self.state_dim)
        mine[:, :n, self.state_dim:] = self.buf_other[:rows].view(T, n, self.other_dim)
        parts = [torch.empty_like(mine) for _ in range(world)]
        dist.all_gather(parts, mine)
        full = torch.cat([p[:, :k] for p, k in zip(parts, ns)], dim=1)       # [T, sum(ns), S + 4]
        out = ReplayBuffer(T * sum(ns), self.state_dim, 1, True, False, True, num_envs=sum(ns), device=str(self.device))
        out.buf_state[:] = full[..., :self.state_dim].reshape(-1, self.state_dim)
        out.buf_other[:] = full[..., self.state_dim:].reshape(-1, self.other_dim)
        out.next_idx = out.now_len = T * sum(ns)
        return out

    def sample_all(self):
        """(reward[L], mask[L], action[L,1], noise[L,1], state[L,S]) -- replay.py:353-368."""
        o = self.buf_other[:self.now_len]
        return o[:, 0], o[:, 1], o[:, 2:3], o[:, 3:4], self.buf_state[:self.now_len]


# ====================================================================================================== agents
def _device_env(env):
    """The pime_b200 gym_api env behind (possibly) a PreprocessEnv wrapper, or None for a foreign gym env."""
    base = getattr(env, "env", env)
    return base if hasattr(base, "vec") else None


def _episode_len(env, dev):
    """env.max_step (water tank: 200) or the TimeLimit of the pH ids (50), elegantrl/env.py:221-231."""
    return int(getattr(env, "max_step", None) or getattr(dev, "max_step", None) or dev._max_episode_steps)


class AgentPPO:
    """elegantrl/agent.py:536-708."""
    actor_cls = ActorPPO

    def __init__(self):
        self.learning_rate = 1e-4
        self.ratio_clip, self.lambda_entropy, self.lambda_gae_adv = 0.2, 0.02, 0.97
        self.if_use_gae, self.if_on_policy, self.if_use_dn = True, True, False
        self.state = None
        self.device = None
        self.act = self.cri = self.optimizer = self.criterion = None
        self.compute_reward = None
        self.priorK = None
        self._n_updates = 0
        self._packs = {}
        self._graph = None
        self.use_cuda_graph = True      # record the minibatch step into a CUDA graph when it is launch bound
        self.graph_max_batch = 8192
        self.graph_steps = 4            # minibatch steps per recorded graph
        self.use_fused_learner = True   # pime_ppo_step (two launches per minibatch) when FusedLearner.eligible
        self.fused_max_batch = 4096     # the fp32 SIMT kernels (pime_ppo_step) up to here
        self.tc_learner_min_batch = 2048  # from here on the tcgen05 step (pime_ppo_grad_tc) when net_dim is 128 or 256
        self._fused = None
        self.learner_path = None        # which minibatch step the last update_net ran (reported by bench.py)
        self.value_fp32_max_rows = 1 << 20

    # ---- construction
    def _make_actor(self, net_dim, state_dim, action_dim, **kw):
        return self.actor_cls(net_dim, state_dim, action_dim, self.if_use_dn)

    def init(self, net_dim, state_dim, action_dim, if_per=False, **kw):
        assert if_per is False  # on-policy does not need PER
        self.device = torch.device("cuda" if torch.cuda.is_available() else "cpu")
        self.compute_reward = self.compute_reward_gae if self.if_use_gae else self.compute_reward_adv
        self.net_dim, self.state_dim = int(net_dim), int(state_dim)
        self.cri = CriticAdv(state_dim, net_dim, self.if_use_dn).to(self.device)
        self.act = self._make_actor(net_dim, state_dim, action_dim, **kw).to(self.device)
        self._new_optimizer()
        self.criterion = torch.nn.SmoothL1Loss()
        self.priorK = np.zeros((state_dim, 1))

    def _new_optimizer(self):
        # capturable: the minibatch step can be recorded into a CUDA graph (same arithmetic as the eager step)
        on_gpu = self.device is not None and self.device.type == "cuda"
        self.optimizer = torch.optim.Adam([{"params": self.act.parameters(), "lr": self.learning_rate},
                                           {"params": self.cri.parameters(), "lr": self.learning_rate}],
                                          capturable=on_gpu, fused=True if on_gpu else None)   # one Adam kernel per step
        self._graph = None
        self._fused = None      # a new optimizer starts from zero moments on the fused path too

    def init_actor_zero(self):
        """agent_residual.py:45-50: last layer zeroed -> the policy starts exactly at the prior."""
        self.act.net[-1].bias.data.fill_(0.0)
        self.act.net[-1].weight.data.fill_(0.0)
        self._new_optimizer()

    def frozen_transfer(self):
        self.cri.frozen_transfer()
        self.act.frozen_transfer()
        self._invalidate_learner()

    def _invalidate_learner(self):
        """The recorded CUDA graph bakes in which parameters are trained and the fused learner keeps its own Adam moments:
        both are dropped whenever the set of trained parameters changes (the moments restart from zero, as they would for
        the parameters torch.optim.Adam has not seen a gradient of)."""
        self._graph = None
        self._fused = None

    # ---- kernel images of the networks
    def _pack(self, which):
        net = self.act if which == "act" else self.cri
        p = self._packs.get(which)
        if p is None:
            D = getattr(net, "other_dim", None)
            p = V.ActorPack(net.kind, self.state_dim, self.net_dim, self.state_dim - D if D is not None else 0, device=self.device)
            self._packs[which] = p
        return p.update(net.state_dict())

    # ---- acting
    def select_action(self, state, if_deterministic=False):
        """agent.py:577-589.  One observation -> (a_raw[1], noise[1]) or (deterministic action[1], None)."""
        states = torch.as_tensor(np.asarray(state, dtype=np.float32).reshape(1, -1), device=self.device)
        with torch.no_grad():
            if if_deterministic:
                return self.act(states)[0].cpu().numpy(), None
            a, nz = self.act.get_action_noise(states)
        return a[0].cpu().numpy(), nz[0].cpu().numpy()

    def _env_action(self, state, action):
        return np.tanh(action)  # agent.py:601

    def explore_env(self, env, buffer, target_step, reward_scale, gamma) -> int:
        """agent.py:591-609 / agent_residual.py:52-69.  Whole episodes until target_step transitions are stored."""
        buffer.empty_buffer_before_explore()
        dev = _device_env(env)
        if dev is None:
            return self._explore_foreign(env, buffer, target_step, reward_scale, gamma)
        vec, n = dev.vec, dev.num_envs
        assert buffer.num_envs == n, "ReplayBuffer(num_envs=...) must match the env"
        T = _episode_len(env, dev)
        actor = self._pack("act")
        priorK = np.asarray(self.priorK, dtype=np.float64).reshape(-1)
        steps = 0
        while steps < target_step:
            vec.reset(resample_params=dev.if_reset_all)
            dev._reset_done = True
            vec.rollout(T, priorK, actor=actor, deterministic=False, auto_reset=False, reward_scale=reward_scale, gamma=gamma,
                        replay=buffer.rollout_views(T), a_std_log=float(self.act.a_std_log.detach().reshape(-1)[0]))
            buffer.commit_rollout(T)
            steps += T * n
        vec.check_status()
        return steps

    def _explore_foreign(self, env, buffer, target_step, reward_scale, gamma) -> int:
        actual_step = 0
        while actual_step < target_step:
            state = env.reset()
            for _ in range(env.max_step):
                action, noise = self.select_action(state)
                next_state, reward, done, _ = env.step(self._env_action(state, action))
                actual_step += 1
                buffer.append_buffer(state, (reward * reward_scale, 0.0 if done else gamma, *action, *noise))
                if done:
                    break
                state = next_state
        return actual_step

    # ---- learning
    def _values(self, buf_state):
        """Critic over the whole buffer in one launch (the reference loops 1024-row torch slices, agent.py:619).  Buffers up to
        ``value_fp32_max_rows`` rows use the fidelity mode (fp32 CUDA cores: the reference's arithmetic, so GAE sees the
        values torch would produce); larger ones the tcgen05 engine (fp16 hidden operands, ~1e-3 of the output scale)."""
        pack = self._pack("cri")
        pack.set_precision("fp32" if buf_state.shape[0] <= self.value_fp32_max_rows else "tc")
        return pack.forward(buf_state)

    def _time_major(self, buffer, x):
        n = buffer.num_envs
        return x.reshape(-1, n)

    def compute_reward_gae(self, buf_len, buf_reward, buf_mask, buf_value, num_envs=1):
        """agent.py:685-708 with the reverse loop as a per-env CUDA scan."""
        r = buf_reward.reshape(-1, num_envs).contiguous()
        m = buf_mask.reshape(-1, num_envs).contiguous()
        v = buf_value.reshape(-1, num_envs).contiguous()
        r_sum, adv = V.gae_scan(r, m, v, float(self.lambda_gae_adv))
        return r_sum.reshape(-1), self._normalise(adv.reshape(-1))

    def compute_reward_adv(self, buf_len, buf_reward, buf_mask, buf_value, num_envs=1):
        """agent.py:666-683."""
        r = buf_reward.reshape(-1, num_envs).contiguous()
        m = buf_mask.reshape(-1, num_envs).contiguous()
        v = buf_value.reshape(-1, num_envs).contiguous()
        r_sum, _ = V.gae_scan(r, m, v, 0.0)
        r_sum = r_sum.reshape(-1)
        return r_sum, self._normalise(r_sum - buf_mask.reshape(-1) * buf_value.reshape(-1))

    @staticmethod
    def _normalise(adv):
        """(adv - mean) / (std + 1e-5), unbiased std like torch.Tensor.std; global moments under torch.distributed."""
        cnt = torch.tensor([adv.numel()], dtype=torch.float64, device=adv.device)
        mom = torch.stack([adv.double().sum(), (adv.double() ** 2).sum()])
        if _dist_on():
            torch.distributed.all_reduce(cnt)
            torch.distributed.all_reduce(mom)
        mean = mom[0] / cnt[0]
        var = (mom[1] - cnt[0] * mean * mean) / (cnt[0] - 1).clamp_min(1)
        return ((adv - mean.float()) / (var.clamp_min(0).sqrt().float() + 1e-5))

    def ppo_objectives(self, state, action, r_sum, logprob, advantage):
        """The losses of one minibatch, agent.py:635-652."""
        new_logprob = self.act.compute_logprob(state, action)
        ratio = (new_logprob - logprob).exp()
        surrogate = -torch.min(advantage * ratio, advantage * ratio.clamp(1 - self.ratio_clip, 1 + self.ratio_clip)).mean()
        obj_entropy = (new_logprob.exp() * new_logprob).mean()
        obj_actor = surrogate + obj_entropy * self.lambda_entropy
        value = self.cri(state).squeeze(1)
        obj_critic = self.criterion(value, r_sum)
        obj_united = obj_actor + obj_critic / (r_sum.std() + 1e-5)
        return obj_actor, obj_critic, obj_united, obj_entropy

    def update_net(self, buffer, _target_step, batch_size, repeat_times=4):
        """agent.py:611-664."""
        if self.device.type != "cuda":
            raise V.L.PimeError("update_net needs a CUDA device: the value / GAE passes are CUDA kernels (no CPU fallback)")
        buffer.update_now_len_before_sample()
        buf_len = buffer.now_len
        with torch.no_grad():
            buf_reward, buf_mask, buf_action, buf_noise, buf_state = buffer.sample_all()
            buf_value = self._values(buf_state)
            buf_logprob = -(buf_noise.pow(2) * 0.5 + self.act.a_std_log + self.act.sqrt_2pi_log).sum(1)
            buf_r_sum, buf_advantage = self.compute_reward(buf_len, buf_reward, buf_mask, buf_value, buffer.num_envs)
        params = [p for g in self.optimizer.param_groups for p in g["params"]]
        iters = int(repeat_times * buf_len / batch_size)
        data = (buf_state, buf_action, buf_r_sum, buf_logprob, buf_advantage)

        def minibatch(src, out):
            idx = torch.randint(buf_len, size=(batch_size,), device=self.device)
            obj_actor, obj_critic, obj_united, obj_entropy = self.ppo_objectives(*(t[idx] for t in src))
            self.optimizer.zero_grad(set_to_none=False)
            obj_united.backward()
            if _dist_on():
                allreduce_mean_grads(params)
            self.optimizer.step()
            out.copy_(torch.stack([obj_united.detach(), obj_actor.detach(), obj_critic.detach(), obj_entropy.detach()]))

        if self.use_fused_learner and iters and FusedLearner.eligible(self, batch_size):
            return self._update_fused(data, buf_len, batch_size, iters, repeat_times)

        self.learner_path = "torch autograd (cuBLAS, " + ("TF32" if torch.backends.cuda.matmul.allow_tf32 else "fp32") + ")"
        sums = torch.zeros(4, device=self.device)
        last = torch.zeros(4, device=self.device)
        use_graph = self.use_cuda_graph and iters >= 8 and batch_size <= self.graph_max_batch and not _dist_on()
        done = 0
        if use_graph:
            G = self.graph_steps

            def several(src, out):   # G consecutive minibatch steps per recorded graph; out = (sum of the G loss vectors, last)
                out[:4].zero_()
                for _ in range(G):
                    minibatch(src, out[4:])
                    out[:4] += out[4:]

            g = self._graphed_step(several, data, buf_len, batch_size)
            for _ in range(iters // G):
                g.replay()
                sums += self._graph["out"][:4]
            done = (iters // G) * G
            if done:
                last = self._graph["out"][4:].clone()
        for _ in range(iters - done):
            minibatch(data, last)
            sums += last
        self._n_updates += int(repeat_times)
        if iters:
            u, a, c, e = (sums / iters).tolist()
            logger.record("train/united_loss", u)
            logger.record("train/actor_loss", a)
            logger.record("train/critic_loss", c)
            logger.record("train/entropy_losses", e)
            return float(last[1]), float(last[2])
        return 0.0, 0.0

    def _update_fused(self, data, buf_len, batch_size, iters, repeat_times):
        """The minibatch loop of agent.py:635-658 on the fused kernels: index draw (torch) + two launches per step."""
        f = self._fused
        if f is None or f.kind != self.act.kind:
            f = self._fused = FusedLearner(self.act, self.cri, self.state_dim, self.net_dim, self.device)
        f.load(self.act, self.cri)
        data = (data[0].contiguous(),) + tuple(t.reshape(-1).contiguous() for t in data[1:])   # [L, S], then four [L] columns
        first = f.steps
        dist_on = _dist_on()
        if FusedLearner.use_tc(self, batch_size):
            for _ in range(iters):
                idx = torch.randint(buf_len, size=(batch_size,), device=self.device)
                f.step_tc(data, idx, self, dist_on)
            self.learner_path = ("pime_ppo_grad_tc (tcgen05: 128-row tiles, fp16 hi/lo operands, fp32 accumulation in TMEM) -> " +
                                 ("NCCL all-reduce of the flat gradient -> " if dist_on else "") + "pime_ppo_apply_grad (Adam)")
        else:
            grad = f.dist_grad() if dist_on else None
            for _ in range(iters):
                idx = torch.randint(buf_len, size=(batch_size,), device=self.device)
                f.step(data, idx, self, grad)
            self.learner_path = ("pime_ppo_step (rows + weight-gradient kernels, fp32" +
                                 (", NCCL all-reduce of the flat gradient, Adam kernel)" if grad is not None else ", Adam fused)"))
        f.store(self.act, self.cri)
        f._args = None                      # do not keep the replay tensors alive between calls
        self._n_updates += int(repeat_times)
        keep = min(iters, f.RING - 1)
        rows = f.losses(first + iters - keep, keep)
        u, a, c, e = rows.mean(0).tolist()
        logger.record("train/united_loss", u)
        logger.record("train/actor_loss", a)
        logger.record("train/critic_loss", c)
        logger.record("train/entropy_losses", e)
        return float(rows[-1, 1]), float(rows[-1, 2])

    def _graphed_step(self, minibatch, data, buf_len, batch_size):
        """One PPO minibatch (index draw, gather, forward, backward, Adam) recorded ONCE into a CUDA graph and replayed:
        the reference's configurations (batch 128-512) are launch-latency bound (~60 small kernels per minibatch).
        The graph reads static copies of the buffer tensors; it is re-recorded when a shape changes."""
        trainable = tuple(p.requires_grad for grp in self.optimizer.param_groups for p in grp["params"])
        key = (buf_len, batch_size, self.graph_steps, tuple(t.shape for t in data), trainable, float(self.ratio_clip),
               float(self.lambda_entropy), tuple(float(grp["lr"]) for grp in self.optimizer.param_groups))
        if self._graph is None or self._graph["key"] != key:
            static = tuple(torch.empty_like(t) for t in data)
            out = torch.zeros(8, device=self.device)
            for s, t in zip(static, data):
                s.copy_(t)
            # snapshot: the warm-up iterations and the capture itself must not change the training state; everything is
            # restored IN PLACE because the recorded graph holds the addresses of the parameters and Adam moments
            plist = [p for grp in self.optimizer.param_groups for p in grp["params"]]
            p_snap = [p.detach().clone() for p in plist]
            o_snap = {id(p): {k: v.clone() for k, v in self.optimizer.state.get(p, {}).items() if torch.is_tensor(v)} for p in plist}
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                for _ in range(3):
                    minibatch(static, out)
            torch.cuda.current_stream().wait_stream(side)
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                minibatch(static, out)
            with torch.no_grad():
                for p, snap in zip(plist, p_snap):
                    p.copy_(snap)
                    for k, v in self.optimizer.state.get(p, {}).items():
                        if torch.is_tensor(v):
                            v.copy_(o_snap[id(p)][k]) if k in o_snap[id(p)] else v.zero_()
            self._graph = {"key": key, "graph": graph, "static": static, "out": out}
        else:
            for s, t in zip(self._graph["static"], data):
                s.copy_(t)
        return self._graph["graph"]

    # ---- checkpoints (agent.py:86-114): same file names and state-dict keys as the reference
    def save_load_model(self, cwd, if_save):
        act_path, cri_path = f"{cwd}/actor.pth", f"{cwd}/critic.pth"
        if if_save:
            torch.save(self.act.state_dict(), act_path)
            torch.save(self.cri.state_dict(), cri_path)
            return
        for net, path, name in ((self.act, act_path, "act"), (self.cri, cri_path, "cri")):
            if os.path.exists(path):
                net.load_state_dict(torch.load(path, map_location=lambda storage, loc: storage))
                print(f"Loaded {name}:", cwd)
            else:
                print(f"FileNotFound when load {name}: {cwd}")


class Residual:
    """agent_residual.py:15-24."""

    def init_residual(self, residual_kwarg):
        K = np.asarray(residual_kwarg["init_K"], dtype=np.float64)
        self.act.priorK = nn.Parameter(-torch.as_tensor(K, dtype=torch.float32, device=self.device), requires_grad=False)
        self.init_actor_zero()
        self.priorK = -K

    def fix_K(self):
        self.act.priorK.requires_grad = False
        self._invalidate_learner()


class AgentResidualPPO(AgentPPO, Residual):
    """agent_residual.py:32-74: env action = tanh(a_raw) + state @ priorK."""
    actor_cls = ActorResidualPPO

    def _env_action(self, state, action):
        return np.tanh(action) + np.asarray(state) @ self.priorK  # agent_residual.py:61


class AgentResidualIntegratorModularPPO(AgentResidualPPO):
    """agent_residual.py:77-98."""
    actor_cls = ActorResidualIntegratorModularPPO

    def _make_actor(self, net_dim, state_dim, action_dim, integrator_dim=1, **kw):
        return ActorResidualIntegratorModularPPO(net_dim, state_dim, action_dim, integrator_dim, self.if_use_dn)

    def init(self, net_dim, state_dim, action_dim, integrator_dim=1, if_per=False):
        super().init(net_dim, state_dim, action_dim, if_per, integrator_dim=integrator_dim)

    def frozen_integrator(self):
        self.act.frozen_integrator()
        self.cri.frozen_transfer()
        self._invalidate_learner()


MODELS = {"ppo": AgentPPO, "residualppo": AgentResidualPPO, "residualintegratormodularppo": AgentResidualIntegratorModularPPO}
IF_ONPOLICY = {"ppo": True, "residualppo": True, "residualintegratormodularppo": True, "td3": False, "sac": False}
# utils/utils.py also lists td3 / sac: off-policy agents are outside the path this package accelerates (DESIGN.md section 7)


# ====================================================================================================== distributed helpers
def _dist_on():
    return torch.distributed.is_available() and torch.distributed.is_initialized() and torch.distributed.get_world_size() > 1


def allreduce_mean_grads(params):
    """Average the gradients of ``params`` over the job with ONE flat all-reduce (actor + critic ~ 1 MB: latency bound)."""
    grads = [p.grad for p in params if p.grad is not None]
    if not grads:
        return
    flat = torch.cat([g.reshape(-1) for g in grads])
    torch.distributed.all_reduce(flat)
    flat /= torch.distributed.get_world_size()
    off = 0
    for g in grads:
        g.copy_(flat[off:off + g.numel()].view_as(g))
        off += g.numel()


def shard_range(n_total: int, rank: int, world: int):
    """Contiguous env-id range of a rank (SURVEY 8e): [lo, hi).  Philox is keyed by the global id, so any split of the
    same n_total produces the same per-env streams."""
    base, rem = divmod(int(n_total), int(world))
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)


# ====================================================================================================== env wrapper
class PreprocessEnv:
    """elegantrl/env.py:10-72: float32 observations, action scaling, env facts (get_gym_env_info :194-245)."""

    def __init__(self, env, if_print=False, data_type=np.float32):
        if isinstance(env, str):
            from . import gym_api
            env = gym_api.make(env)
        self.env, self.data_type = env, data_type
        spec = getattr(getattr(env, "unwrapped", env), "spec", None)
        self.env_name = getattr(spec, "id", env.__class__.__name__)
        self.state_dim = int(env.observation_space.shape[0])
        self.action_dim = int(env.action_space.shape[0])
        self.action_max = float(env.action_space.high[0])
        self.if_discrete = False
        max_step = getattr(env, "max_step", None)
        if max_step is None:
            max_step = getattr(env, "_max_episode_steps", None) or getattr(spec, "max_episode_steps", None) or 2 ** 10
        self.max_step = int(max_step)
        tr = getattr(env, "target_return", None)
        self.target_return = float(tr if tr is not None else (getattr(spec, "reward_threshold", None) or 2 ** 16))
        self.observation_space, self.action_space = env.observation_space, env.action_space
        if if_print:
            print(f"| env_name: {self.env_name}, state_dim: {self.state_dim}, action_dim: {self.action_dim}, "
                  f"max_step: {self.max_step}, target_return: {self.target_return}")

    @property
    def unwrapped(self):
        return getattr(self.env, "unwrapped", self.env)

    def reset(self):
        return np.asarray(self.env.reset()).astype(self.data_type)

    def step(self, action):
        state, reward, done, info = self.env.step(action * self.action_max)
        return np.asarray(state).astype(self.data_type), reward, done, info

    def __getattr__(self, name):  # delegate everything else (if_reset_all, K, n_integrator, ...)
        # copy / pickle probe dunders (__deepcopy__, __setstate__, ...) on an instance whose __dict__ is still empty
        if name.startswith("__") or "env" not in self.__dict__:
            raise AttributeError(name)
        return getattr(self.__dict__["env"], name)


# ====================================================================================================== evaluation
def get_episode_return(env, act, device, agent=None):
    """run.py:600-619: one deterministic episode -> (return, steps).  With a pime_b200 env and ``agent`` given, all
    ``num_envs`` envs run their episode in one fused launch and a list of (return, steps) comes back."""
    dev = _device_env(env)
    if dev is not None and agent is not None:
        return evaluate_batched(env, agent)
    episode_return, episode_step = 0.0, 0
    state = env.reset()
    for episode_step in range(env.max_step):
        with torch.no_grad():
            action = act(torch.as_tensor(np.asarray(state, dtype=np.float32).reshape(1, -1), device=device))[0].cpu().numpy()
        state, reward, done, _ = env.step(action)
        episode_return += reward
        if done:
            break
    return getattr(env, "episode_return", episode_return), episode_step + 1


def evaluate_batched(env, agent, episodes: Optional[int] = None):
    """Deterministic episodes of every env of a pime_b200 env object: [(return, steps)] * num_envs (run.py:593-619)."""
    dev = _device_env(env)
    vec, n = dev.vec, dev.num_envs
    T = _episode_len(env, dev)
    out = []
    while len(out) < (episodes or n):
        vec.reset(resample_params=dev.if_reset_all)
        dev._reset_done = True
        vec.ep_return.zero_()
        vec.rollout(T, np.asarray(agent.priorK, dtype=np.float64).reshape(-1), actor=agent._pack("act"), deterministic=True)
        out += [(float(r), T) for r in vec.ep_return.cpu().numpy()]
    vec.check_status()
    return out[:episodes] if episodes else out


class Evaluator:
    """run.py:478-597 (the parts train_and_evaluate uses)."""

    def __init__(self, cwd, agent_id, eval_times1, eval_times2, eval_gap, env, device):
        self.recorder = []
        self.r_max = -np.inf
        self.total_step = 0
        self.cwd, self.agent_id, self.device, self.env = cwd, agent_id, device, env
        self.eval_gap, self.eval_times1, self.eval_times2 = eval_gap, eval_times1, eval_times2
        self.target_return = env.target_return
        self.used_time, self.start_time = None, time.time()
        self.eval_func_time = 1

    def _episodes(self, agent, k):
        if _device_env(self.env) is not None:
            return evaluate_batched(self.env, agent, k)
        return [get_episode_return(self.env, agent.act, self.device) for _ in range(k)]

    @staticmethod
    def get_r_avg_std_s_avg_std(rewards_steps_list):
        a = np.array(rewards_steps_list, dtype=np.float64)
        r_avg, s_avg = a.mean(axis=0)
        r_std, s_std = a.std(axis=0)
        return r_avg, r_std, s_avg, s_std

    def evaluate_act(self, agent):
        if self.eval_times1 == 0:
            return False
        r_avg, r_std, _, _ = self.get_r_avg_std_s_avg_std(self._episodes(agent, self.eval_times1))
        if r_avg > self.r_max:
            self.r_max = r_avg
            agent.save_load_model(self.cwd, if_save=True)
        logger.record("rollout/ep_rew_mean", r_avg)
        logger.record("rollout/ep_rew_std", r_std)
        logger.record("rollout/log_rew_max", self.r_max)
        os.makedirs(os.path.join(self.cwd, "init"), exist_ok=True)
        agent.save_load_model(os.path.join(self.cwd, "init"), if_save=True)
        self.recorder.append((self.total_step, r_avg, r_std, 0.0, 0.0))
        return bool(self.r_max > self.target_return)

    def evaluate_save(self, agent, steps, obj_a, obj_c) -> bool:
        if self.eval_times1 == 0:
            return False
        self.total_step += steps
        reach = False
        if self.eval_func_time % self.eval_gap == 0:
            eps = self._episodes(agent, self.eval_times1)
            r_avg, r_std, _, _ = self.get_r_avg_std_s_avg_std(eps)
            if r_avg > self.r_max and self.eval_times2 > self.eval_times1:
                eps += self._episodes(agent, self.eval_times2 - self.eval_times1)
                r_avg, r_std, _, _ = self.get_r_avg_std_s_avg_std(eps)
            if r_avg > self.r_max:
                self.r_max = r_avg
                agent.save_load_model(self.cwd, if_save=True)
            logger.record("rollout/ep_rew_mean", r_avg)
            logger.record("rollout/ep_rew_std", r_std)
            logger.record("rollout/log_rew_max", self.r_max)
            self.recorder.append((self.total_step, r_avg, r_std, obj_a, obj_c))
            reach = bool(self.r_max > self.target_return)
            if reach and self.used_time is None:
                self.used_time = int(time.time() - self.start_time)
        self.eval_func_time += 1
        return reach


# ====================================================================================================== trainer
class Arguments:
    """run.py:14-93 (on-policy defaults; the fields train.py sets)."""

    def __init__(self, agent=None, env=None, gpu_id=None, if_on_policy=True):
        self.agent, self.env, self.env_eval, self.gpu_id, self.cwd = agent, env, None, gpu_id, None
        self.net_dim, self.batch_size, self.repeat_times, self.target_step = 2 ** 9, 2 ** 9, 2 ** 4, 2 ** 12
        self.max_memo = self.target_step
        self.learning_start = 0
        self.gamma, self.reward_scale, self.if_per = 0.99, 2 ** 0, False
        self.break_step, self.if_remove, self.if_allow_break = 2 ** 20, True, True
        self.eval_gap, self.eval_times1, self.eval_times2, self.random_seed = 5, 2 ** 2, 2 ** 4, 0
        self.fix_K = self.frozen_modular_integrator = self.frozen_transfer = False
        self.if_residual = True
        self.SCN_kwargs, self.residual_kwargs, self.Modular_kwargs, self.Q_kwargs = {}, {}, {}, {}
        self.load, self.test_render, self.test_render_times = "None", None, 10 ** 9

    def init_before_training(self, if_main=True):
        if self.agent is None or not hasattr(self.agent, "init"):
            raise RuntimeError("args.agent must be an agent INSTANCE (AgentXXX())")
        if self.env is None or not hasattr(self.env, "env_name"):
            raise RuntimeError("args.env must be a PreprocessEnv")
        if self.cwd is None:
            self.cwd = f"./{self.agent.__class__.__name__}/{self.env.env_name}_{self.gpu_id or 0}"
        if if_main:
            if self.if_remove:
                import shutil
                shutil.rmtree(self.cwd, ignore_errors=True)
            os.makedirs(self.cwd, exist_ok=True)
        torch.manual_seed(self.random_seed)
        np.random.seed(self.random_seed)


def train_and_evaluate(args):
    """run.py:99-225: explore -> update -> evaluate until break_step (or the target return)."""
    args.init_before_training()
    env, agent, cwd = args.env, args.agent, args.cwd
    env_eval = args.env_eval if args.env_eval is not None else deepcopy(env)
    max_step, state_dim, action_dim = env.max_step, env.state_dim, env.action_dim
    if "integrator_dim" in args.Modular_kwargs:
        agent.init(args.net_dim, state_dim, action_dim, args.Modular_kwargs["integrator_dim"], args.if_per)
    else:
        agent.init(args.net_dim, state_dim, action_dim, args.if_per)
    if args.residual_kwargs:
        agent.init_residual(args.residual_kwargs)
    if args.if_residual:
        agent.init_actor_zero()
    if args.fix_K and hasattr(agent, "fix_K"):
        agent.fix_K()
    if args.frozen_modular_integrator:
        agent.frozen_integrator()
    if args.frozen_transfer:
        agent.frozen_transfer()
    if args.load != "None":
        agent.save_load_model(args.load, if_save=False)
    dev = _device_env(env)
    n = dev.num_envs if dev is not None else 1
    rows = max(args.max_memo + max_step, int(math.ceil(args.target_step / (n * max_step))) * n * max_step)
    buffer = ReplayBuffer(max_len=rows, state_dim=state_dim, action_dim=action_dim, if_on_policy=True, if_per=False, if_gpu=True,
                          num_envs=n)
    evaluator = Evaluator(cwd=cwd, agent_id=args.gpu_id or 0, device=agent.device, env=env_eval, eval_gap=args.eval_gap,
                          eval_times1=args.eval_times1, eval_times2=args.eval_times2)
    if_reach_goal = evaluator.evaluate_act(agent)
    logger.dump(step=0)
    agent.state = env.reset()
    total_step = 0
    if args.test_render is not None:                       # run.py:188-191: the self-designed evaluation at step 0
        save_path = os.path.join(cwd, "step_0")
        os.makedirs(save_path, exist_ok=True)
        args.test_render(agent, save_path)
    while not ((args.if_allow_break and if_reach_goal) or total_step >= args.break_step or os.path.exists(f"{cwd}/stop")):
        steps = agent.explore_env(env, buffer, args.target_step, args.reward_scale, args.gamma)
        total_step += steps
        obj_a, obj_c = agent.update_net(buffer, args.target_step, args.batch_size, args.repeat_times)
        if_reach_goal = evaluator.evaluate_save(agent, steps, obj_a, obj_c)
        if args.test_render is not None and total_step % args.test_render_times == 0:
            save_path = os.path.join(cwd, f"step_{total_step}")
            os.makedirs(save_path, exist_ok=True)
            args.test_render(agent, save_path)
        logger.record("training/total_step", total_step)
        logger.dump(step=total_step)
    return agent, buffer
