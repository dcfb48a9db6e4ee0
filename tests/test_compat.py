"""compat/: the reference's module names (gym_control, elegantrl.*, utils.*) on top of pime_b200, so that the reference's
unmodified train.py / run_*_changing.sh drive the library (SURVEY.md 8b).

Host tests: every compat module imports, the agent / env methods the reference's train.py, elegantrl/run.py and utils/
call exist, plus the SB3-style logger.  GPU test: the flow of train.py:main() written against the compat names only, in a
subprocess with PYTHONPATH = repo : compat : compat/_shims.
"""
import csv
import importlib
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
COMPAT = os.path.join(ROOT, "compat")
PATHS = [ROOT, COMPAT, os.path.join(COMPAT, "_shims")]


@pytest.fixture()
def compat_path(monkeypatch):
    for p in reversed(PATHS):
        monkeypatch.syspath_prepend(p)
    # `utils` / `gym` may have been imported from elsewhere by another test: drop stale entries
    for name in [m for m in sys.modules if m.split(".")[0] in ("utils", "gym", "gym_control", "elegantrl", "matplotlib")]:
        monkeypatch.delitem(sys.modules, name, raising=False)
    yield


# names the reference's train.py takes from `from utils.test import *` for the env families on the PIME path (train.py:135-200)
STAR_NAMES = ["test_watertank", "test_ph_integrator", "test_ph", "test_realwatertank", "test_realwatertank_integrator",
              "test_realwatertankobserver", "test_watertankobserver", "test_quadcopter", "test_reacher"]


def test_every_compat_module_imports(compat_path):
    for mod in ["gym", "gym_control", "gym_control.envs", "gym_control.envs.nonlinear_watertank", "gym_control.envs.ph",
                "elegantrl", "elegantrl.logger", "elegantrl.run", "elegantrl.env", "elegantrl.utils", "elegantrl.agent",
                "elegantrl.agent_residual", "elegantrl.net", "elegantrl.net_residual", "elegantrl.replay", "utils.utils",
                "utils.test", "utils.robust_test", "matplotlib.pyplot"]:
        importlib.import_module(mod)
    import gym
    ids = set(gym.envs.registry.env_specs)
    assert len([i for i in ids if i.startswith(("PH1D", "NonLinearWaterTank"))]) == 7          # gym_control/__init__.py:3-142
    t = importlib.import_module("utils.test")
    for n in STAR_NAMES:
        assert callable(getattr(t, n)), n
    u = importlib.import_module("utils.utils")
    assert set(u.MODELS) == set(u.IF_ONPOLICY) == {"td3", "ppo", "sac", "residualintegratormodularppo", "residualppo"}
    with pytest.raises(NotImplementedError):
        u.MODELS["td3"]()


def test_agent_and_env_methods_the_reference_scripts_call_exist(compat_path):
    import pime_b200.gym_api as G
    import pime_b200.rl as R
    # the import statements of the train.py flow (FLOW below) resolve without a GPU
    exec("\n".join(line for line in FLOW.splitlines() if line.startswith(("import ", "from "))), {})
    # the call sites of elegantrl/run.py:train_and_evaluate on the agent and the evaluator
    for name in ("init", "init_residual", "init_actor_zero", "fix_K", "frozen_integrator", "frozen_transfer", "save_load_model",
                 "explore_env", "update_net", "select_action"):
        assert callable(getattr(R.AgentResidualIntegratorModularPPO, name)), name
    # the env API utils/test.py:1056-1067,1369-1407 and utils/robust_test.py use on a deep-copied env
    for name in ("set_state", "set_r", "get_linear_action", "reset", "step", "set_reset_all", "get_changable_parameters",
                 "__deepcopy__"):
        assert callable(getattr(G.NonLinearWaterTankChangingParamUniformGoalIntegrator, name)), name
    for name in ("set_state", "set_r", "set_params", "set_reset_all", "reset", "step", "get_changable_parameters"):
        assert callable(getattr(G.PH1DChangingParamUniformGoalIntegrator, name)), name
    for prop in ("a1", "a2", "Kp", "h1", "h2", "r", "max_step"):      # robust_test.py:12-19 assigns them
        assert getattr(G.NonLinearWaterTankChangingParamUniformGoal, prop).fset is not None, prop


def test_logger_is_sb3_style(tmp_path, compat_path):
    from elegantrl import logger
    from elegantrl.utils import configure_logger
    configure_logger(0, str(tmp_path / "tb"), "PPO-16", True)           # train.py:258-261
    run_dir = logger.get_dir()
    assert os.path.basename(run_dir) == "PPO-16_1"
    logger.record("rollout/ep_rew_mean", -12.5)
    logger.record("train/actor_loss", np.float32(0.25), exclude="tensorboard")   # agent.py:335 passes exclude=
    logger.record("only/stdout", 1.0, exclude=("csv", "tensorboard"))
    assert logger.values["rollout/ep_rew_mean"] == -12.5
    logger.dump(step=0)
    assert logger.values == {}
    logger.record("rollout/ep_rew_mean", -10.0)
    logger.record("training/total_step", 2000)                          # a new key: the csv is rewritten with a wider header
    logger.dump(step=2000)
    rows = list(csv.DictReader(open(os.path.join(run_dir, "progress.csv"))))
    assert [r["step"] for r in rows] == ["0", "2000"]
    assert float(rows[0]["rollout/ep_rew_mean"]) == -12.5 and rows[0]["training/total_step"] == ""
    assert float(rows[1]["training/total_step"]) == 2000 and "only/stdout" not in rows[0]
    assert logger.history[-1]["training/total_step"] == 2000
    if logger.SummaryWriter is not None:
        assert any(f.startswith("events.out.tfevents") for f in os.listdir(run_dir))
    configure_logger(0, str(tmp_path / "tb"), "PPO-16", True)           # the next run of the same name gets the next id
    assert os.path.basename(logger.get_dir()) == "PPO-16_2"
    configure_logger(0, None)                                           # verbose 0, no folder: nothing is written
    logger.record("x", 1.0)
    logger.dump(0)
    assert isinstance(logger.Figure(object(), close=True), logger.Figure)
    logger.close()


def test_preprocess_env_survives_deepcopy_and_pickle_probes():
    """copy / pickle probe dunders on an instance whose __dict__ is still empty (advisor finding, round 1)."""
    import copy
    sys.path.insert(0, ROOT)
    import pime_b200.rl as R

    class FakeSpace:
        shape, high = (3,), np.ones(1)

    class FakeEnv:
        observation_space, action_space, max_step, K = FakeSpace(), FakeSpace(), 7, np.zeros(3)

        def reset(self):
            return np.zeros(3)

    p = R.PreprocessEnv(FakeEnv())
    q = copy.deepcopy(p)
    assert q.max_step == 7 and q.K.shape == (3,) and q.env is not p.env
    with pytest.raises(AttributeError):
        p.no_such_attribute


FLOW = r"""
import os, sys, numpy as np, torch
import matplotlib.pyplot as plt
from utils.utils import MODELS, IF_ONPOLICY
from utils.test import *
from utils.robust_test import robust_test_nonlinear_watertank
import gym, gym_control
from elegantrl.run import Arguments, train_and_evaluate
from elegantrl.env import PreprocessEnv
from elegantrl.utils import configure_logger
from elegantrl import logger
from gym_control.envs.nonlinear_watertank import StackingHistoryPreprocessing
gym.logger.set_level(40)
env_id, algo, out = sys.argv[1], sys.argv[2], sys.argv[3]
env = gym.make(env_id, noise_scale=0., reward_type='distance', r=4.0) if 'NonLinearWaterTank' in env_id else gym.make(env_id)
env.seed(0); np.random.seed(0)
env.target_return = 1e6
kargs = Arguments(if_on_policy=IF_ONPOLICY[algo])
kargs.repeat_times, kargs.gpu_id, kargs.if_remove, kargs.random_seed = 2, 0, False, 0
kargs.env, kargs.env_eval = PreprocessEnv(env=env), PreprocessEnv(env=env)
kargs.net_dim, kargs.batch_size, kargs.target_step = 32, 64, 2 * kargs.env.max_step
kargs.break_step, kargs.eval_times1, kargs.eval_times2, kargs.eval_gap = 2 * kargs.target_step, 2, 3, 1
kargs.fix_K, kargs.frozen_modular_integrator, kargs.frozen_transfer, kargs.test_render_times, kargs.load = True, False, False, kargs.target_step, 'None'
kargs.agent = MODELS[algo]()
configure_logger(0, os.path.join(out, 'tb'), algo, True)
kargs.cwd = os.path.join(out, 'run')
kargs.SCN_kwargs, kargs.Q_kwargs, kargs.if_residual = {}, {}, True
kargs.residual_kwargs = {'init_K': env.K.reshape(-1, 1)} if 'residual' in algo else {}
kargs.Modular_kwargs = {'integrator_dim': env.n_integrator} if 'modular' in algo else {}
if_uniform = 'Uniform' in env_id
if 'NonLinearWaterTankChangingParam' in env_id:
    kargs.test_render = lambda agent, d: [test_watertank(env, agent, d, if_uniform), robust_test_nonlinear_watertank(env, agent, d, if_uniform)]
else:
    kargs.test_render = lambda agent, d: test_ph_integrator(env, agent, d, if_uniform)
agent, _ = train_and_evaluate(kargs)
agent.save_load_model(kargs.cwd, if_save=False)
print('FLOW_OK', sum(p.numel() for p in agent.act.parameters() if p.requires_grad))
env.close()
"""


@pytest.mark.gpu
@pytest.mark.parametrize("env_id,algo", [
    ("NonLinearWaterTankChangingParamUniformGoalStacking10-SquareDistance-v2", "residualppo"),          # run_watertank_changing.sh
    ("PH1DChangingParamUniformGoalIntegrator-SqaureDistance-v35", "residualintegratormodularppo"),       # run_ph_changing.sh
])
def test_train_py_flow_through_compat_names(tmp_path, env_id, algo):
    script = tmp_path / "flow.py"
    script.write_text(FLOW)
    env = dict(os.environ, PYTHONPATH=os.pathsep.join(PATHS))
    res = subprocess.run([sys.executable, str(script), env_id, algo, str(tmp_path)], capture_output=True, text=True, env=env, timeout=600)
    assert res.returncode == 0 and "FLOW_OK" in res.stdout, res.stdout[-2000:] + res.stderr[-4000:]
    run = tmp_path / "run"
    assert (run / "actor.pth").exists() and (run / "step_0" / "staircase.npz").exists()
    rows = list(csv.DictReader(open(next((tmp_path / "tb").glob("*/progress.csv")))))
    assert any(r.get("training/total_step") for r in rows) and "rollout/ep_rew_mean" in rows[0]
    z = np.load(run / "step_0" / "staircase.npz")
    assert np.isfinite(z["agent.actions"]).all()
    if "WaterTank" in env_id:
        assert (run / "step_0" / "robust_test" / "test3" / "params.txt").exists()
        assert z["agent.xs"].shape == (1000, 2) and z["linear.xs"].shape == (1000, 2)
    else:
        assert (run / "step_0" / "robust8" / "params.txt").exists() and z["agent.ys"].shape == (250,)
