"""The Python boundary north_star names: the reference's module paths (`sample_factory.*`) resolve to the device engine, the
model registry exists, plain gymnasium-API envs are adapted automatically, and the reference's own example script
`sf_examples/train_gym_env.py` (BASELINE.json config 1: CartPole-v1) runs UNMODIFIED against this repository.

The example scripts are reference code: they are executed from the reference that __graft_entry__.build() pip-installs into
oracle/_ref (oracle/build_ref.py) -- never copied into the repo."""
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _examples_root():
    ref = os.path.join(ROOT, "oracle", "_ref")
    return ref if os.path.isfile(os.path.join(ref, "sf_examples", "train_gym_env.py")) else None


def _run(args, timeout=600):
    ex = _examples_root()
    env = dict(os.environ, PYTHONPATH=os.pathsep.join([ROOT, ex]))
    return subprocess.run([sys.executable] + args, cwd="/tmp", env=env, capture_output=True, text=True, timeout=timeout)


def test_reference_module_paths_resolve_to_the_engine():
    """every import an sf_examples entry script makes (surveyed over sf_examples/*.py) resolves, to the engine's objects"""
    code = """
import sample_factory, sample_factory_b200.train, sample_factory_b200.cfg, sample_factory_b200.envs
from sample_factory.cfg.arguments import parse_full_cfg, parse_sf_args, checkpoint_override_defaults
from sample_factory.envs.env_utils import register_env, RewardShapingInterface, TrainingInfoInterface
from sample_factory.train import run_rl, make_runner
from sample_factory.enjoy import enjoy
from sample_factory.algo.utils.context import global_model_factory, global_env_registry
from sample_factory.utils.typing import Config, ObsSpace, Env
from sample_factory.model.encoder import Encoder
from sample_factory.model.model_utils import create_mlp, nonlinearity
from sample_factory.algo.utils.torch_utils import calc_num_elements
from sample_factory.algo.utils.gymnasium_utils import convert_space
from sample_factory.utils.utils import str2bool, is_module_available, log
from sample_factory.utils.attr_dict import AttrDict
from sample_factory.pbt.population_based_training import PopulationBasedTraining, perturb_float, policy_cfg_file
from sample_factory.algo.utils.agent_policy_mapping import AgentPolicyMapping
from sample_factory.algo.runners.runner import AlgoObserver, Runner
from sample_factory.algo.utils.misc import EPS, EPISODIC, ExperimentStatus
from sample_factory.algo.utils.rl_utils import make_dones, samples_per_trajectory, total_num_envs
from sample_factory.algo.sampling.sync_sampling_api import SyncSamplingAPI
from sample_factory.eval import do_eval
from sample_factory.utils.algo_version import ALGO_VERSION
from sample_factory.utils.utils import static_vars, project_tmp_dir, safe_ensure_dir_exists, experiment_dir, ensure_dir_exists
from sample_factory.model.utils import orthogonal_init, he_normal_init
from sample_factory.model.model_utils import model_device
from sample_factory.launcher.run_description import Experiment, ParamGrid, RunDescription
from sample_factory.launcher.launcher_utils import seeds
rd = RunDescription("run", [Experiment("exp", "python -m x", ParamGrid([("seed", [1, 2]), (("a", "b"), [(3, 4), (5, 6)])]).generate_params())])
cmds = list(rd.generate_experiments("/tmp/t"))
assert len(cmds) == 4 and cmds[0][0] == "python -m x --seed=1 --a=3 --b=4 --experiment=00_exp_s_1_a_3_b_4 --train_dir=/tmp/t/run/exp", cmds[0]
assert make_dones([True, False], [False, True]) == [True, True] and ExperimentStatus.INTERRUPTED == 2
# observers: hooks of AlgoObserver are called by the runner (only the ones an observer defines)
class Obs(AlgoObserver):
    def __init__(self): self.calls = []
    def on_start(self, runner): self.calls.append("start")
    def on_training_step(self, runner, it): self.calls.append(("step", it))
import sample_factory_b200.multi_policy
cfg = sample_factory_b200.cfg.default_cfg(env="x", experiment="y")
r0 = Runner(cfg); o = Obs(); r0.register_observer(o); r0._notify("on_start"); r0._notify("on_training_step", 3); r0._notify("on_stop")
assert o.calls == ["start", ("step", 3)]
cfg.num_policies = 3
assert isinstance(make_runner(cfg)[1], sample_factory_b200.multi_policy.MultiPolicyRunner)
assert [AgentPolicyMapping(cfg).get_policy_for_agent(0, 0, i) for i in range(4)] == [0, 1, 2, 0]
assert run_rl is sample_factory_b200.train.run_rl and parse_sf_args is sample_factory_b200.cfg.parse_sf_args
register_env("x", lambda *a, **k: None)
assert "x" in global_env_registry() and global_env_registry() is sample_factory_b200.envs.global_env_registry()
print("BOUNDARY_IMPORTS_OK")
"""
    res = subprocess.run([sys.executable, "-c", code], cwd="/tmp", env=dict(os.environ, PYTHONPATH=ROOT), capture_output=True,
                         text=True, timeout=300)
    assert res.returncode == 0 and "BOUNDARY_IMPORTS_OK" in res.stdout, res.stdout[-2000:] + res.stderr[-3000:]


def test_model_registry_api_and_explicit_error():
    """model_factory.py:16-60: registration works (import-time register_* calls of user scripts succeed); a registered
    custom torch module makes the runner refuse with an explicit error instead of silently ignoring it"""
    sys.path.insert(0, ROOT)
    from sample_factory.algo.utils.context import global_model_factory, reset_global_context
    from sample_factory.model.encoder import Encoder
    from sample_factory_b200.model_factory import UnsupportedCustomModel

    reset_global_context()
    mf = global_model_factory()
    mf.check_supported()                       # nothing registered: fine

    class MyEncoder(Encoder):
        def __init__(self, cfg, obs_space):
            super().__init__(cfg)

        def get_out_size(self):
            return 7

    mf.register_encoder_factory(lambda cfg, obs_space: MyEncoder(cfg, obs_space))
    assert global_model_factory().make_model_encoder_func is not None
    with pytest.raises(UnsupportedCustomModel, match="custom model parts are registered: encoder"):
        global_model_factory().check_supported()
    reset_global_context()
    global_model_factory().check_supported()


def test_gymnasium_fallback_is_a_fallback():
    """the vendored gymnasium stand-in provides what cfg-1 needs and steps aside when a real gymnasium is importable"""
    code = """
import gymnasium as gym, numpy as np
assert getattr(gym, "IS_SFB200_FALLBACK", False), "a real gymnasium is installed: the fallback must not shadow it"
e = gym.make("CartPole-v1")
o, info = e.reset(seed=3)
assert o.shape == (4,) and o.dtype == np.float32 and e.action_space.n == 2 and e.observation_space.shape == (4,)
n = 0
while True:
    o, r, tm, tr, info = e.step(1); n += 1
    if tm or tr: break
assert tm and 5 <= n <= 15 and r == 1.0          # pushing right only: the pole falls within ~10 steps
e = gym.make("CartPole-v1"); e.reset(seed=0)
for t in range(500):
    o, r, tm, tr, _ = e.step(t % 2)
    if tm or tr: break
assert isinstance(gym.spaces.Dict({"obs": gym.spaces.Box(-1, 1, (3,))})["obs"], gym.spaces.Box)
print("GYM_FALLBACK_OK")
"""
    res = subprocess.run([sys.executable, "-c", code], cwd="/tmp", env=dict(os.environ, PYTHONPATH=ROOT), capture_output=True,
                         text=True, timeout=120)
    if "a real gymnasium is installed" in res.stderr:
        pytest.skip("real gymnasium present")
    assert res.returncode == 0 and "GYM_FALLBACK_OK" in res.stdout, res.stdout[-2000:] + res.stderr[-3000:]


@pytest.mark.gpu
def test_sf_examples_train_gym_env_runs_unmodified(tmp_path):
    """BASELINE.json config 1: `python -m sf_examples.train_gym_env --env=CartPole-v1 ...` with the command line of the
    script's own docstring (train_gym_env.py:4), the script taken unmodified from the reference, then
    `python -m sf_examples.enjoy_gym_env` on the checkpoint it wrote."""
    if _examples_root() is None:
        pytest.skip("the reference's sf_examples are not available (oracle/_ref not installed)")
    common = ["--algo=APPO", "--use_rnn=False", "--num_envs_per_worker=20", "--policy_workers_per_policy=2", "--recurrence=1",
              "--with_vtrace=False", "--batch_size=512", "--reward_scale=0.1", "--experiment=example_gym_cartpole-v1",
              "--env=CartPole-v1", f"--train_dir={tmp_path}"]
    res = _run(["-m", "sf_examples.train_gym_env"] + common + ["--save_every_sec=10", "--experiment_summaries_interval=1",
                                                              "--train_for_env_steps=1000000", "--seed=0"])
    assert res.returncode == 0, res.stdout[-3000:] + res.stderr[-3000:]
    assert "Collected {0: " in res.stdout and "FPS" in res.stdout, res.stdout[-2000:]
    ckpt_dir = os.path.join(tmp_path, "example_gym_cartpole-v1", "checkpoint_p0")
    assert os.path.isdir(ckpt_dir) and any(f.endswith(".pth") for f in os.listdir(ckpt_dir))
    # the policy learns: the running mean episode reward printed by the runner rises well above a random policy's ~22
    rewards = [float(line.split("reward ")[1].split()[0]) for line in res.stdout.splitlines() if line.startswith("[sf_b200] env_steps")
               and "reward nan" not in line]
    print("CartPole running mean episode rewards:", rewards)
    assert rewards and max(rewards) > 35.0, rewards
    res = _run(["-m", "sf_examples.enjoy_gym_env"] + common + ["--max_num_episodes=20", "--no_render"])
    # (enjoy() returns (status, avg_reward) like the reference's, so the example's sys.exit(main()) exits non-zero there too)
    assert "avg episode reward" in res.stdout, res.stdout[-3000:] + res.stderr[-3000:]
