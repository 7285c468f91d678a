"""TEST / MEASUREMENT INFRASTRUCTURE ONLY -- never imported by the product (sample_factory_b200/).

Drives the UNMODIFIED reference (alex-petrenko/sample-factory 2.1.3, pip-installed into oracle/_ref by
`__graft_entry__.build()`, oracle/build_ref.py) through its own classes on the host CPU, for `bench.py --impl reference`
and the `cpu_baseline` leg:

    BatchedVectorEnvRunner.{init, update_trajectory_buffers, generate_policy_request, advance_rollouts}
                                                           (algo/sampling/batched_sampling.py:154-388)
    the body of InferenceWorker._handle_policy_steps       (algo/sampling/inference_worker.py:313-341; the worker class
                                                            itself needs a live signal_slot event loop, so its body is
                                                            inlined exactly as tests/golden/make_golden.py does)
    BufferMgr / alloc_trajectory_tensors                   (algo/utils/shared_buffers.py)
    Learner.init / Learner.train                           (algo/learning/learner.py:178-255, 1036-1067)

i.e. serial mode, batched sampling, one worker -- the configuration SURVEY.md section 8d prescribes for the CPU timing.
The five third-party imports the reference makes at module load and that are absent offline (signal_slot, faster_fifo,
colorlog, tensorboardX, gymnasium) come from oracle/ref_shims.py; none of them is on the timed path's arithmetic.
The env is the same synthetic tape env as the GPU arm (oracle.appo_oracle.TapeVecEnv, CPU torch).
"""
from __future__ import annotations

import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF_DIR = os.path.join(ROOT, "oracle", "_ref")


def available() -> bool:
    from oracle import build_ref

    return build_ref.installed(REF_DIR)


def run(n_envs: int, rollout: int, obs_dim: int, num_actions: int, hidden, batch_size: int, num_batches_per_epoch: int,
        num_epochs: int, steps: int, warmup: int, tape_len: int, threads: int, seed: int = 0) -> dict:
    """Time `steps` iterations (one rollout of `rollout` env steps for all `n_envs` envs + Learner.train) after `warmup`."""
    import numpy as np
    import torch

    if ROOT not in sys.path:
        sys.path.insert(0, ROOT)
    from oracle import ref_shims

    ref_shims.install(REF_DIR)
    import gymnasium as gym  # the shim

    from oracle.appo_oracle import TapeVecEnv
    from sample_factory.algo.learning.learner import Learner
    from sample_factory.algo.sampling.batched_sampling import BatchedVectorEnvRunner
    from sample_factory.algo.utils.env_info import extract_env_info
    from sample_factory.algo.utils.make_env import make_env_func_batched
    from sample_factory.algo.utils.model_sharing import ParameterServer
    from sample_factory.algo.utils.rl_utils import prepare_and_normalize_obs
    from sample_factory.algo.utils.shared_buffers import BufferMgr
    from sample_factory.algo.utils.tensor_dict import TensorDict
    from sample_factory.cfg.arguments import default_cfg, preprocess_cfg
    from sample_factory.envs.env_utils import register_env
    from sample_factory.utils.timing import Timing

    torch.set_num_threads(threads)
    torch.manual_seed(seed)
    np.random.seed(seed)
    gen = torch.Generator().manual_seed(seed)
    tape = torch.randn(tape_len, n_envs, obs_dim, generator=gen)
    tape_env = TapeVecEnv(tape, num_actions)

    class RefTapeEnv(gym.Env):
        """TapeVecEnv behind the reference's batched-env contract (algo/utils/make_env.py:147-237)"""

        def __init__(self):
            self.num_agents = tape_env.num_agents
            self.is_multiagent = True
            self.observation_space = gym.spaces.Dict({"obs": gym.spaces.Box(-np.inf, np.inf, (obs_dim,), np.float32)})
            self.action_space = gym.spaces.Discrete(num_actions)

        def reset(self, **kw):
            return {"obs": tape_env.reset().clone()}, {}

        def step(self, actions):
            obs, rew, term, trunc = tape_env.step(torch.as_tensor(actions))
            return {"obs": obs.clone()}, rew, term, trunc, {}

        def close(self):
            pass

    env_name = f"sfb200_bench_tape_{n_envs}"
    register_env(env_name, lambda full_env_name, cfg, env_config, render_mode=None: RefTapeEnv())
    cfg = default_cfg(env=env_name, experiment="sfb200_reference_arm")
    cfg.device = "cpu"
    cfg.serial_mode, cfg.async_rl, cfg.batched_sampling = True, False, True
    cfg.num_workers, cfg.num_envs_per_worker, cfg.worker_num_splits = 1, 1, 1
    cfg.use_rnn, cfg.recurrence = False, 1
    cfg.encoder_mlp_layers = list(hidden)
    cfg.rollout, cfg.batch_size = rollout, batch_size
    cfg.num_batches_per_epoch, cfg.num_epochs = num_batches_per_epoch, num_epochs
    cfg.seed = seed
    cfg.train_dir = "/tmp/sfb200_reference_arm"
    cfg.env_gpu_actions = cfg.env_gpu_observations = False
    cfg.use_env_info_cache = False
    cfg.save_every_sec = 10 ** 9

    tmp_env = make_env_func_batched(cfg, env_config=None)
    env_info = extract_env_info(tmp_env, cfg)
    assert preprocess_cfg(cfg, env_info)
    buffer_mgr = BufferMgr(cfg, env_info)
    policy_versions = buffer_mgr.policy_versions
    learner = Learner(cfg, env_info, policy_versions, 0, ParameterServer(0, policy_versions, cfg.serial_mode))
    learner.init()
    ac = learner.actor_critic
    timing = Timing()
    runner = BatchedVectorEnvRunner(cfg, env_info, 1, 0, 0, buffer_mgr, "cpu", [None])
    runner.init(timing)

    def iteration():
        complete = []
        for _t in range(rollout):
            assert runner.update_trajectory_buffers(timing)
            traj_slice, step = runner.generate_policy_request()[0]
            with torch.no_grad():     # InferenceWorker._handle_policy_steps body (inference_worker.py:313-341)
                obs = TensorDict({k: v[traj_slice, step] for k, v in runner.traj_tensors["obs"].items()})
                rnn_states = runner.traj_tensors["rnn_states"][traj_slice, step]
                if ac.training:
                    ac.eval()
                normalized_obs = prepare_and_normalize_obs(ac, obs)
                policy_outputs = ac(normalized_obs, rnn_states)
                policy_outputs["policy_version"] = torch.empty([n_envs]).fill_(int(policy_versions[0].item()))
                if policy_outputs["actions"].ndim < 2:      # _prepare_policy_outputs_batched :235-269
                    policy_outputs["actions"] = policy_outputs["actions"].unsqueeze(-1)
                for key in runner.policy_output_tensors.keys():
                    runner.policy_output_tensors[key][:] = policy_outputs[key].reshape(runner.policy_output_tensors[key].shape)
            complete, _stats = runner.advance_rollouts(0, timing)
        assert len(complete) == 1
        sl = complete[0]["traj_buffer_idx"]
        learner.train(runner.traj_tensors[sl])
        runner.traj_buffer_queue.put(sl)       # sync mode: the batcher releases the buffers after training

    times = []
    for it in range(warmup + steps):
        t0 = time.perf_counter()
        iteration()
        dt = time.perf_counter() - t0
        if it >= warmup:
            times.append(dt)
    total = sum(times)
    return dict(value=n_envs * rollout * len(times) / total, ms_per_step=1e3 * total / len(times), cores=threads,
                train_step=int(learner.train_step), version="sample-factory 2.1.3 (oracle/_ref)")


def main(argv=None) -> None:
    """python -m oracle.ref_driver --n_envs ... : prints ONE JSON line (last line of stdout) with the timing"""
    import argparse
    import json

    ap = argparse.ArgumentParser()
    for name, default in (("n_envs", 4096), ("rollout", 32), ("obs_dim", 64), ("num_actions", 8), ("batch_size", 32768),
                          ("num_batches_per_epoch", 4), ("num_epochs", 1), ("steps", 3), ("warmup", 1), ("tape_len", 97),
                          ("threads", os.cpu_count() or 1)):
        ap.add_argument(f"--{name}", type=int, default=default)
    ap.add_argument("--hidden", type=int, nargs="*", default=[512, 512])
    a = ap.parse_args(argv)
    r = run(a.n_envs, a.rollout, a.obs_dim, a.num_actions, a.hidden, a.batch_size, a.num_batches_per_epoch, a.num_epochs,
            a.steps, a.warmup, a.tape_len, a.threads)
    print("REF_DRIVER_RESULT " + json.dumps(r), flush=True)


if __name__ == "__main__":
    main()
