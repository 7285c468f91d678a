"""Device rollout sampler: the reference's RolloutWorker + InferenceWorker + BatchedVectorEnvRunner collapsed into one
stream of CUDA kernels (no process tree, no queues, no per-step host sync).

Per env step (reference call stack SURVEY section 3.2):
  generate_policy_request  (batched_sampling.py:374-388)  + obs normalisation (inference_worker.py:326)
        -> sfb200_sampler_pre_step   : traj.obs[:, t] <- obs, traj.rnn_states[:, t] <- rnn, x = normalize(obs)
  actor_critic forward     (actor_critic.py:188-195)
        -> sfb200_linear_act_forward per hidden layer
        -> sfb200_heads_forward      : values, logits, sample, log-prob, policy_version -- written straight into
                                       traj[:, t] (replaces policy_output_tensors staging, inference_worker.py:235-269,
                                       batched_sampling.py:308-311)
  vec_env.step(actions)    (batched_sampling.py:316)      -> the env's own kernel (GPU env) or host round trip
  advance_rollouts part 2  (batched_sampling.py:319-357)  -> sfb200_sampler_post_step
After `rollout` steps: _finalize_trajectories (:289-296) -> obs/rnn at index T.

With a GPU env the whole rollout is a fixed launch sequence, so it is captured once into a CUDA graph and replayed.
"""
from __future__ import annotations

from typing import Dict, List, Optional

import torch
from torch import Tensor

from . import ops
from .model import PolicyModel
from .policy import HeadsPlan, forward_policy
from .rnn_core import RnnCore


class DeviceSampler:
    def __init__(self, cfg, env, model: PolicyModel, traj: Dict[str, Tensor], engine: int = ops.GEMM_SIMT,
                 use_cuda_graph: bool = False, philox_seed: int = 0, record_episodes: bool = False,
                 deterministic: bool = False):
        self.cfg = cfg
        self.env = env
        # argmax / mean actions instead of draws (enjoy.py:165-171 eval_deterministic)
        self.deterministic = deterministic
        # obs dict entry "action_mask" (inference_worker.py:324-331): kept in a static bool [N, A] buffer the heads read
        self.action_mask: Optional[Tensor] = None
        self.model = model
        self.traj = traj
        self.engine = engine
        self.device = model.device
        self.N = env.num_agents
        self.T = cfg.rollout
        spec = model.spec
        assert traj["obs"].shape == (self.N, self.T + 1, spec.obs_dim)
        assert (traj["obs"].dtype == torch.uint8) == spec.obs_uint8
        self.act = ops.ACT[spec.nonlinearity]
        dev = self.device
        f32 = dict(dtype=torch.float32, device=dev)
        # per-step scratch (never reallocated)
        self.x_norm = torch.empty((self.N, spec.obs_dim), **f32)
        self.h = [torch.empty((self.N, h), **f32) for h in spec.hidden]
        if getattr(model, "f16_twins", None) is not None and engine == ops.GEMM_TC_3XTF32:
            # fp16-split form of the GEMM engine: bounds of the activation buffers the per-step GEMMs read (model._register_f16)
            ops.register_operand_bounds(self, [(self.x_norm, model.bound_x)] +
                                        [(self.h[i], model.bound_h[4 * i: 4 * i + 1]) for i in range(len(spec.hidden) - 1)])
        # what env.step() receives (preprocess_actions, batched_sampling.py:30-82): int32 [N] for Discrete, float32 [N, A]
        # for a Box action space
        if spec.continuous:
            self.env_actions = torch.empty((self.N, spec.num_actions), dtype=torch.float32, device=dev)
        elif spec.action_segments:      # Tuple of Discretes: int32 [N, K] (batched_sampling.py:40-41)
            self.env_actions = torch.empty((self.N, len(spec.action_segments)), dtype=torch.int32, device=dev)
        else:
            self.env_actions = torch.empty(self.N, dtype=torch.int32, device=dev)
        self.heads_plan = HeadsPlan(model, engine, self.N)
        self.last_rnn_state = torch.zeros((self.N, traj["rnn_states"].shape[2]), **f32)
        self.rnn: Optional[RnnCore] = None
        if spec.use_rnn:
            assert traj["rnn_states"].shape[2] == spec.rnn_state_size
            self.rnn = RnnCore(model, engine)
            self.rnn_step_bufs = self.rnn.alloc_step(self.N)
            self.new_rnn_state = torch.zeros((self.N, spec.rnn_state_size), **f32)
        # policy version lives on the device so a captured graph always stamps the current one (inference_worker.py:332)
        self.policy_version = torch.zeros(1, **f32)
        # episode accounting on device (batched_sampling.py:201-204, :215-287)
        self.ep_return = torch.zeros(self.N, **f32)
        self.ep_len = torch.zeros(self.N, dtype=torch.int32, device=dev)
        self.ep_min_raw = torch.full((self.N,), float("inf"), **f32)
        self.ep_max_raw = torch.full((self.N,), float("-inf"), **f32)
        self.episode_stats = torch.zeros(8, dtype=torch.float64, device=dev)
        # optional per-episode report (the reference's episodic stats messages, batched_sampling.py:228-234): return /
        # length of the episode that ended at [n, t], NaN / -1 elsewhere
        self.fin_return = torch.full((self.N, self.T), float("nan"), **f32) if record_episodes else None
        self.fin_len = torch.full((self.N, self.T), -1, dtype=torch.int32, device=dev) if record_episodes else None
        self.last_obs: Optional[Tensor] = None
        self.philox_seed = philox_seed
        self.step_counter = torch.zeros(1, dtype=torch.int64, device=dev)  # policy steps taken = Philox offset
        self.noise: Optional[Tensor] = None  # [T, N, A] explicit Exp(1) noise (parity tests); None -> Philox
        self.use_cuda_graph = use_cuda_graph and getattr(env, "is_gpu_env", False)
        self._graph: Optional[torch.cuda.CUDAGraph] = None
        # host envs: the env step is a host round trip, but the device work on either side of it is a fixed launch
        # sequence per rollout step -> one small CUDA graph before and one after every env.step()
        self.use_step_graphs = (use_cuda_graph and not getattr(env, "is_gpu_env", False)
                                and getattr(env, "static_outputs", False))
        self._step_graphs = None
        self._merged_graphs = None
        self._eager_rollouts = 0
        self.kernel_launches_per_rollout = 0
        # Fused step tail (csrc/heads.cu sampler_tail_tape_kernel): for the synthetic tape env the heads' finishing step,
        # the env step, post-step(t) and pre-step(t+1) are ONE launch.  Needs the fused-partials heads path, a plain Discrete
        # action space, float32 observations, no recurrent core and an env whose step is the tape rule.  SFB200_TAIL_FUSED=0
        # restores the separate launches.
        import os

        from .envs import TapeVecEnv
        self.fused_tail = (os.environ.get("SFB200_TAIL_FUSED", "1") != "0" and type(env) is TapeVecEnv and
                           not env.continuous and not env.action_segments and not env.with_action_mask and
                           not env.obs_uint8 and self.rnn is None and self.heads_plan.P > 0 and
                           not self.heads_plan.separate and
                           not spec.continuous and not spec.action_segments)
        # Whole rollout as ONE persistent kernel (csrc/rollout_fused.cu): clusters of H2/128 CTAs own a 128-env row block for
        # all T steps.  Same conditions as the fused tail plus a two-layer MLP the kernel covers.  SFB200_ROLLOUT_FUSED=0
        # restores the per-step launches.
        self.fused_rollout = False
        if (self.fused_tail and os.environ.get("SFB200_ROLLOUT_FUSED", "1") != "0" and not deterministic and
                len(spec.fc_encoder_layers) == 2 and not spec.decoder_mlp_layers and self.heads_plan.conv is None):
            (W1, _), (W2, _) = model.encoder_layers()
            self.fused_rollout = ops.rollout_mlp2_partials(W1, W2, spec.num_linear_action_outputs, engine) == self.heads_plan.P

    # ------------------------------------------------------------------------------------------------------------
    def _take_obs(self, obs):
        """Envs may return the observation tensor or the reference's obs dict {"obs": ..., "action_mask": [N, A]}; the
        mask (any dtype, 0 = not allowed) is popped like the inference worker does and never reaches the model."""
        if not isinstance(obs, dict):
            return obs
        mask = obs.get("action_mask")
        if mask is not None:
            spec = self.model.spec
            if spec.continuous or spec.action_segments:
                raise NotImplementedError("action masks are supported for plain Discrete action spaces only")
            if self.action_mask is None:
                self.action_mask = torch.empty((self.N, spec.num_actions), dtype=torch.bool, device=self.device)
            torch.ne(mask.view(self.N, spec.num_actions), 0, out=self.action_mask)
        return obs["obs"]

    def reset(self) -> None:
        self.last_obs = self._take_obs(self.env.reset())
        self.last_rnn_state.zero_()

    def set_policy_version(self, version: int) -> None:
        self.policy_version.fill_(float(version))

    def _pre_step(self, t: int) -> None:
        """generate_policy_request (batched_sampling.py:374-388) + inference-side normalisation for step t."""
        m, spec, tr = self.model, self.model.spec, self.traj
        mean = m.obs_mean if spec.normalize_input else None
        var = m.obs_var if spec.normalize_input else None
        ops.sampler_pre_step(self.last_obs, tr["obs"][:, t], self.last_rnn_state, tr["rnn_states"][:, t], self.x_norm,
                             mean, var, spec.obs_subtract_mean, 1.0 / spec.obs_scale)

    def _policy_step(self, t: int, fused_tail: bool = False) -> None:
        """policy forward + sampling on the pre-step's x_norm; outputs go straight into traj[:, t].  fused_tail: the same
        launch that finishes the heads also steps the tape env and runs post-step(t) + pre-step(t+1)."""
        cfg, m, spec, tr = self.cfg, self.model, self.model.spec, self.traj
        rnn_fn = None
        if self.rnn is not None:   # ModelCoreRNN.forward (core.py:37-64), one step
            rnn_fn = lambda head: self.rnn.step(head, self.last_rnn_state, self.new_rnn_state, self.rnn_step_bufs)
        noise_t = None if self.noise is None else self.noise[t]
        heads_kwargs = dict(
            values=tr["values"][:, t], values_stride=tr["values"].stride(0),
            logits=tr["action_logits"][:, t], logits_stride=tr["action_logits"].stride(0),
            noise=noise_t, philox_seed=self.philox_seed, philox_offset=0, philox_offset_dev=self.step_counter,
            actions_f32=tr["actions"][:, t], actions_stride=tr["actions"].stride(0),
            env_actions=self.env_actions,
            log_prob=tr["log_prob_actions"][:, t], log_prob_stride=tr["log_prob_actions"].stride(0),
            policy_version_scalar=self.policy_version,
            policy_version_out=tr["policy_version"][:, t], pv_stride=tr["policy_version"].stride(0),
        )
        # the sampler never needs the last hidden activation again: with the fused path it is not written to HBM
        special = self.action_mask is not None or self.deterministic
        if special:
            ops.set_sampling_mode(self.action_mask, self.deterministic)
        finish_fn = None
        if fused_tail:
            last = t + 1 == self.T
            env = self.env

            def finish_fn(part, P, M, bv, ba):
                ops.sampler_tail_tape_step(
                    part, P, M, bv, ba, values=tr["values"][:, t], values_stride=tr["values"].stride(0),
                    logits=tr["action_logits"][:, t], logits_stride=tr["action_logits"].stride(0), noise=noise_t,
                    philox_seed=self.philox_seed, sampler_step=self.step_counter, actions_f32=tr["actions"][:, t],
                    actions_stride=tr["actions"].stride(0), env_actions=self.env_actions,
                    log_prob=tr["log_prob_actions"][:, t], log_prob_stride=tr["log_prob_actions"].stride(0),
                    policy_version_scalar=self.policy_version, policy_version_out=tr["policy_version"][:, t],
                    pv_stride=tr["policy_version"].stride(0), env=env, reward_scale=cfg.reward_scale,
                    reward_clip=cfg.reward_clip, policy_id=cfg.policy_id, traj_rewards=tr["rewards"][:, t],
                    traj_dones=tr["dones"][:, t], traj_time_outs=tr["time_outs"][:, t], traj_policy_id=tr["policy_id"][:, t],
                    ep_return=self.ep_return, ep_len=self.ep_len, ep_min_raw=self.ep_min_raw, ep_max_raw=self.ep_max_raw,
                    len_increment=cfg.env_frameskip if cfg.summaries_use_frameskip else 1, stats=self.episode_stats,
                    fin_return=None if self.fin_return is None else self.fin_return[:, t],
                    fin_len=None if self.fin_len is None else self.fin_len[:, t], traj_obs_next=tr["obs"][:, t + 1],
                    rnn=self.last_rnn_state, traj_rnn_next=tr["rnn_states"][:, t + 1], x_norm=None if last else self.x_norm,
                    mean=m.obs_mean if spec.normalize_input else None, var=m.obs_var if spec.normalize_input else None,
                    sub_mean=spec.obs_subtract_mean, inv_scale=1.0 / spec.obs_scale)

        try:
            forward_policy(m, self.x_norm, self.h, self.act, self.engine, self.heads_plan, heads_kwargs, rnn_fn,
                           store_tail=False, finish_fn=finish_fn)
        finally:
            if special:
                ops.set_sampling_mode(None, False)

    def _env_and_post_step(self, t: int) -> None:
        obs, rew, terminated, truncated = self.env.step(self.env_actions)   # batched_sampling.py:316
        self.last_obs = self._take_obs(obs)
        self._post_step(t, rew, terminated, truncated)
        self._mask_inactive(t)

    def _mask_inactive(self, t: int) -> None:
        inactive = getattr(self.env, "inactive", None)
        if inactive is not None:      # multi-agent host envs: steps of inactive agents carry policy id -1 (masked by the learner)
            self.traj["policy_id"][:, t].masked_fill_(inactive, -1)

    def _post_step(self, t: int, rew: Tensor, terminated: Tensor, truncated: Tensor) -> None:
        """advance_rollouts part 2 for step t, then the pre-step of t+1 (or, at t = T-1, _finalize_trajectories
        batched_sampling.py:289-296: obs / rnn state recorded at index T).  Without a recurrent core both halves only
        consume the env's outputs -> one fused launch."""
        cfg, m, spec, tr = self.cfg, self.model, self.model.spec, self.traj
        post_args = (rew, terminated, truncated, cfg.reward_scale, cfg.reward_clip, cfg.policy_id,
                     tr["rewards"][:, t], tr["dones"][:, t], tr["time_outs"][:, t], tr["policy_id"][:, t],
                     self.ep_return, self.ep_len, self.ep_min_raw, self.ep_max_raw,
                     cfg.env_frameskip if cfg.summaries_use_frameskip else 1, self.episode_stats,
                     self.step_counter,
                     None if self.fin_return is None else self.fin_return[:, t],
                     None if self.fin_len is None else self.fin_len[:, t])
        last = t + 1 == self.T
        if self.rnn is None:
            # non-recurrent core: new_rnn_states == rnn_states (core.py:76-77), times (1-done) stays zero
            mean = m.obs_mean if spec.normalize_input else None
            var = m.obs_var if spec.normalize_input else None
            ops.sampler_post_pre_step(*post_args, obs=self.last_obs, traj_obs_next=tr["obs"][:, t + 1],
                                      rnn=self.last_rnn_state, traj_rnn_next=tr["rnn_states"][:, t + 1],
                                      x_norm=None if last else self.x_norm, mean=mean, var=var,
                                      sub_mean=spec.obs_subtract_mean, inv_scale=1.0 / spec.obs_scale)
            return
        ops.sampler_post_step(*post_args)
        # last_rnn_state = new_rnn_states * (1 - done)  (batched_sampling.py:332-335); the dones were just written
        ops.mask_rows(self.new_rnn_state, self.last_rnn_state, tr["dones"][:, t])
        if last:
            self._finalize_trajectories()
        else:
            self._pre_step(t + 1)

    def advance_rollouts(self, t: int) -> None:
        """One env step for all envs: policy step then env step (reference: inference then advance_rollouts)."""
        if self.fused_tail and self.last_obs is self.env.obs:
            self._policy_step(t, fused_tail=True)      # heads + env step + post-step(t) + pre-step(t+1): one launch
            return
        self._policy_step(t)
        self._env_and_post_step(t)

    def _finalize_trajectories(self) -> None:
        tr = self.traj
        if self.last_obs.dtype == torch.float32:
            ops.copy_rows(self.last_obs, tr["obs"][:, self.T])                   # batched_sampling.py:292
        else:
            tr["obs"][:, self.T].copy_(self.last_obs)                            # uint8 frames (recurrent path only)
        ops.copy_rows(self.last_rnn_state, tr["rnn_states"][:, self.T])          # :293

    def _rollout_persistent(self) -> None:
        """pre-step(0) + ONE kernel for the T steps of the rollout"""
        cfg, m, spec = self.cfg, self.model, self.model.spec
        (W1, b1), (W2, b2) = m.encoder_layers()
        Wv, bv = m.critic
        Wa, ba = m.actor
        assert self.noise is None or (self.noise.is_contiguous() and self.noise.shape[0] >= self.T)
        ops.rollout_mlp2_tape(
            self.T, W1, b1, W2, b2, self.act, self.engine, Wv, bv, Wa, ba, self.h[0], self.heads_plan.part, self.x_norm,
            self.traj, self.env, self.noise, self.philox_seed, self.step_counter, self.env_actions, self.policy_version,
            cfg.reward_scale, cfg.reward_clip, cfg.policy_id, self.ep_return, self.ep_len, self.ep_min_raw, self.ep_max_raw,
            cfg.env_frameskip if cfg.summaries_use_frameskip else 1, self.episode_stats, self.fin_return, self.fin_len,
            self.last_rnn_state, m.obs_mean if spec.normalize_input else None, m.obs_var if spec.normalize_input else None,
            spec.obs_subtract_mean, 1.0 / spec.obs_scale)

    def _rollout_eager(self) -> None:
        n0 = ops.launch_count()
        self._pre_step(0)
        if self.fused_rollout and self.action_mask is None and self.last_obs is self.env.obs:
            self._rollout_persistent()
        else:
            for t in range(self.T):
                self.advance_rollouts(t)
        self.kernel_launches_per_rollout = ops.launch_count() - n0   # counted by the library itself

    def rollout(self) -> None:
        """Collect `rollout` steps for every env into the trajectory buffers (in place)."""
        if self.last_obs is None:
            self.reset()
        if self.use_step_graphs:
            self._rollout_step_graphs()
            return
        if not self.use_cuda_graph:
            self._rollout_eager()
            return
        if self._graph is None:
            # the Philox offset and the env step are device-side counters, so replays draw fresh noise
            assert self.noise is None, "explicit noise and CUDA graphs are mutually exclusive"
            torch.cuda.synchronize()
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                self._rollout_eager()   # warm-up on the side stream (allocator-free path, but be safe)
            torch.cuda.current_stream().wait_stream(side)
            torch.cuda.synchronize()
            # the capture bakes in the address of the observation tensor step 0 reads: a device env must hand out the SAME
            # tensors from every step() / reset() (ADVICE r1) -- otherwise fall back to eager launches instead of replaying
            # stale pointers
            obs_ptr = self.last_obs.data_ptr()
            self._graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(self._graph):
                self._rollout_eager()
            if self.last_obs.data_ptr() != obs_ptr:
                print("[sf_b200] the env returns fresh observation tensors from step(): rollout CUDA graph disabled "
                      "(expose static output buffers to enable it)", flush=True)
                self._graph = None
                self.use_cuda_graph = False
                self._rollout_eager()
                return
            self._graph_launches = self.kernel_launches_per_rollout
        self._graph.replay()
        self.kernel_launches_per_rollout = self._graph_launches

    def _rollout_step_graphs(self) -> None:
        """Host-env rollout: graph(policy step t) -> env.step (host) -> graph(post step t)."""
        assert self.noise is None, "explicit noise and CUDA graphs are mutually exclusive"
        if self._eager_rollouts < 1:       # first rollout eager: warms up every kernel (attributes, module load)
            self._rollout_eager()
            self._eager_rollouts += 1
            return
        if all(hasattr(self.env, a) for a in ("enqueue_actions_d2h", "mark_actions_enqueued", "step_wait")):
            self._rollout_merged_graphs()
            return
        if self._step_graphs is None:
            self._capture_step_graph_pairs()
        for t in range(self.T):
            gp, gq = self._step_graphs[t]
            gp.replay()
            obs, _, _, _ = self.env.step(self.env_actions)
            assert self._take_obs(obs) is self.last_obs
            gq.replay()
        self.kernel_launches_per_rollout = self._graph_launches

    def _rollout_merged_graphs(self) -> None:
        """Host envs whose step() splits into "enqueue the D2H copy of the actions" / "wait, simulate, enqueue the H2D copies":
        ONE graph per env step = post-step(t) + policy step(t+1) + the actions' D2H copy (pinned staging buffer: static
        pointers), so the host issues one replay, one event record and the env's own copies per step."""
        env, T = self.env, self.T
        if self._merged_graphs is None:
            assert self.last_obs is env.obs, "host env must expose static output buffers (obs/rew/terminated/truncated)"
            torch.cuda.synchronize()
            n0 = ops.launch_count()
            first, last = torch.cuda.CUDAGraph(), torch.cuda.CUDAGraph()
            with torch.cuda.graph(first):
                self._pre_step(0)
                self._policy_step(0)
                env.enqueue_actions_d2h(self.env_actions)
            mids = []
            for t in range(T - 1):
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g):
                    self._post_step(t, env.rew, env.terminated, env.truncated)
                    self._mask_inactive(t)
                    self._policy_step(t + 1)
                    env.enqueue_actions_d2h(self.env_actions)
                mids.append(g)
            with torch.cuda.graph(last):
                self._post_step(T - 1, env.rew, env.terminated, env.truncated)
                self._mask_inactive(T - 1)
            self._merged_graphs = (first, mids, last)
            self._graph_launches = ops.launch_count() - n0
        first, mids, last = self._merged_graphs
        first.replay()
        env.mark_actions_enqueued()
        for t in range(T):
            obs, _, _, _ = env.step_wait()
            assert self._take_obs(obs) is self.last_obs
            if t + 1 < T:
                mids[t].replay()
                env.mark_actions_enqueued()
            else:
                last.replay()
        self.kernel_launches_per_rollout = self._graph_launches

    def _capture_step_graph_pairs(self) -> None:
        if True:
            env = self.env
            assert self.last_obs is env.obs, "host env must expose static output buffers (obs/rew/terminated/truncated)"
            torch.cuda.synchronize()
            n0 = ops.launch_count()
            graphs = []
            for t in range(self.T):
                gp, gq = torch.cuda.CUDAGraph(), torch.cuda.CUDAGraph()
                with torch.cuda.graph(gp):
                    if t == 0:
                        self._pre_step(0)
                    self._policy_step(t)
                with torch.cuda.graph(gq):
                    self._post_step(t, env.rew, env.terminated, env.truncated)
                    self._mask_inactive(t)
                graphs.append((gp, gq))
            self._step_graphs = graphs
            self._graph_launches = ops.launch_count() - n0

    @property
    def graph_replay_launches(self) -> int:
        """Kernel launches per rollout that happen through graph replay (not seen by the library's launch counter)."""
        if self._graph is not None or self._step_graphs is not None or self._merged_graphs is not None:
            return self._graph_launches
        return 0

    def finished_episodes(self):
        """(returns, lengths) of the episodes that ended during the LAST rollout, in (step, env) order -- host sync."""
        assert self.fin_return is not None, "construct the sampler with record_episodes=True"
        ret, ln = self.fin_return.t().cpu().numpy(), self.fin_len.t().cpu().numpy()
        m = ln >= 0
        return ret[m], ln[m]

    def pop_episode_stats(self) -> Dict[str, float]:
        """Aggregate of episodes finished since the last call (host sync; call at reporting time only)."""
        s = self.episode_stats.cpu().tolist()
        self.episode_stats.zero_()
        n = s[0]
        if n <= 0:
            return dict(episodes=0)
        return dict(episodes=int(n), reward=s[1] / n, len=s[2] / n, min_raw_reward=s[3] / n, max_raw_reward=s[4] / n)


class SplitSampler:
    """The reference's double-buffered sampling (cfg.worker_num_splits, rollout_worker.py:97-143, "while one group of
    envs waits for actions the other one is stepping"): the env instances of a worker are split into groups that advance
    independently.  Here every group is a DeviceSampler over its own env instance and its own ROW RANGE of the shared
    trajectory buffers, and the groups' per-step kernel chains run concurrently on separate CUDA streams (fork / join
    captured into ONE graph).  A 4096-env policy step is latency-bound (five dependent kernels moving 2 MB), so two
    2048-env chains in flight use the idle SMs instead of waiting on each other."""

    def __init__(self, cfg, envs: List, model: PolicyModel, traj: Dict[str, Tensor], engine: int = ops.GEMM_SIMT,
                 use_cuda_graph: bool = False, philox_seed: int = 0, record_episodes: bool = False):
        assert len(envs) >= 2
        self.cfg, self.model, self.traj = cfg, model, traj
        self.subs: List[DeviceSampler] = []
        lo = 0
        for s, env in enumerate(envs):
            n = env.num_agents
            view = {k: v[lo: lo + n] for k, v in traj.items()}
            self.subs.append(DeviceSampler(cfg, env, model, view, engine=engine, use_cuda_graph=False,
                                           philox_seed=philox_seed + 7919 * s, record_episodes=record_episodes))
            lo += n
        self.N, self.T = lo, cfg.rollout
        assert traj["obs"].shape[0] == self.N
        self.env = envs[0]
        self.side_streams = [torch.cuda.Stream(device=model.device) for _ in envs[1:]]
        self.use_cuda_graph = use_cuda_graph and all(getattr(e, "is_gpu_env", False) for e in envs)
        # host envs that can split step() into step_async / step_wait: step-interleaved double buffering
        self.host_interleaved = (not any(getattr(e, "is_gpu_env", False) for e in envs) and
                                 all(hasattr(e, "step_async") and hasattr(e, "step_wait") for e in envs))
        if self.host_interleaved and use_cuda_graph:
            for sub in self.subs:          # the per-step graphs of the host-env path (DeviceSampler._rollout_step_graphs)
                sub.use_step_graphs = (getattr(sub.env, "static_outputs", False) and sub.noise is None)
        self._graph: Optional[torch.cuda.CUDAGraph] = None
        self._graph_launches = 0
        self.kernel_launches_per_rollout = 0

    # ---- the DeviceSampler surface the runner / bench use ------------------------------------------------------
    def reset(self) -> None:
        for s in self.subs:
            s.reset()

    def set_policy_version(self, version: int) -> None:
        for s in self.subs:
            s.set_policy_version(version)

    @property
    def noise(self):
        return None

    @noise.setter
    def noise(self, value: Optional[Tensor]) -> None:
        """[T, N, A] explicit sampling noise (parity tests), cut into the groups' row ranges"""
        lo = 0
        for s in self.subs:
            s.noise = None if value is None else value[:, lo: lo + s.N].contiguous()
            lo += s.N

    def _rollout_all(self) -> None:
        main = torch.cuda.current_stream()
        n0 = ops.launch_count()
        for sub, st in zip(self.subs[1:], self.side_streams):      # fork
            st.wait_stream(main)
            with torch.cuda.stream(st):
                sub._rollout_eager()
        self.subs[0]._rollout_eager()
        for st in self.side_streams:                               # join
            main.wait_stream(st)
        self.kernel_launches_per_rollout = ops.launch_count() - n0

    def _rollout_host_interleaved(self) -> None:
        """Double-buffered sampling over HOST env groups (rollout_worker.py:97-143: "while one group of envs waits for actions
        the other one is stepping"): group g's GPU work -- results H2D, post-step(t), policy step(t+1), actions D2H -- runs on
        its own stream while the host waits for and steps the next group.  Same per-step launches (or per-step graphs) as the
        single-group path; only the order in which the host issues them changes."""
        main = torch.cuda.current_stream()
        streams = [main] + self.side_streams
        T = self.T
        graphs = [sub._step_graphs for sub in self.subs]

        def policy(sub, g, t):
            if graphs[g] is not None:
                graphs[g][t][0].replay()
            else:
                if t == 0:
                    sub._pre_step(0)
                sub._policy_step(t)
            sub.env.step_async(sub.env_actions)

        for st in self.side_streams:
            st.wait_stream(main)
        n0 = ops.launch_count()
        for g, sub in enumerate(self.subs):
            with torch.cuda.stream(streams[g]):
                policy(sub, g, 0)
        for t in range(T):
            for g, sub in enumerate(self.subs):
                with torch.cuda.stream(streams[g]):
                    obs, rew, term, trunc = sub.env.step_wait()
                    sub.last_obs = sub._take_obs(obs)
                    if graphs[g] is not None:
                        graphs[g][t][1].replay()
                    else:
                        sub._post_step(t, rew, term, trunc)
                        sub._mask_inactive(t)
                    if t + 1 < T:
                        policy(sub, g, t + 1)
        for st in self.side_streams:
            main.wait_stream(st)
        n = ops.launch_count() - n0
        self.kernel_launches_per_rollout = n if n else sum(s._graph_launches for s in self.subs)

    def rollout(self) -> None:
        if any(s.last_obs is None for s in self.subs):
            self.reset()
        if self.host_interleaved:
            if any(s.use_step_graphs and s._step_graphs is None for s in self.subs):
                if any(s._eager_rollouts < 1 for s in self.subs):
                    for s in self.subs:        # first rollout: every group eager, one after the other (kernel warm-up)
                        s._rollout_eager()
                        s._eager_rollouts += 1
                    self.kernel_launches_per_rollout = sum(s.kernel_launches_per_rollout for s in self.subs)
                    return
                for s in self.subs:            # then capture the groups' per-step graph pairs (nothing executes here)
                    s._capture_step_graph_pairs()
            self._rollout_host_interleaved()
            return
        if not self.use_cuda_graph:
            self._rollout_all()
            return
        if self._graph is None:
            assert all(s.noise is None for s in self.subs), "explicit noise and CUDA graphs are mutually exclusive"
            torch.cuda.synchronize()
            warm = torch.cuda.Stream()
            warm.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(warm):
                self._rollout_all()            # warm-up (kernel attributes, module load) outside the capture
            torch.cuda.current_stream().wait_stream(warm)
            torch.cuda.synchronize()
            self._graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(self._graph):
                self._rollout_all()
            self._graph_launches = self.kernel_launches_per_rollout
        self._graph.replay()
        self.kernel_launches_per_rollout = self._graph_launches

    @property
    def graph_replay_launches(self) -> int:
        if self.host_interleaved:
            return sum(s.graph_replay_launches for s in self.subs)
        return self._graph_launches if self._graph is not None else 0

    def pop_episode_stats(self) -> Dict[str, float]:
        tot = torch.stack([s.episode_stats for s in self.subs]).sum(0).cpu().tolist()
        for s in self.subs:
            s.episode_stats.zero_()
        n = tot[0]
        if n <= 0:
            return dict(episodes=0)
        return dict(episodes=int(n), reward=tot[1] / n, len=tot[2] / n, min_raw_reward=tot[3] / n, max_raw_reward=tot[4] / n)
