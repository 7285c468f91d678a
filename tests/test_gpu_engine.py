"""End-to-end parity of the device engine (DeviceSampler + Learner, through the C ABI) against
  (a) the committed golden vectors produced by the reference itself (tests/golden/*.npz), and
  (b) the CPU oracle on larger seeded inputs,
plus size-independent properties at BASELINE.json's full size (N=4096, T=32)."""
import numpy as np
import pytest
import torch

from oracle import appo_oracle as O
from tests.golden_utils import load_case, state_from, traj_from

pytestmark = pytest.mark.gpu
TOL = 1e-5


def make_cfg(ocfg: O.OracleCfg, **over):
    from sample_factory_b200.cfg import default_cfg

    cfg = default_cfg()
    for k in ["rollout", "recurrence", "batch_size", "num_batches_per_epoch", "num_epochs", "gamma", "gae_lambda",
              "ppo_clip_ratio", "ppo_clip_value", "exploration_loss_coeff", "value_loss_coeff", "kl_loss_coeff",
              "max_grad_norm", "learning_rate", "adam_eps", "adam_beta1", "adam_beta2", "normalize_input",
              "normalize_returns", "value_bootstrap", "with_vtrace", "vtrace_rho", "vtrace_c", "reward_scale",
              "reward_clip", "max_policy_lag", "nonlinearity", "obs_subtract_mean", "obs_scale", "use_rnn", "rnn_type",
              "rnn_size", "adaptive_stddev", "continuous_tanh_scale", "initial_stddev", "exploration_loss", "optimizer", "actor_critic_share_weights"]:
        setattr(cfg, k, getattr(ocfg, k))
    cfg.encoder_mlp_layers = list(ocfg.encoder_mlp_layers)
    cfg.decoder_mlp_layers = list(ocfg.decoder_mlp_layers)
    cfg.encoder_conv_architecture = ocfg.encoder_conv_architecture
    cfg.encoder_conv_mlp_layers = list(ocfg.encoder_conv_mlp_layers)
    cfg.async_rl = False
    for k, v in over.items():
        setattr(cfg, k, v)
    return cfg


def build(ocfg: O.OracleCfg, N: int, state, tape, dev, engine="simt", graph=False):
    from sample_factory_b200 import ops
    from sample_factory_b200.envs import TapeVecEnv
    from sample_factory_b200.learner import Learner
    from sample_factory_b200.model import ModelSpec, PolicyModel
    from sample_factory_b200.sampler import DeviceSampler
    from sample_factory_b200.trajectory import alloc_for_spec

    ops.bind_device(dev)
    cfg = make_cfg(ocfg)
    spec = ModelSpec(ocfg.obs_dim, ocfg.num_actions, list(ocfg.encoder_mlp_layers), list(ocfg.decoder_mlp_layers),
                     ocfg.nonlinearity, ocfg.normalize_input, ocfg.normalize_returns, ocfg.obs_subtract_mean,
                     ocfg.obs_scale, ocfg.use_rnn, ocfg.rnn_type, ocfg.rnn_size, continuous=ocfg.continuous,
                     adaptive_stddev=ocfg.adaptive_stddev, continuous_tanh_scale=ocfg.continuous_tanh_scale,
                     initial_stddev=ocfg.initial_stddev, obs_shape=ocfg.obs_shape,
                     encoder_conv_architecture=ocfg.encoder_conv_architecture,
                     encoder_conv_mlp_layers=list(ocfg.encoder_conv_mlp_layers), obs_uint8=tape.dtype == torch.uint8,
                     action_segments=ocfg.action_segments, share_weights=ocfg.actor_critic_share_weights)
    model = PolicyModel(spec, dev)
    model.load_state_dict(state, strict=False)
    traj = alloc_for_spec(spec, N, ocfg.rollout, dev)
    env = TapeVecEnv(tape.to(dev).contiguous(), ocfg.num_actions, continuous=ocfg.continuous, obs_shape=ocfg.obs_shape,
                     action_segments=ocfg.action_segments, with_action_mask=ocfg.action_mask)
    sampler = DeviceSampler(cfg, env, model, traj, engine=ops.ENGINES[engine], use_cuda_graph=graph)
    learner = Learner(cfg, model, N, engine=ops.ENGINES[engine])
    return cfg, model, traj, env, sampler, learner


def upload_traj(traj_dev, traj_cpu):
    for k, v in traj_cpu.items():
        traj_dev[k].copy_(v.view(traj_dev[k].shape))


ENGINES = ["simt", "3xtf32"]


def _need(engine):
    from sample_factory_b200 import ops

    if engine != "simt" and not ops.tc_available():
        pytest.skip("tcgen05 engine not available")


GOLDEN_CASES = ["tiny_gae", "tiny_vtrace", "tiny_gru", "tiny_lstm", "cfg2_small", "tiny_gauss", "tiny_gauss_adaptive", "tiny_conv", "tiny_symkl", "tiny_lamb", "tiny_tuple", "tiny_separate", "tiny_mask"]


@pytest.mark.parametrize("engine", ENGINES)
@pytest.mark.parametrize("name", GOLDEN_CASES)
def test_rollout_matches_reference_golden(name, engine):
    """Sampler vs the REFERENCE's own trajectories (same weights, same obs tape, same Exp(1) noise)."""
    _need(engine)
    dev = torch.device("cuda", 0)
    z, meta, ocfg = load_case(name)
    tape = torch.from_numpy(z["tape"])
    cfg, model, traj, env, sampler, learner = build(ocfg, meta["N"], state_from(z, "init/"), tape, dev, engine=engine)
    sampler.reset()
    for it in range(meta["iters"]):
        st = state_from(z, "init/") if it == 0 else state_from(z, f"it{it - 1}/state/")
        model.load_state_dict(st, strict=False)
        sampler.set_policy_version(int(z[f"it{it}/train_step_before"]))
        sampler.noise = torch.from_numpy(z[f"it{it}/noise"]).to(dev).contiguous()
        sampler.rollout()
        poisoned = meta["poison"] and it == meta["iters"] - 1
        got = {k: v.cpu() for k, v in traj.items()}
        ref = {k: torch.from_numpy(z[f"it{it}/traj/{k}"]) for k in
               ["obs", "actions", "action_logits", "log_prob_actions", "values", "policy_version", "rewards", "dones",
                "time_outs", "policy_id", "rnn_states"]}
        for k in ["obs", "rewards", "dones", "time_outs"]:
            if k == "rewards" and ocfg.continuous:   # reward = f(float action): tolerance, not bit-exactness
                np.testing.assert_allclose(got[k].numpy(), ref[k].numpy(), atol=TOL)
                continue
            assert torch.equal(got[k].view(ref[k].shape), ref[k]), k
        np.testing.assert_allclose(got["rnn_states"].numpy(), ref["rnn_states"].numpy(), atol=TOL)
        if not poisoned:
            assert torch.equal(got["policy_id"], ref["policy_id"])
            assert torch.equal(got["policy_version"], ref["policy_version"])
        np.testing.assert_allclose(got["action_logits"].numpy(), ref["action_logits"].numpy(), atol=TOL)
        np.testing.assert_allclose(got["values"][:, :-1].numpy(), ref["values"][:, :-1].numpy(), atol=TOL)
        if ocfg.continuous:
            # Box actions are floats: a = eps*std + mean inherits the 1e-6-level differences of means / log_std
            np.testing.assert_allclose(got["actions"].numpy(), ref["actions"].numpy(), atol=TOL)
        else:
            # action indices: bit-exact (BASELINE.json). A flip would need p_i/q_i == p_j/q_j to within the 1e-6 logit
            # difference -- none occurs on these seeded inputs.
            assert torch.equal(got["actions"].view(ref["actions"].shape), ref["actions"]), "action indices must be bit-exact"
        np.testing.assert_allclose(got["log_prob_actions"].numpy(), ref["log_prob_actions"].numpy(), atol=TOL)


@pytest.mark.parametrize("engine", ENGINES)
@pytest.mark.parametrize("name", GOLDEN_CASES)
def test_learner_matches_reference_golden(name, engine):
    """Learner.train on the REFERENCE's trajectories: returns / advantages / loss terms / post-Adam weights /
    normalizer statistics against what the reference itself computed."""
    from sample_factory_b200 import ops

    _need(engine)
    dev = torch.device("cuda", 0)
    z, meta, ocfg = load_case(name)
    tape = torch.from_numpy(z["tape"])
    cfg, model, traj, env, sampler, learner = build(ocfg, meta["N"], state_from(z, "init/"), tape, dev, engine=engine)
    for it in range(meta["iters"]):
        assert learner.train_step == int(z[f"it{it}/train_step_before"])
        upload_traj(traj, traj_from(z, it, ocfg))
        learner.train(traj)
        torch.cuda.synchronize()
        assert learner.train_step == int(z[f"it{it}/train_step_after"])
        p = f"it{it}/prep/"
        assert torch.equal(learner.valids_flat.view(-1).cpu(), torch.from_numpy(z[p + "valids"]))
        np.testing.assert_allclose(traj["values"][:, -1].cpu().numpy(), z[p + "bootstrap_values"], atol=TOL)
        np.testing.assert_allclose(traj["rewards"].view(-1).cpu().numpy(), z[p + "rewards"], atol=1e-6)
        if not ocfg.with_vtrace:
            np.testing.assert_allclose(learner.advantages.view(-1).cpu().numpy(), z[p + "advantages"], atol=TOL)
            np.testing.assert_allclose(learner.returns.view(-1).cpu().numpy(), z[p + "returns"], atol=TOL)
        log = learner.minibatch_log().numpy()
        n_ref = len(z[f"it{it}/loss/policy_loss"])
        assert log.shape[0] == n_ref
        for key in ["policy_loss", "value_loss", "exploration_loss", "kl_loss", "adv_mean", "adv_std"]:
            np.testing.assert_allclose(log[:, ops.LS[key]], z[f"it{it}/loss/{key}"], atol=TOL, rtol=1e-5, err_msg=key)
        ref_state = state_from(z, f"it{it}/state/")
        got_state = model.state_dict()
        for k, v in ref_state.items():
            # float64 normaliser state: the obs statistics are functions of exact inputs (1e-8); the returns statistics
            # are moments of fp32 returns that themselves carry the 1e-5 tolerance (1e-6 on the moments)
            # post-Adam weights: an element whose gradient is comparable to adam_eps moves by lr * g / (|g| + eps), which
            # amplifies a 1e-6 gradient difference to ~1e-5 on the weight (seen on 2 of 8192 conv weights) -> 2e-5
            tol = (1e-6 if k.startswith("returns_normalizer") else 1e-8) if v.dtype == torch.float64 else 2 * TOL
            np.testing.assert_allclose(got_state[k].cpu().numpy().reshape(v.shape), v.numpy(), atol=tol, rtol=1e-6, err_msg=k)


@pytest.mark.parametrize("engine", ENGINES)
def test_closed_loop_vs_oracle_cfg2_shape(engine):
    """Sampler + learner for 2 iterations at N=256, T=32, cfg-2 model/hyper-parameters vs the oracle run on the same
    tape / noise / initial weights (the tape env keeps both rollouts aligned)."""
    from sample_factory_b200 import ops

    dev = torch.device("cuda", 0)
    N, T = 256, 32
    ocfg = O.OracleCfg(rollout=T, recurrence=1, batch_size=N * T // 4, num_batches_per_epoch=4, num_epochs=1)
    st0 = O.init_state(ocfg, seed=3)
    gen = torch.Generator().manual_seed(11)
    tape = torch.randn(2 * T + 1, N, ocfg.obs_dim, generator=gen) * 1.2 - 0.2
    _need(engine)
    cfg, model, traj, env, sampler, learner = build(ocfg, N, st0, tape, dev, engine=engine)
    olearner = O.OracleLearner(ocfg, st0)
    oenv = O.TapeVecEnv(tape, ocfg.num_actions)
    olast = oenv.reset()
    sampler.reset()
    for it in range(2):
        noise = torch.empty(T, N, ocfg.num_actions).exponential_(generator=gen)
        otraj = O.alloc_trajectories(ocfg, N)
        olast = O.rollout(ocfg, olearner.st, oenv, olast, otraj, noise, olearner.train_step)
        sampler.noise = noise.to(dev)
        sampler.set_policy_version(learner.train_step)
        sampler.rollout()
        got = {k: v.cpu() for k, v in traj.items()}
        mism = (got["actions"] != otraj["actions"]).float().mean().item()
        assert mism == 0.0, f"action mismatch fraction {mism}"
        for k in ["obs", "rewards", "dones", "time_outs", "policy_id", "policy_version"]:
            assert torch.equal(got[k], otraj[k]), k
        np.testing.assert_allclose(got["action_logits"].numpy(), otraj["action_logits"].numpy(), atol=TOL)
        np.testing.assert_allclose(got["values"][:, :-1].numpy(), otraj["values"][:, :-1].numpy(), atol=TOL)
        n0 = len(olearner.log)
        buff = olearner.train(otraj)
        learner.train(traj)
        np.testing.assert_allclose(learner.returns.view(-1).cpu().numpy(), buff["returns"].numpy(), atol=TOL)
        np.testing.assert_allclose(learner.advantages.view(-1).cpu().numpy(), buff["advantages"].numpy(), atol=TOL)
        log = learner.minibatch_log().numpy()
        for j, d in enumerate(olearner.log[n0:]):
            for key in ["policy_loss", "value_loss", "exploration_loss", "kl_loss"]:
                assert abs(log[j, ops.LS[key]] - d[key]) < TOL, (it, j, key, log[j, ops.LS[key]], d[key])
            assert abs(learner.grad_norm_log[j].item() - d["grad_norm"]) < 1e-4
        sd = model.state_dict()
        for k in O.param_names(ocfg):
            np.testing.assert_allclose(sd[k].cpu().numpy(), olearner.st[k].numpy(), atol=TOL, err_msg=k)


def test_full_size_properties_and_graph_replay():
    """N=4096, T=32 (BASELINE.json config 2): size-independent properties.
    * CUDA-graph replay and eager execution of the same rollout produce identical trajectories (Philox noise is a
      pure function of (seed, env, step) and both counters live on the device)
    * GAE linearity in the rewards; value targets = adv + values; returns-normaliser round trip
    * a training iteration changes the weights, keeps everything finite, and leaves padding untouched."""
    from sample_factory_b200 import ops

    dev = torch.device("cuda", 0)
    N, T = 4096, 32
    ocfg = O.OracleCfg(rollout=T, recurrence=1, batch_size=N * T // 4, num_batches_per_epoch=4)
    st0 = O.init_state(ocfg, seed=5)
    tape = torch.randn(3 * T + 1, N, ocfg.obs_dim, generator=torch.Generator().manual_seed(12))
    cfgA, modelA, trajA, envA, samplerA, learnerA = build(ocfg, N, st0, tape, dev, graph=False)
    cfgB, modelB, trajB, envB, samplerB, learnerB = build(ocfg, N, st0, tape, dev, graph=True)
    samplerA.reset()
    samplerB.reset()
    samplerA.rollout()
    samplerB.rollout()   # warm-up + capture + first replay start from the same counters? -> compare second rollouts
    # Graph capture runs the rollout eagerly once (warm-up) before replaying, so B is ahead; re-align both and compare
    for s, e in ((samplerA, envA), (samplerB, envB)):
        s.reset()
        s.step_counter.zero_()
    samplerA.rollout()
    samplerB.rollout()
    torch.cuda.synchronize()
    for k in trajA:
        assert torch.equal(trajA[k], trajB[k]), f"graph replay differs from eager for {k}"
    a = trajA["actions"]
    assert a.min().item() >= 0 and a.max().item() <= ocfg.num_actions - 1
    assert torch.all(trajA["policy_id"] == 0) and torch.isfinite(trajA["action_logits"]).all()
    freq = torch.bincount(a.view(-1).long(), minlength=ocfg.num_actions).float() / a.numel()
    assert freq.min().item() > 0.01, "every action should be sampled under near-uniform initial logits"

    # GAE linearity at full size
    r1 = torch.randn(N, T, device=dev)
    r2 = torch.randn(N, T, device=dev)
    dones = trajA["dones"]
    zeros_v = torch.zeros(N, T + 1, device=dev)
    ones_valid = torch.ones(N, T + 1, dtype=torch.bool, device=dev)
    outs = []
    for r in (r1, r2, r1 + r2):
        adv = torch.empty(N, T, device=dev)
        ret = torch.empty(N, T, device=dev)
        ops.gae_returns(r.clone(), dones, trajA["time_outs"], zeros_v, ones_valid, 0.99, 0.95, False, None, None, adv, ret)
        outs.append(adv)
        assert torch.equal(adv, ret)   # values == 0 -> returns == advantages
    assert (outs[0] + outs[1] - outs[2]).abs().max().item() < 1e-4

    before = modelA.flat.clone()
    learnerA.train(trajA)
    torch.cuda.synchronize()
    assert torch.isfinite(modelA.flat).all() and not torch.equal(before, modelA.flat)
    stats = learnerA.fetch_stats()
    assert all(np.isfinite(v) for v in stats.values()), stats
    assert stats["num_valid"] == N * T // 4
    assert torch.isfinite(learnerA.advantages).all() and torch.isfinite(learnerA.returns).all()
    # padding between tensors in the flat buffer must stay zero (zero grad -> zero Adam update)
    mask = torch.ones_like(modelA.flat, dtype=torch.bool)
    for n in modelA.names:
        o, shp = modelA._slices[n]
        mask[o:o + int(np.prod(shp))] = False
    assert torch.all(modelA.flat[mask] == 0)


def test_action_mask_graph_replay_and_mask_respected():
    """Action-mask env (obs dict) under the production path: in-kernel Philox noise, CUDA-graph replay == eager, every
    sampled action is allowed by the mask of its step (rows that allow nothing excepted), and the fused GEMM + heads path
    (hidden 128) honours the mask too."""
    dev = torch.device("cuda", 0)
    N, T = 512, 16
    ocfg = O.OracleCfg(obs_dim=32, num_actions=8, encoder_mlp_layers=[128, 128], rollout=T, recurrence=1,
                       batch_size=N * T // 2, num_batches_per_epoch=2, action_mask=True)
    st0 = O.init_state(ocfg, seed=6)
    tape = torch.randn(3 * T + 1, N, ocfg.obs_dim, generator=torch.Generator().manual_seed(13))
    engine = "3xtf32" if _tc() else "simt"
    _, _, trajA, envA, samplerA, _ = build(ocfg, N, st0, tape, dev, engine=engine, graph=False)
    _, _, trajB, envB, samplerB, _ = build(ocfg, N, st0, tape, dev, engine=engine, graph=True)
    for s in (samplerA, samplerB):
        s.reset()
        s.rollout()
    for s in (samplerA, samplerB):
        s.reset()
        s.step_counter.zero_()
        s.rollout()
    torch.cuda.synchronize()
    for k in trajA:
        assert torch.equal(trajA[k], trajB[k]), f"graph replay differs from eager for {k}"
    a = trajB["actions"][:, :, 0].cpu().long()
    env_idx = torch.arange(N)
    some_allowed = torch.zeros(N, T, dtype=torch.bool)
    for t in range(T):
        m = O.tape_action_mask(t, env_idx, ocfg.num_actions)
        some_allowed[:, t] = m.sum(1) > 0
        ok = m.gather(1, a[:, t:t + 1]).view(-1).bool() | ~some_allowed[:, t]
        assert bool(ok.all()), f"forbidden action sampled at step {t}"
    assert int(some_allowed.sum()) > 0.9 * N * T and not bool(some_allowed.all())
    # log-probs are the masked ones: exp(lp) sums over allowed actions only -> lp >= unmasked log-softmax of the action
    lg = trajB["action_logits"].cpu()
    lp_unmasked = torch.log_softmax(lg, -1).gather(2, a.unsqueeze(-1)).squeeze(-1)
    assert bool((trajB["log_prob_actions"].cpu() >= lp_unmasked - 1e-5)[some_allowed].all())
    np.testing.assert_allclose(trajB["log_prob_actions"].cpu()[~some_allowed].numpy(), -np.log(ocfg.num_actions), atol=1e-6)


def _tc():
    from sample_factory_b200 import ops

    return ops.tc_available()


def test_async_double_buffered_runner_matches_lagged_oracle(tmp_path):
    """async_rl=True (train.py): the sampler collects rollout i+1 on its own stream with a weight snapshot while the
    learner trains on rollout i.  The schedule is deterministic, so the oracle can replay it: rollout r is sampled
    with the weights published at the join before it (r0, r1 <- W0; r2 <- W after train(0); ...), stamped with that
    version, and trained on one iteration later (policy lag = 4 SGD steps, inside max_policy_lag)."""
    import copy

    from sample_factory_b200 import ops
    from sample_factory_b200.envs import TapeVecEnv, register_env
    from sample_factory_b200.train import Runner

    dev = torch.device("cuda", 0)
    N, T, ITERS = 128, 16, 3
    ocfg = O.OracleCfg(obs_dim=32, num_actions=8, encoder_mlp_layers=[128, 128], rollout=T, recurrence=1,
                       batch_size=N * T // 4, num_batches_per_epoch=4, num_epochs=1)
    st0 = O.init_state(ocfg, seed=13)
    gen = torch.Generator().manual_seed(17)
    tape = torch.randn((ITERS + 1) * T + 1, N, ocfg.obs_dim, generator=gen)
    noises = [torch.empty(T, N, ocfg.num_actions).exponential_(generator=gen) for _ in range(ITERS + 1)]
    register_env("async_tape", lambda n, c, e, render_mode=None: TapeVecEnv(tape.to(dev).contiguous(), ocfg.num_actions))
    cfg = make_cfg(ocfg, env="async_tape", train_dir=str(tmp_path), experiment="async", cuda_graph=False, seed=0,
                   gemm_engine="simt", async_rl=True, restart_behavior="overwrite")
    runner = Runner(cfg)
    assert runner.init() == 0
    runner.load_state_dict(st0)
    runner.rollout_hook = lambda r: setattr(runner.sampler, "noise", noises[r].to(dev))

    olearner = O.OracleLearner(ocfg, copy.deepcopy(st0))
    oenv = O.TapeVecEnv(tape, ocfg.num_actions)
    olast = oenv.reset()
    snap, snap_version = copy.deepcopy(olearner.st), 0
    pending = O.alloc_trajectories(ocfg, N)
    olast = O.rollout(ocfg, snap, oenv, olast, pending, noises[0], snap_version)      # priming rollout
    for it in range(ITERS):
        runner.iteration()
        torch.cuda.synchronize()
        nxt = O.alloc_trajectories(ocfg, N)
        olast = O.rollout(ocfg, snap, oenv, olast, nxt, noises[it + 1], snap_version)   # overlaps train(it) on the device
        olearner.train(pending)
        snap, snap_version = copy.deepcopy(olearner.st), olearner.train_step              # the join
        # the learner's buffer now holds rollout it+1, sampled with the PREVIOUS snapshot
        got = {k: v.cpu() for k, v in runner.traj.items()}
        for k in ["obs", "actions", "rewards", "dones", "policy_version"]:
            assert torch.equal(got[k], nxt[k]), (it, k)
        np.testing.assert_allclose(got["action_logits"].numpy(), nxt["action_logits"].numpy(), atol=TOL)
        sd = runner.model.state_dict()
        for k in O.param_names(ocfg):
            np.testing.assert_allclose(sd[k].cpu().numpy(), olearner.st[k].numpy(), atol=TOL, err_msg=f"{it} {k}")
        assert runner.learner.train_step == olearner.train_step == 4 * (it + 1)
        pending = nxt
    assert runner.rollouts_started == ITERS + 1 and runner.env_steps == ITERS * N * T
    lag = runner.learner.train_step - got["policy_version"].max().item()
    assert lag == 4.0      # samples in the buffer are one iteration (4 SGD steps) behind the learner


def test_split_sampler_matches_single_sampler():
    """worker_num_splits = 2 (two env groups on two streams, one graph) fills the trajectory buffers exactly like one
    sampler over all envs: same weights, same tape, same explicit noise -> identical trajectories (eager), and the
    graph-captured fork/join rollout reproduces the eager one with Philox noise."""
    from sample_factory_b200 import ops
    from sample_factory_b200.envs import TapeVecEnv
    from sample_factory_b200.sampler import DeviceSampler, SplitSampler

    dev = torch.device("cuda", 0)
    N, T = 256, 8
    ocfg = O.OracleCfg(rollout=T, recurrence=1, batch_size=N * T, num_batches_per_epoch=1, encoder_mlp_layers=[128, 128])
    st0 = O.init_state(ocfg, seed=8)
    tape = (torch.randn(2 * T + 1, N, ocfg.obs_dim, generator=torch.Generator().manual_seed(5)) * 1.1).to(dev)
    cfg, model, traj, env, sampler, _ = build(ocfg, N, st0, tape.cpu(), dev, engine="3xtf32" if ops.tc_available() else "simt")
    eng = sampler.engine
    noise = torch.empty(T, N, ocfg.num_actions).exponential_(generator=torch.Generator().manual_seed(9)).to(dev)
    sampler.reset()
    sampler.noise = noise
    sampler.rollout()
    ref = {k: v.clone() for k, v in traj.items()}
    for v in traj.values():
        v.zero_()
    h = N // 2
    envs = [TapeVecEnv(tape[:, :h].contiguous(), ocfg.num_actions, env_index_offset=0),
            TapeVecEnv(tape[:, h:].contiguous(), ocfg.num_actions, env_index_offset=h)]
    split = SplitSampler(cfg, envs, model, traj, engine=eng, use_cuda_graph=False)
    split.reset()
    split.noise = noise
    split.rollout()
    torch.cuda.synchronize()
    for k in ref:
        if k == "valids":
            continue
        if k == "values":      # column T (bootstrap value) belongs to the learner
            assert torch.equal(traj[k][:, :T], ref[k][:, :T]), k
            continue
        assert torch.equal(traj[k], ref[k]), k
    # graph-captured fork / join: replays are deterministic functions of (weights, tape, Philox counters)
    def run(use_graph, n):
        es = [TapeVecEnv(tape[:, :h].contiguous(), ocfg.num_actions, env_index_offset=0),
              TapeVecEnv(tape[:, h:].contiguous(), ocfg.num_actions, env_index_offset=h)]
        sp = SplitSampler(cfg, es, model, traj, engine=eng, use_cuda_graph=use_graph, philox_seed=3)
        sp.reset()
        outs = []
        for _ in range(n):
            sp.rollout()
            torch.cuda.synchronize()
            outs.append({k: traj[k].clone() for k in ("actions", "values", "rewards", "dones", "obs")})
        return outs, sp
    eager, _ = run(False, 4)
    graphed, sp = run(True, 3)
    assert sp.graph_replay_launches > 0
    # the graph path runs one un-captured warm-up rollout first (its trajectories are overwritten by the first replay), so
    # replay i continues from env step / Philox offset (i+1)*T
    for a, b in zip(eager[1:], graphed):
        for k in a:
            assert torch.equal(a[k], b[k]), k


@pytest.mark.parametrize("use_graph", [False, True])
def test_double_buffered_host_sampling_matches_one_group_after_the_other(use_graph):
    """worker_num_splits = 2 over HOST envs (rollout_worker.py:97-143): stepping the two env groups interleaved -- the GPU serves
    one group on its own stream while the host simulates the other -- fills the trajectory buffers exactly like running the
    groups' rollouts one after the other (same weights, tapes, Philox streams), with per-step launches and with per-step graphs"""
    from sample_factory_b200 import ops
    from sample_factory_b200.envs import HostTapeVecEnv
    from sample_factory_b200.sampler import SplitSampler

    dev = torch.device("cuda", 0)
    N, T = 256, 8
    ocfg = O.OracleCfg(rollout=T, recurrence=1, batch_size=N * T, num_batches_per_epoch=1, encoder_mlp_layers=[128, 128])
    st0 = O.init_state(ocfg, seed=8)
    tape = torch.randn(5 * T + 1, N, ocfg.obs_dim, generator=torch.Generator().manual_seed(5)) * 1.1
    cfg, model, traj, env, sampler, _ = build(ocfg, N, st0, tape, dev, engine="3xtf32" if ops.tc_available() else "simt")
    h = N // 2

    def run(interleaved, n):
        es = [HostTapeVecEnv(tape[:, :h].contiguous().numpy(), ocfg.num_actions, dev, env_index_offset=0),
              HostTapeVecEnv(tape[:, h:].contiguous().numpy(), ocfg.num_actions, dev, env_index_offset=h)]
        sp = SplitSampler(cfg, es, model, traj, engine=sampler.engine, use_cuda_graph=use_graph, philox_seed=3)
        assert sp.host_interleaved
        if not interleaved:
            sp.host_interleaved = False      # the groups' whole rollouts one after the other (sub-samplers on their streams)
        sp.reset()
        outs = []
        for _ in range(n):
            sp.rollout()
            torch.cuda.synchronize()
            outs.append({k: traj[k].clone() for k in ("actions", "values", "rewards", "dones", "obs", "policy_version")})
        return outs, sp

    seq, _ = run(False, 4)
    inter, sp = run(True, 4)
    if use_graph:
        assert all(s._step_graphs is not None for s in sp.subs) and sp.graph_replay_launches > 0
    for a, b in zip(seq, inter):
        for k in a:
            if k == "values":
                assert torch.equal(a[k][:, :T], b[k][:, :T]), k
            else:
                assert torch.equal(a[k], b[k]), k


def test_graphed_learner_matches_eager():
    """cfg.learner_cuda_graph: Learner.train() replayed as ONE CUDA graph (device-resident step counters / lr) produces the
    same parameters, Adam moments and loss statistics as the launch-by-launch learner, iteration after iteration."""
    from sample_factory_b200 import ops

    dev = torch.device("cuda", 0)
    N, T = 128, 8
    ocfg = O.OracleCfg(rollout=T, recurrence=1, batch_size=N * T // 2, num_batches_per_epoch=2, encoder_mlp_layers=[128, 128])
    st0 = O.init_state(ocfg, seed=2)
    tape = torch.randn(6 * T + 1, N, ocfg.obs_dim, generator=torch.Generator().manual_seed(3))
    eng = "3xtf32" if ops.tc_available() else "simt"
    cfgA, modelA, trajA, envA, samplerA, learnerA = build(ocfg, N, st0, tape, dev, engine=eng)
    cfgB, modelB, trajB, envB, samplerB, _ = build(ocfg, N, st0, tape, dev, engine=eng)
    from sample_factory_b200.learner import Learner

    cfgB.learner_cuda_graph = True
    learnerB = Learner(cfgB, modelB, N, engine=ops.ENGINES[eng])
    assert learnerB.use_graph and not learnerA.use_graph
    samplerA.reset()
    for it in range(5):
        noise = torch.empty(T, N, ocfg.num_actions).exponential_(generator=torch.Generator().manual_seed(20 + it)).to(dev)
        samplerA.noise = noise
        samplerA.set_policy_version(learnerA.train_step)
        samplerA.rollout()
        for k in trajA:
            trajB[k].copy_(trajA[k])
        learnerA.train(trajA)
        learnerB.train(trajB)
        torch.cuda.synchronize()
        assert learnerA.train_step == learnerB.train_step == 2 * (it + 1)
        assert torch.equal(modelA.flat, modelB.flat), it
        assert torch.equal(modelA.exp_avg_sq, modelB.exp_avg_sq) and torch.equal(modelA.obs_mean, modelB.obs_mean)
        assert torch.equal(learnerA.minibatch_log(), learnerB.minibatch_log())
        sa, sb = learnerA.fetch_stats(), learnerB.fetch_stats()
        assert sa["grad_norm"] == sb["grad_norm"] and sa["loss"] == sb["loss"]
    assert learnerB.graph_replay_launches > 0 and learnerB.kernel_launches == learnerA.kernel_launches + 2  # + advance_counters


@pytest.mark.parametrize("explicit_noise", [True, False])
def test_fused_policy_step_paths_match_separate_launches(explicit_noise, monkeypatch):
    """A policy step as per-layer GEMMs + ONE step-tail launch (csrc/heads.cu sampler_tail_tape_kernel: heads finish +
    sampling + tape-env step + post-step(t) + pre-step(t+1); what tape-env models outside the persistent kernel run), and a
    whole rollout as one persistent kernel, produce the same trajectories, episode statistics, env state and next policy
    input as the per-stage launches: bit-identical for everything downstream of the logits (same device functions),
    logits / values at rounding level."""
    _need("3xtf32")
    dev = torch.device("cuda", 0)
    N, T = 1000, 12
    ocfg = O.OracleCfg(rollout=T, recurrence=1, batch_size=N * T // 4, num_batches_per_epoch=4)
    st0 = O.init_state(ocfg, seed=9)
    gen = torch.Generator().manual_seed(3)
    tape = torch.randn(2 * T + 1, N, ocfg.obs_dim, generator=gen)
    noise = torch.empty(T, N, ocfg.num_actions).exponential_(generator=gen).to(dev)
    runs = {}
    for mode in ("separate", "fused", "persistent"):
        monkeypatch.setenv("SFB200_TAIL_FUSED", "0" if mode == "separate" else "1")
        monkeypatch.setenv("SFB200_ROLLOUT_FUSED", "1" if mode == "persistent" else "0")
        cfg, model, traj, env, sampler, learner = build(ocfg, N, st0, tape, dev, engine="3xtf32")
        assert sampler.fused_tail == (mode != "separate")
        assert sampler.fused_rollout == (mode == "persistent")
        sampler.reset()
        out = []
        for it in range(2):
            if explicit_noise:
                sampler.noise = noise
            sampler.set_policy_version(5 + it)
            sampler.rollout()
            out.append({k: v.clone() for k, v in traj.items()})
        torch.cuda.synchronize()
        runs[mode] = dict(traj=out, x_norm=sampler.x_norm.clone(), obs=env.obs.clone(), rew=env.rew.clone(),
                          term=env.terminated.clone(), step=env.step_counter.clone(), pstep=sampler.step_counter.clone(),
                          stats=sampler.episode_stats.clone(), ep=(sampler.ep_return.clone(), sampler.ep_len.clone()),
                          launches=sampler.kernel_launches_per_rollout)
    # pre-step(0), then per step: layer 1, layer 2 + head partials, step tail.  (The test-suite runs with SFB200_CHECK_LO=1:
    # one extra verification launch per GEMM that reads tf32-lo twins, two per persistent kernel on the tf32 path.)
    assert runs["fused"]["launches"] in (1 + 3 * T, 1 + 5 * T) and runs["separate"]["launches"] > runs["fused"]["launches"]
    assert runs["persistent"]["launches"] in (2, 4), runs["persistent"]["launches"]     # pre-step(0) + ONE kernel for T steps
    for other in ("fused", "persistent"):
        _compare_rollout_runs(runs["separate"], runs[other], other)


def _compare_rollout_runs(a, b, what):
    # the persistent kernel and the per-layer GEMMs split their operands into scaled fp16 pairs (22 significand bits) with
    # different partial-sum orders: logits agree to ~2 ulp of their size
    atol = 2e-6
    for ta, tb in zip(a["traj"], b["traj"]):
        for k in ta:
            if k in ("action_logits", "values", "log_prob_actions"):
                np.testing.assert_allclose(ta[k].cpu().numpy(), tb[k].cpu().numpy(), rtol=0, atol=atol, err_msg=f"{what} {k}")
            elif k != "valids":
                assert torch.equal(ta[k], tb[k]), (what, k)
    for k in ("obs", "rew", "term", "step", "pstep"):
        assert torch.equal(a[k], b[k]), (what, k)
    np.testing.assert_allclose(a["stats"].cpu().numpy(), b["stats"].cpu().numpy(), rtol=1e-12)
    assert torch.equal(a["ep"][0], b["ep"][0]) and torch.equal(a["ep"][1], b["ep"][1])


@pytest.mark.parametrize("rnn", [False, True])
@pytest.mark.parametrize("engine", ENGINES)
def test_shuffle_minibatches_matches_oracle(engine, rnn):
    """cfg.shuffle_minibatches (learner.py:498-526, a new permutation every epoch :707-713): the same permutations of
    recurrence-length chunks on both sides -> same minibatches -> same losses and post-Adam weights; with a recurrent core the
    chunks keep their BPTT structure."""
    from sample_factory_b200 import ops

    _need(engine)
    dev = torch.device("cuda", 0)
    N, T = 64, 16
    R = 8 if rnn else 1
    kw = dict(use_rnn=True, rnn_type="gru", rnn_size=64, recurrence=R) if rnn else dict(recurrence=1)
    ocfg = O.OracleCfg(obs_dim=24, num_actions=5, encoder_mlp_layers=[128, 128], rollout=T, batch_size=N * T // 4,
                       num_batches_per_epoch=4, num_epochs=2, **kw)
    st0 = O.init_state(ocfg, seed=2)
    gen = torch.Generator().manual_seed(8)
    tape = torch.randn(T + 1, N, ocfg.obs_dim, generator=gen)
    cfg, model, traj, env, sampler, learner = build(ocfg, N, st0, tape, dev, engine=engine)
    # (build() copies the oracle cfg; switch shuffling on in a fresh learner)
    from sample_factory_b200.learner import Learner
    cfg.shuffle_minibatches = True
    learner = Learner(cfg, model, N, engine=ops.ENGINES[engine])
    assert learner.shuffle
    olearner = O.OracleLearner(ocfg, st0)
    oenv = O.TapeVecEnv(tape, ocfg.num_actions)
    otraj = O.alloc_trajectories(ocfg, N)
    noise = torch.empty(T, N, ocfg.num_actions).exponential_(generator=gen)
    O.rollout(ocfg, olearner.st, oenv, oenv.reset(), otraj, noise, 0)
    otraj["policy_id"][torch.rand(N, T, generator=gen) < 0.1] = -1
    for k, v in otraj.items():
        if k in traj:
            traj[k].copy_(v.view(traj[k].shape))
    E = N * T
    rng = np.random.RandomState(4)
    perms = []
    for _ in range(ocfg.num_epochs):
        starts = rng.permutation(np.arange(0, E, R))
        perms.append((starts[:, None] + np.arange(R)[None, :]).reshape(-1))
    assert not np.array_equal(perms[0], perms[1])
    learner.set_minibatch_permutation(np.stack(perms))
    buff = olearner.train(otraj, mb_indices=[torch.from_numpy(p) for p in perms])
    learner.train(traj)
    log = learner.minibatch_log().numpy()
    assert log.shape[0] == len(olearner.log) == 8
    for j, d in enumerate(olearner.log):
        for key in ["policy_loss", "value_loss", "exploration_loss", "kl_loss"]:
            assert abs(log[j, ops.LS[key]] - d[key]) < TOL, (j, key, log[j, ops.LS[key]], d[key])
        assert abs(log[j, ops.LS["adv_mean"]] - d["adv_mean"]) < TOL
    sd = model.state_dict()
    for k in O.param_names(ocfg):
        np.testing.assert_allclose(sd[k].cpu().numpy(), olearner.st[k].numpy(), atol=2e-5, err_msg=k)
    # without an explicit permutation every train() draws its own (np.random, like the reference)
    np.random.seed(0)
    learner.train(traj)
    p1 = learner.perm_host.clone()
    learner.train(traj)
    assert not torch.equal(p1, learner.perm_host) and torch.equal(torch.sort(p1.long())[0], torch.arange(E))
    assert torch.isfinite(model.flat).all()
