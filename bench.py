#!/usr/bin/env python
"""Headline benchmark: env-steps/sec (sampler + learner) on the synthetic Box(64)/Discrete(8) vector env,
4096 envs per GPU (BASELINE.json configs[1]).

  python bench.py --gpus 1 --steps K --warmup W                 # our engine (libsfb200 on B200)
  python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...
  python bench.py --impl reference --gpus N --steps K --warmup W  # the reference's CPU path (oracle port) on the host
  python bench.py ... --dump-outputs DIR                        # also write the last timed step's outputs as DIR/<name>.npy

A "step" is one training iteration = one rollout of 32 env steps for all envs of the rank (131 072 env steps) followed
by one learner pass (4 minibatches x 1 epoch, forward + backward + Adam).  Prints ONE JSON line (rank 0).
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

N_ENVS, ROLLOUT, OBS_DIM, N_ACTIONS, HIDDEN = 4096, 32, 64, 8, [512, 512]
BATCH, N_MINIBATCH, N_EPOCHS = 32768, 4, 1
TAPE_LEN = 97   # 97 x 4096 x 64 x 4 B = 101 MB of env observations cycled through
METRIC = "env-steps/sec (sampler+learner) at 4096 envs"
UNIT = "env-steps/s"
WORKLOAD = ("synthetic Box(64)/Discrete(8) vec-env, 4096 envs per GPU, MLP 512-512 ELU, rollout 32, batch 32768 x 4 "
            "minibatches x 1 epoch, normalize_input+returns, GAE, Adam (BASELINE.json configs[1])")


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(p):
        d = json.load(open(p))
        return dict(hbm_gbs=d["hbm_gbs"], tflops_burst=d["bf16_tflops"],
                    tflops_sustained=d.get("bf16_tflops_sustained", d["bf16_tflops"]), source="measured (MEASURED_PEAKS.json)")
    return dict(hbm_gbs=6650.0, tflops_burst=1590.0, tflops_sustained=1400.0, source="fallback (B200_PROFILING.md)")


class ClockSampler:
    """Samples nvidia-smi clocks / throttle reasons DURING the timed region."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu_index = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "20", "-i", str(self.gpu_index)], stdout=subprocess.PIPE, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def num_samples(self) -> int:
        return sum(1 for ln in self.lines if len(ln.split(",")) >= 9)

    def stop(self):
        if self.proc is None:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["nvidia-smi unavailable"])
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, smax, reasons = [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                smax.append(float(f[2]))
            except ValueError:
                continue
            for name, val in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return dict(sm_mhz=statistics.median(sm) if sm else None, sm_max_mhz=max(smax) if smax else None,
                    reasons=sorted(reasons), samples=len(sm))


# --------------------------------------------------------------------------------------------------- reference arm
def _best_thread_count(O) -> int:
    """torch CPU throughput on this workload is NOT monotone in the thread count (on a 128-thread host, 128 intra-op
    threads run this path ~10x slower than 16-32 because most ops are small).  To give the CPU baseline its best shot we
    time one reduced iteration (1024 envs) per candidate and keep the fastest; the count used is reported as `cores`."""
    total = os.cpu_count() or 1
    cands = sorted({c for c in (4, 8, 16, 32, 64, total) if c <= total})
    n = 1024
    ocfg = O.OracleCfg(obs_dim=OBS_DIM, num_actions=N_ACTIONS, encoder_mlp_layers=list(HIDDEN), rollout=ROLLOUT,
                       recurrence=1, batch_size=n * ROLLOUT // N_MINIBATCH, num_batches_per_epoch=N_MINIBATCH)
    gen = torch.Generator().manual_seed(1)
    tape = torch.randn(ROLLOUT + 1, n, OBS_DIM, generator=gen)
    best, best_t = cands[0], float("inf")
    for c in cands:
        torch.set_num_threads(c)
        learner = O.OracleLearner(ocfg, O.init_state(ocfg, seed=0))
        env = O.TapeVecEnv(tape, N_ACTIONS)
        ts = []
        for _ in range(2):
            t0 = time.perf_counter()
            with torch.no_grad():
                noise = torch.empty(ROLLOUT, n, N_ACTIONS).exponential_(generator=gen)
                traj = O.alloc_trajectories(ocfg, n)
                O.rollout(ocfg, learner.st, env, env.reset(), traj, noise, 0)
            learner.train(traj)
            ts.append(time.perf_counter() - t0)
            if ts[-1] > 4 * best_t:
                break
        if min(ts) < best_t:
            best, best_t = c, min(ts)
    return best


def oracle_cpu_run(steps: int, warmup: int, n_envs: int = N_ENVS, calibrate: bool = True):
    """The reference's CPU path for this workload: the oracle port (torch CPU, best intra-op thread count), one process."""
    from oracle import appo_oracle as O

    cores = _best_thread_count(O) if calibrate else (os.cpu_count() or 1)
    torch.set_num_threads(cores)
    ocfg = O.OracleCfg(obs_dim=OBS_DIM, num_actions=N_ACTIONS, encoder_mlp_layers=list(HIDDEN), rollout=ROLLOUT,
                       recurrence=1, batch_size=n_envs * ROLLOUT // N_MINIBATCH, num_batches_per_epoch=N_MINIBATCH,
                       num_epochs=N_EPOCHS)
    gen = torch.Generator().manual_seed(0)
    tape = torch.randn(TAPE_LEN, n_envs, OBS_DIM, generator=gen)
    learner = O.OracleLearner(ocfg, O.init_state(ocfg, seed=0))
    env = O.TapeVecEnv(tape, N_ACTIONS)
    last = env.reset()
    times = []
    for it in range(warmup + steps):
        t0 = time.perf_counter()
        with torch.no_grad():
            noise = torch.empty(ROLLOUT, n_envs, N_ACTIONS).exponential_(generator=gen)
            traj = O.alloc_trajectories(ocfg, n_envs)
            last = O.rollout(ocfg, learner.st, env, last, traj, noise, learner.train_step)
        learner.train(traj)
        dt = time.perf_counter() - t0
        if it >= warmup:
            times.append(dt)
    total = sum(times)
    return dict(value=n_envs * ROLLOUT * len(times) / total, ms_per_step=1e3 * total / len(times), cores=cores)


def _ref_driver_call(n_envs: int, steps: int, warmup: int, threads: int, timeout: int = 1500):
    """One run of the UNMODIFIED reference (oracle/_ref, driven by oracle/ref_driver.py) in a subprocess (its logger is
    chatty and its thread settings are process-wide).  Returns the result dict or None."""
    cmd = [sys.executable, "-m", "oracle.ref_driver", "--n_envs", str(n_envs), "--rollout", str(ROLLOUT), "--obs_dim",
           str(OBS_DIM), "--num_actions", str(N_ACTIONS), "--batch_size", str(n_envs * ROLLOUT // N_MINIBATCH),
           "--num_batches_per_epoch", str(N_MINIBATCH), "--num_epochs", str(N_EPOCHS), "--steps", str(steps), "--warmup",
           str(warmup), "--tape_len", str(TAPE_LEN), "--threads", str(threads), "--hidden"] + [str(h) for h in HIDDEN]
    try:
        res = subprocess.run(cmd, cwd=ROOT, capture_output=True, text=True, timeout=timeout)
    except subprocess.TimeoutExpired:
        return None
    for line in reversed(res.stdout.splitlines()):
        if line.startswith("REF_DRIVER_RESULT "):
            return json.loads(line[len("REF_DRIVER_RESULT "):])
    sys.stderr.write(res.stdout[-2000:] + res.stderr[-2000:])
    return None


def reference_cpu_run(steps: int, warmup: int, n_envs: int = N_ENVS):
    """The reference's own CPU implementation of the path (sample-factory 2.1.3 installed in oracle/_ref): serial mode,
    batched sampling, torch CPU.  torch CPU throughput on this workload is not monotone in the thread count, so the count
    is calibrated on a reduced run (1024 envs) and reported as `cores`.  None when oracle/_ref is absent."""
    from oracle import ref_driver

    if not ref_driver.available():
        return None
    total = os.cpu_count() or 1
    best, best_v = None, 0.0
    for c in sorted({c for c in (8, 16, 32, 64, total) if c <= total}):
        r = _ref_driver_call(1024, 1, 1, c, timeout=300)
        if r is not None and r["value"] > best_v:
            best, best_v = c, r["value"]
    if best is None:
        return None
    return _ref_driver_call(n_envs, steps, warmup, best)


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    # same GLOBAL env count as our arm at this N (weak scaling: 4096 envs per GPU) -- on one host, like the reference runs
    n_envs = N_ENVS * args.gpus
    what = f"{args.steps} full iterations ({n_envs} envs x {ROLLOUT} steps + learner) after {args.warmup} warm-up"
    r = reference_cpu_run(args.steps, args.warmup, n_envs)
    if r is not None:
        kind = "reference"
        sample = (f"{what}; the unmodified reference (sample-factory 2.1.3 pip-installed into oracle/_ref) driven through "
                  f"BatchedVectorEnvRunner + ActorCritic forward + Learner.train, serial mode, torch CPU, "
                  f"{r['cores']} of {os.cpu_count()} host threads (best of a calibration sweep)")
    else:
        kind = "port"
        r = oracle_cpu_run(args.steps, args.warmup, n_envs)
        sample = (f"{what}; oracle port (oracle/_ref absent), torch CPU with the best-performing intra-op thread count "
                  f"({r['cores']} of {os.cpu_count()} host threads)")
    workload = WORKLOAD if args.gpus == 1 else WORKLOAD.replace("4096 envs per GPU", f"{n_envs} envs (= 4096 per GPU of our arm)")
    out = dict(impl="reference", metric=METRIC, value=r["value"], unit=UNIT, n_gpus=args.gpus, steps=args.steps,
               warmup=args.warmup, ms_per_step=r["ms_per_step"], higher_is_better=True, scaling="weak",
               vs_baseline=None, dtype="f32", data="synthetic", config=dict(workload=workload, global_envs=n_envs),
               cpu_baseline=dict(value=r["value"], unit=UNIT, cores=r["cores"], kind=kind, sample=sample),
               e2e=dict(value=r["value"], unit=UNIT, h2d_bytes_per_step=0, d2h_bytes_per_step=0))
    print(json.dumps(out), flush=True)


# --------------------------------------------------------------------------------------------------- our arm
def make_cfg(env_name: str, engine: str, cuda_graph: bool, async_rl: bool = False, splits: int = 1,
             learner_graph: bool = False, batch: int = BATCH):
    from sample_factory_b200.cfg import parse_full_cfg, parse_sf_args

    argv = [f"--env={env_name}", "--experiment=bench", "--train_dir=/tmp/sfb200_bench", "--restart_behavior=overwrite",
            "--use_rnn=False", f"--async_rl={async_rl}", "--serial_mode=True", "--batched_sampling=True", "--num_workers=1",
            f"--num_envs_per_worker={splits}", f"--worker_num_splits={splits}", f"--rollout={ROLLOUT}", f"--batch_size={batch}",
            f"--num_batches_per_epoch={N_MINIBATCH}", f"--num_epochs={N_EPOCHS}", "--encoder_mlp_layers", "512", "512",
            "--env_gpu_actions=True", "--env_gpu_observations=True", "--seed=0", f"--gemm_engine={engine}",
            f"--cuda_graph={cuda_graph}", f"--learner_cuda_graph={learner_graph}", "--save_every_sec=1000000000"]
    parser, _ = parse_sf_args(argv)
    return parse_full_cfg(parser, argv)



def dp_check(rank: int, world: int, dev, engine_flag: str, bench_model) -> dict:
    """Outside the timed region, on the box the driver measures scaling on: (1) the replicas of the benchmark run are
    bit-identical across ranks (weights and normaliser state), (2) G ranks x n envs == ONE process x G*n envs on the cfg-2
    model: rank 0 collects three rollouts of G*n envs, every rank trains on its env shard with the data-parallel learner
    exactly as the timed region runs it (NVLink peer exchanges, replayed as one CUDA graph), rank 0 also trains a
    single-process learner on the whole batch, and parameters / normaliser statistics / loss terms are compared."""
    import numpy as np

    from sample_factory_b200 import ops
    from sample_factory_b200.envs import TapeVecEnv
    from sample_factory_b200.learner import Learner
    from sample_factory_b200.model import ModelSpec, PolicyModel
    from sample_factory_b200.sampler import DeviceSampler
    from sample_factory_b200.train import select_engine
    from sample_factory_b200.trajectory import alloc_for_spec

    dist = torch.distributed
    out = {}

    def same_everywhere(t):
        ref = t.clone()
        dist.broadcast(ref, src=0)
        ok = torch.tensor([1 if torch.equal(ref, t) else 0], device=dev)
        dist.all_reduce(ok, op=dist.ReduceOp.MIN)
        return bool(ok.item())

    m = bench_model
    out["replicas_identical_after_bench"] = all(same_everywhere(t) for t in (m.flat, m.obs_mean, m.obs_var, m.ret_mean, m.ret_var))

    n, n_iter = 256, 3                       # envs per rank; iteration 1 runs eagerly, 2 captures + replays, 3 replays
    n_all = n * world
    cfg_dp = make_cfg("dp_check", engine_flag, False, learner_graph=True, batch=n * ROLLOUT // N_MINIBATCH)
    cfg_one = make_cfg("dp_check", engine_flag, False, learner_graph=False, batch=n_all * ROLLOUT // N_MINIBATCH)
    engine = select_engine(cfg_dp)
    tape = torch.randn(n_iter * ROLLOUT + 1, n_all, OBS_DIM, generator=torch.Generator().manual_seed(4321)).to(dev)
    env = TapeVecEnv(tape, N_ACTIONS)
    spec = ModelSpec.from_cfg(cfg_one, env)
    init = PolicyModel(spec, dev, seed=11)
    dist.broadcast(init.flat, src=0)
    init.weights_changed()
    batches = []
    full = alloc_for_spec(spec, n_all, ROLLOUT, dev)
    if rank == 0:
        sampler = DeviceSampler(cfg_one, env, init, full, engine=engine, use_cuda_graph=False, philox_seed=99)
        sampler.reset()
    for it in range(n_iter):
        if rank == 0:
            sampler.rollout()
            g = torch.Generator(device=dev).manual_seed(it)
            full["policy_id"][torch.rand(n_all, ROLLOUT, device=dev, generator=g) < 0.1] = -1    # some invalid samples
        for k in full:
            t = full[k].view(torch.uint8) if full[k].dtype == torch.bool else full[k]
            dist.broadcast(t, src=0)
        batches.append({k: v.clone() for k, v in full.items()})
    # the single-process minibatch b is envs [b*n_all/NMB, (b+1)*n_all/NMB); each rank takes its slice of every minibatch
    per_mb = n_all // N_MINIBATCH
    per_rank = per_mb // world
    idx = torch.cat([torch.arange(b * per_mb + rank * per_rank, b * per_mb + (rank + 1) * per_rank) for b in range(N_MINIBATCH)]).to(dev)

    def run(parallel):
        model = PolicyModel(spec, dev, seed=11)
        model.flat.copy_(init.flat)
        model.weights_changed()
        rows = n if parallel else n_all
        traj = alloc_for_spec(spec, rows, ROLLOUT, dev)
        learner = Learner(cfg_dp if parallel else cfg_one, model, rows, engine=engine, data_parallel=parallel)
        logs = []
        for b in batches:
            for k, v in b.items():
                traj[k].copy_(v[idx] if parallel else v)
            learner.train(traj)
            logs.append(learner.minibatch_log().numpy().copy())
        torch.cuda.synchronize()
        return model, learner, logs

    model_dp, learner_dp, logs_dp = run(True)
    out["learner_graph_replayed"] = bool(learner_dp.use_graph and learner_dp.graph_replay_launches > 0)
    out["exchange"] = "nvlink-peer kernels (csrc/comm.cu)" if learner_dp.comm is not None else "nccl"
    out["replicas_identical"] = all(same_everywhere(t) for t in (model_dp.flat, model_dp.obs_mean, model_dp.obs_var,
                                                                 model_dp.ret_mean, model_dp.ret_var))
    if rank == 0:
        model_1, learner_1, logs_1 = run(False)
        dparam = float((model_dp.flat - model_1.flat).abs().max())
        moved = float((model_1.flat - init.flat).abs().max())
        dstat = float(max((a - b).abs().max() for a, b in ((model_dp.obs_mean, model_1.obs_mean), (model_dp.obs_var, model_1.obs_var),
                                                          (model_dp.ret_mean, model_1.ret_mean), (model_dp.ret_var, model_1.ret_var))))
        keys = ["num_valid", "adv_mean", "adv_std", "policy_loss", "value_loss", "exploration_loss", "total_loss", "value_mean"]
        dloss = max(float(np.abs(a[:, ops.LS[k]] - b[:, ops.LS[k]]).max()) for a, b in zip(logs_dp, logs_1) for k in keys)
        out.update(max_abs_param_diff_vs_single_gpu=dparam, max_abs_param_change=moved, max_abs_normalizer_diff=dstat,
                   max_abs_loss_term_diff=dloss, equals_single_gpu=bool(dparam < 2e-6 and dstat < 1e-5 and dloss < 2e-5 and moved > 1e-4),
                   shape=f"{world} ranks x {n} envs x {ROLLOUT} steps vs 1 process x {n_all} envs, {n_iter} iterations, 10% invalid samples")
    dist.barrier()
    return out


def timed_path_outputs(runner) -> dict:
    """Host copies of what the last Runner.iteration() left for its caller: the trajectories of its rollout (what the learner
    trained on), the learner's advantages / returns / per-minibatch loss terms / grad norms, and the trained policy's
    state_dict (weights + normaliser statistics).  float64 stays float64, everything else becomes float32 (44 MB)."""
    lrn = runner.learner
    n = lrn.num_minibatches_done
    out = {f"traj.{k}": v for k, v in runner.traj.items()}
    out.update({"learner.advantages": lrn.advantages, "learner.returns": lrn.returns,
                "learner.loss_stats": lrn.loss_stats_log[:n], "learner.grad_norm": lrn.grad_norm_log[:n]})
    out.update({f"model.{k}": v for k, v in runner.model.state_dict().items()})
    return {k: v.detach().cpu().numpy().astype("float64" if v.dtype == torch.float64 else "float32") for k, v in out.items()}


def write_outputs(path: str, arrays: dict) -> None:
    import numpy as np

    total = sum(a.nbytes for a in arrays.values())
    assert total <= 64 << 20, f"--dump-outputs: {total} bytes exceed 64 MB"
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(path, f"{name}.npy"), a)


def run_ours(args):
    from sample_factory_b200 import ops
    from sample_factory_b200.dist_utils import init_from_env
    from sample_factory_b200.envs import HostTapeVecEnv, TapeVecEnv, register_env
    from sample_factory_b200.train import Runner

    rank, local_rank, world = init_from_env()
    assert world == args.gpus, f"--gpus {args.gpus} but WORLD_SIZE={world}"
    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    ops.bind_device(dev)
    dist = torch.distributed
    peaks = load_peaks()

    gen = torch.Generator().manual_seed(1234 + rank)
    tape_cpu = torch.randn(TAPE_LEN, N_ENVS, OBS_DIM, generator=gen)
    tape_dev = tape_cpu.to(dev)

    def make_tape_env(name, cfg, env_config, render_mode=None):
        # worker_num_splits groups (the reference's double-buffered sampling): group g owns envs [g*n, (g+1)*n)
        splits = int(cfg.worker_num_splits) if cfg.num_envs_per_worker == cfg.worker_num_splits else 1
        n = N_ENVS // splits
        g = int(env_config["vector_index"]) if splits > 1 else 0
        tape_g = tape_dev if splits == 1 else tape_dev[:, g * n: (g + 1) * n].contiguous()
        return TapeVecEnv(tape_g, N_ACTIONS, env_index_offset=rank * N_ENVS + g * n)

    register_env("synthetic_tape", make_tape_env)
    def make_host_env(name, cfg, env_config, render_mode=None):
        # the same env simulated on the host; worker_num_splits groups -> double-buffered sampling (the reference's default 2)
        splits = int(cfg.worker_num_splits) if cfg.num_envs_per_worker == cfg.worker_num_splits else 1
        n = N_ENVS // splits
        g = int(env_config["vector_index"]) if splits > 1 else 0
        tape_g = tape_cpu.numpy() if splits == 1 else tape_cpu[:, g * n: (g + 1) * n].contiguous().numpy()
        return HostTapeVecEnv(tape_g, N_ACTIONS, dev, env_index_offset=rank * N_ENVS + g * n)

    register_env("synthetic_tape_host", make_host_env)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def _ncu_traffic(key):
        """DRAM bytes per launch of the dominant kernel from the committed `ncu --set full` capture
        (profiles/traffic.json records the capture it came from); None when no capture is committed."""
        try:
            with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "profiles", "traffic.json")) as f:
                return json.load(f)[key]["traffic_bytes"]
        except (OSError, KeyError, ValueError):
            return None

    def max_over_ranks(x: float) -> float:
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ------------------------------------------------------------------ device-resident arm ("value")
    runner = Runner(make_cfg("synthetic_tape", args.engine, not args.no_graph, splits=args.splits,
                             learner_graph=not (args.no_learner_graph or args.no_graph)))
    runner.init()
    engine_name = {0: "simt-fp32", 1: "tcgen05-3xTF32", 2: "tcgen05-TF32"}[runner.engine]

    # live per-kernel timing of the dominant kernel (the learner's layer-2 forward GEMM, M=32768 N=K=512) and of the
    # main HBM-bound kernels, with CUDA events on the launching stream, inside the timed region
    timed = {}
    orig = {}

    def wrap(name, pred, work):
        fn = getattr(ops, name)
        orig[name] = fn

        def wrapped(*a, **k):
            w = pred(*a, **k)
            if w is None or not timing_on[0]:
                return fn(*a, **k)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            r = fn(*a, **k)
            e1.record()
            timed.setdefault(w, dict(events=[], work=work(*a, **k)))["events"].append((e0, e1))
            return r

        setattr(ops, name, wrapped)

    timing_on = [False]
    wrap("linear_act_forward", lambda x, W, b, out, act, eng: "gemm_fwd_l2" if (x.shape[0] == BATCH and W.shape == (512, 512)) else None,
         lambda x, W, b, out, act, eng: 2.0 * x.shape[0] * W.shape[0] * W.shape[1])
    # (the layer-2 forward now carries the heads' dot products in its epilogue: same GEMM flops are credited, the
    # 2*M*N*(A+1) head flops are not)
    for fused_name in ("linear_act_heads_forward", "linear_act_heads_forward_fused"):
        wrap(fused_name,
             lambda x, W, *a, **k: "gemm_fwd_l2" if (x.shape[0] == BATCH and W.shape == (512, 512)) else None,
             lambda x, W, *a, **k: 2.0 * x.shape[0] * W.shape[0] * W.shape[1])
    wrap("heads_backward", lambda h, *a, **k: "heads_backward" if h.shape[0] == BATCH else None,
         lambda h, Wv, Wa, dlogits, *a, **k: float(h.numel() * 4 * 2 + dlogits.numel() * 4 + h.shape[0] * 4))
    wrap("normalize_obs", lambda x, out, mean, *a, **k: "normalize_obs" if (x.shape[0] == N_ENVS * (ROLLOUT + 1) and mean is not None) else None,
         lambda x, out, *a, **k: float(x.numel() * 4 * 2))
    wrap("gae_returns", lambda rewards, *a, **k: "gae_returns", lambda rewards, *a, **k: float(rewards.numel() * 22))
    # (learner / sampler resolve ops.<fn> through the module at call time, so the wrappers take effect)
    clocks = ClockSampler(local_rank)
    clocks.start()             # before the warm-up: nvidia-smi needs ~100 ms before its first sample
    for _ in range(args.warmup):
        runner.iteration()
    barrier()
    clocks.lines.clear()       # keep the samples of the timed region only
    launches0 = ops.launch_count()
    replay_launches = 0
    timing_on[0] = True
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for _ in range(args.steps):
        runner.iteration()
        replay_launches += runner.sampler.graph_replay_launches + runner.learner.graph_replay_launches
    e1.record()
    barrier()
    timing_on[0] = False
    ms_total = max_over_ranks(e0.elapsed_time(e1))
    outputs = timed_path_outputs(runner) if (args.dump_outputs and rank == 0) else None
    gpu_launches = (ops.launch_count() - launches0) + replay_launches
    learner_graphed = bool(runner.learner.use_graph)
    if runner.learner.use_graph:
        # the learner was replayed as a graph: per-kernel CUDA events need eager launches -> three more (untimed for the
        # headline) iterations with the same kernels launched one by one
        runner.learner.use_graph = False
        timing_on[0] = True
        for _ in range(3):
            runner.iteration()
        barrier()
        timing_on[0] = False
    ms_per_step = ms_total / args.steps
    value = world * N_ENVS * ROLLOUT * args.steps / (ms_total / 1e3)

    kern = {}
    for name, d in timed.items():
        ms = [a.elapsed_time(b) for a, b in d["events"]]
        kern[name] = dict(avg_ms=sum(ms) / len(ms), launches=len(ms), work=d["work"])
    for name, fn in orig.items():
        setattr(ops, name, fn)

    roofline = None
    if "gemm_fwd_l2" in kern:
        k = kern["gemm_fwd_l2"]
        ach = k["work"] / (k["avg_ms"] * 1e-3) / 1e12
        roofline = dict(kernel=f"learner layer-2 forward GEMM [32768x512x512] + fused heads epilogue ({engine_name})", bound="tensor",
                        achieved=ach, peak=peaks["tflops_sustained"], unit="TFLOP/s", frac=ach / peaks["tflops_sustained"],
                        traffic=_ncu_traffic("gemm_fwd_l2"), avg_kernel_ms=k["avg_ms"], launches_timed=k["launches"],
                        peak_source=peaks["source"] + ", bf16 sustained (kernel timed inside a long step)",
                        note="fp32-parity GEMM = 3 tensor-core passes per product (hi*hi, hi*lo, lo*hi): the forward layers and dX run "
                             "them as kind::f16 MMAs on scaled fp16 operand pairs (ceiling = peak/3), dW as kind::tf32 MMAs "
                             "(ceiling = peak/6); the simt engine runs on CUDA cores (no tensor pipe)")
    roof2 = []
    for name in ("heads_backward", "normalize_obs", "gae_returns"):
        if name in kern:
            k = kern[name]
            ach = k["work"] / (k["avg_ms"] * 1e-3) / 1e9
            roof2.append(dict(kernel=name, bound="hbm", achieved=ach, peak=peaks["hbm_gbs"], unit="GB/s",
                              frac=ach / peaks["hbm_gbs"], avg_kernel_ms=k["avg_ms"], algorithmic_bytes=k["work"]))
    sampler_launches = runner.sampler.kernel_launches_per_rollout
    learner_launches = runner.learner.kernel_launches

    # sampler-only pass: the rollout's share of the step and its fraction of the HBM roofline (SURVEY 8d: 574
    # algorithmic bytes per env-step -- obs read + trajectory record)
    s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    s0.record()
    for _ in range(args.steps):
        runner.sampler.rollout()
    s1.record()
    barrier()
    rollout_ms = s0.elapsed_time(s1) / args.steps
    # nvidia-smi needs 0.1 s (one GPU) to well over a second (eight GPUs) before its first sample, and the timed region is
    # ~60 ms: keep the SAME workload running (untimed) until a few samples of the clocks under load exist
    # (sampler rollouts only: they involve no cross-rank exchange, so every rank can wait for its own nvidia-smi)
    extra_rollouts = 0
    t_wait = time.perf_counter()
    while clocks.proc is not None and clocks.num_samples() < 3 and time.perf_counter() - t_wait < 6.0:
        for _ in range(16):
            runner.sampler.rollout()
        torch.cuda.synchronize()
        extra_rollouts += 16
    clock_info = clocks.stop()
    clock_info["window"] = ("timed region + the per-kernel timing iterations and the sampler-only pass right after it (same workload)"
                            + (f" + {extra_rollouts} more untimed rollouts until nvidia-smi had delivered samples" if extra_rollouts else ""))
    samp_bytes = 574.0 * N_ENVS * ROLLOUT
    samp_gbs = samp_bytes / (rollout_ms * 1e-3) / 1e9
    persistent = bool(getattr(runner.sampler, "fused_rollout", False))
    samp_flops = 2.0 * (OBS_DIM * HIDDEN[0] + HIDDEN[0] * HIDDEN[1] + HIDDEN[1] * (N_ACTIONS + 1)) * N_ENVS * ROLLOUT
    samp_tf = samp_flops / (rollout_ms * 1e-3) / 1e12
    roof_sampler = dict(kernel=("sampler rollout = pre-step(0) + ONE persistent cluster kernel for the 32 policy steps "
                                "(csrc/rollout_fused.cu)" if persistent else
                                "sampler rollout (32 policy steps: layer-1 GEMM, layer-2 GEMM + head partials, fused step tail)"),
                        bound="hbm", achieved=samp_gbs, peak=peaks["hbm_gbs"], unit="GB/s", frac=samp_gbs / peaks["hbm_gbs"],
                        algorithmic_bytes=samp_bytes, rollout_ms=rollout_ms, share_of_step=rollout_ms / ms_per_step,
                        launches=int(sampler_launches),
                        tensor=dict(achieved=samp_tf, unit="TFLOP/s", peak=peaks["tflops_burst"], frac=samp_tf / peaks["tflops_burst"],
                                    algorithmic_flops=samp_flops,
                                    note="policy forward only (0.599 MFLOP per env step, SURVEY 8d) over the whole rollout time; "
                                         "3-pass fp16-split ceiling = peak / 3; 128 of 148 SMs hold a CTA"),
                        note="a 4096-env policy step moves 2.35 MB and 2.45 GFLOP: the rollout is bound by the per-step dependency "
                             "chain (tensor-pipe time of the two layers + epilogues + cluster barriers, profiles/r02_r_rollout_trace.md), "
                             "not by HBM bandwidth")
    dp_info = None
    if world > 1 and not args.no_dp_check:
        dp_info = dp_check(rank, world, dev, args.engine, runner.model)
    del runner
    torch.cuda.empty_cache()

    # ------------------------------------------------------------------ strong-scaling point (BASELINE metric: "at 4096 envs")
    strong = None
    if world > 1 and not args.no_strong:
        n_loc = N_ENVS // world
        tape_loc = tape_dev[:, :n_loc].contiguous()
        register_env("synthetic_tape_strong", lambda name, cfg, env_config, render_mode=None: TapeVecEnv(
            tape_loc, N_ACTIONS, env_index_offset=rank * n_loc))
        srunner = Runner(make_cfg("synthetic_tape_strong", args.engine, not args.no_graph, batch=BATCH // world,
                                  learner_graph=not (args.no_learner_graph or args.no_graph)))
        srunner.init()
        for _ in range(args.warmup):
            srunner.iteration()
        q0, q1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        q0.record()
        for _ in range(args.steps):
            srunner.iteration()
        q1.record()
        barrier()
        q_ms = max_over_ranks(q0.elapsed_time(q1))
        strong = dict(value=N_ENVS * ROLLOUT * args.steps / (q_ms / 1e3), unit=UNIT, ms_per_step=q_ms / args.steps,
                      scaling="strong", envs_total=N_ENVS, envs_per_gpu=n_loc, global_batch=BATCH * N_MINIBATCH,
                      note="the SAME 4096-env job split over the ranks (1/N of the envs and of every minibatch per GPU): a "
                           "policy step is latency-bound at 4096 rows already, so fewer rows per GPU shorten it only a little")
        del srunner
        torch.cuda.empty_cache()

    # ------------------------------------------------------------------ async double-buffered arm (async_rl=True)
    async_info = None
    if not args.no_async:
        arunner = Runner(make_cfg("synthetic_tape", args.engine, not args.no_graph, async_rl=True, splits=args.splits,
                                  learner_graph=not (args.no_learner_graph or args.no_graph)))
        arunner.init()
        for _ in range(args.warmup):
            arunner.iteration()
        a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        a0.record()
        for _ in range(args.steps):
            arunner.iteration()
        a1.record()
        barrier()
        a_ms = max_over_ranks(a0.elapsed_time(a1))
        async_info = dict(value=world * N_ENVS * ROLLOUT * args.steps / (a_ms / 1e3), unit=UNIT, ms_per_step=a_ms / args.steps,
                          policy_lag_sgd_steps=N_MINIBATCH * N_EPOCHS,
                          note="async_rl=True (the reference's default mode): rollout i+1 on a high-priority stream with a "
                               "weight snapshot while the learner trains on rollout i; same kernels, same work per step")
        del arunner
        torch.cuda.empty_cache()

    # ------------------------------------------------------------------ end-to-end arm (host env, H2D/D2H inside)
    e2e = None
    if not args.no_e2e:
        def run_e2e(async_rl: bool):
            # the host is the bottleneck of this arm (it steps the envs): the learner's ~90 launches are replayed as one graph
            r2 = Runner(make_cfg("synthetic_tape_host", args.engine, not args.no_graph, async_rl=async_rl,
                                 learner_graph=not args.no_graph, splits=args.e2e_splits))
            r2.init()
            for _ in range(max(3, args.warmup)):
                r2.iteration()
                r2.learner.fetch_stats()
            barrier()
            envs = r2.envs
            h0, d0 = sum(e.h2d_bytes for e in envs), sum(e.d2h_bytes for e in envs)
            stats_bytes = 0
            t0 = time.perf_counter()
            for _ in range(args.steps):
                r2.iteration()
                st = r2.learner.fetch_stats()            # D2H read of the step's result (loss terms)
                stats_bytes += 8 * sum(1 for v in st.values() if isinstance(v, float))
            barrier()
            dt = max_over_ranks(time.perf_counter() - t0)
            out = dict(value=world * N_ENVS * ROLLOUT * args.steps / dt, unit=UNIT,
                       h2d_bytes_per_step=(sum(e.h2d_bytes for e in envs) - h0) // args.steps,
                       d2h_bytes_per_step=(sum(e.d2h_bytes for e in envs) - d0 + stats_bytes) // args.steps,
                       ms_per_step=1e3 * dt / args.steps)
            del r2
            torch.cuda.empty_cache()
            return out

        e2e = run_e2e(False)
        e2e["api"] = ("sample_factory_b200.train.Runner.iteration() with a HOST env (numpy simulator, pinned staging): "
                      "obs H2D + actions D2H every env step, loss stats D2H every iteration; learner_cuda_graph=True; "
                      f"worker_num_splits={args.e2e_splits}; per env step ONE graph replay (post-step(t) + policy step(t+1) + the "
                      "actions' D2H copy) between the env's host simulation and its H2D copies")
        e2e["worker_num_splits"] = args.e2e_splits
        if not args.no_async:
            ea = run_e2e(True)
            e2e["async_rl"] = dict(value=ea["value"], ms_per_step=ea["ms_per_step"],
                                   note="same arm with async_rl=True (the reference's default): the learner's graph runs "
                                        "on the GPU while the host steps the envs of the next rollout")

    cpu_baseline = None
    if world == 1 and rank == 0 and not args.no_cpu_baseline:
        r = reference_cpu_run(steps=6, warmup=2)
        if r is not None:
            cpu_baseline = dict(value=r["value"], unit=UNIT, cores=r["cores"], kind="reference", ms_per_step=r["ms_per_step"],
                                sample="6 full iterations (4096 envs x 32 steps + learner) after 2 warm-up; the unmodified reference "
                                       "(sample-factory 2.1.3 in oracle/_ref: BatchedVectorEnvRunner + ActorCritic + Learner.train, "
                                       f"serial mode, torch CPU), {r['cores']} of {os.cpu_count()} host threads")
        rp = oracle_cpu_run(steps=6, warmup=2)
        port = dict(value=rp["value"], unit=UNIT, cores=rp["cores"], kind="port", ms_per_step=rp["ms_per_step"],
                    sample="6 full iterations after 2 warm-up, oracle port (oracle/appo_oracle.py), torch CPU with the "
                           f"best-performing intra-op thread count of {os.cpu_count()} host threads")
        if cpu_baseline is None:
            cpu_baseline = port
        else:
            cpu_baseline["oracle_port"] = port

    if outputs is not None:
        write_outputs(args.dump_outputs, outputs)
    if rank == 0:
        out = dict(metric=METRIC, value=value, unit=UNIT, n_gpus=world, steps=args.steps, warmup=args.warmup,
                   ms_per_step=ms_per_step, higher_is_better=True, scaling="weak", vs_baseline=None,
                   dtype="f32" + (" (3-pass operand split on tcgen05 -- scaled fp16 hi/lo pairs where the operand ranges are known, tf32 hi/lo pairs elsewhere -- fp32 accumulate in TMEM)" if engine_name == "tcgen05-3xTF32" else ""),
                   data="synthetic",
                   config=dict(workload=WORKLOAD, envs_per_gpu=N_ENVS, rollout=ROLLOUT, global_batch=BATCH * N_MINIBATCH * world,
                               parallelism=f"dp{world} (env shards; per SGD step ONE kernel = NVLink peer all-reduce + grad-norm + clip + Adam)", gemm_engine=engine_name,
                               cuda_graph_rollout=not args.no_graph,
                               cuda_graph_learner=learner_graphed, worker_num_splits=args.splits,
                               l2_policy="per-step working set (trajectories 45 MB + obs tape 101 MB + learner "
                                         "activations 4x64 MB + workspaces) exceeds the 126 MB L2; no explicit flush"),
                   clocks=clock_info, e2e=e2e, gpu_launches=int(gpu_launches),
                   launches_per_step=dict(sampler_rollout=int(sampler_launches), learner_train=int(learner_launches)),
                   roofline=roofline, roofline_sampler=roof_sampler, roofline_secondary=roof2, async_rl=async_info,
                   cpu_baseline=cpu_baseline, dp_check=dp_info, strong_scaling=strong)
        print(json.dumps(out), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", type=int, default=2, choices=[2, 3, 4, 5],
                    help="BASELINE.json config (1-based): 2 = the headline synthetic 4096-env MLP job (default); 3 / 4 / 5 = the "
                         "mujoco-, atari- and isaacgym-shaped jobs (bench_configs.py), same JSON contract")
    ap.add_argument("--engine", default="auto", choices=["auto", "simt", "3xtf32", "tf32"])
    ap.add_argument("--splits", type=int, default=1,
                    help="worker_num_splits: env groups whose per-step kernel chains run concurrently on separate streams "
                         "(measured at 4096 envs: 1.29 ms per rollout with 2 or 4 groups vs 1.32 ms with 1 -- a policy step is "
                         "a chain of one-wave kernels, so halving the rows per kernel does not shorten it)")
    ap.add_argument("--e2e-splits", dest="e2e_splits", type=int, default=1,
                    help="worker_num_splits of the end-to-end (host env) arm: 2 = double-buffered sampling over two env groups (the "
                         "GPU serves one group while the host steps the other).  Measured with the numpy tape env, whose host step "
                         "costs ~25 us: 22.8 M env-steps/s with 2 groups vs 25.0 M with 1 -- the host thread's per-call overhead, "
                         "not the GPU, is what a second group doubles; the mode pays off for envs whose host step is expensive")
    ap.add_argument("--no-graph", dest="no_graph", action="store_true")
    ap.add_argument("--no-learner-graph", dest="no_learner_graph", action="store_true",
                    help="launch the learner's kernels one by one instead of replaying Learner.train() as one CUDA graph "
                         "(--learner_cuda_graph=True; measured 40.4M vs 38.0M env-steps/s, profiles/r01_m_*).  With the graph "
                         "the per-kernel roofline timings come from three extra eager iterations after the timed region")
    ap.add_argument("--no-e2e", dest="no_e2e", action="store_true")
    ap.add_argument("--no-async", dest="no_async", action="store_true")
    ap.add_argument("--no-cpu-baseline", dest="no_cpu_baseline", action="store_true")
    ap.add_argument("--no-dp-check", dest="no_dp_check", action="store_true",
                    help="N > 1: skip the (untimed) replica / single-GPU equivalence check printed as `dp_check`")
    ap.add_argument("--no-strong", dest="no_strong", action="store_true",
                    help="N > 1: skip the strong-scaling point (4096 envs in total, split over the ranks)")
    ap.add_argument("--dump-outputs", dest="dump_outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one computed (trajectories, advantages / returns, loss "
                         "terms, trained state_dict; rank 0) as DIR/<name>.npy, to compare two builds output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.config != 2):
        ap.error("--dump-outputs applies to the headline workload of our engine (--impl ours --config 2)")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    if args.config != 2:
        import bench_configs

        if args.impl == "reference":
            bench_configs.run_config_reference(args)
        else:
            bench_configs.run_config(args, load_peaks, ClockSampler)
    elif args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
