"""CPU-only tests (-m "not gpu"): the C-ABI library loads and exports every symbol include/sfb200.h declares (no compute
calls without a GPU), the host-side logic (config surface, model/checkpoint naming, LR schedulers), and the
data-parallel host logic under gloo with world_size 2."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_the_declared_abi():
    import ctypes

    from sample_factory_b200._lib import ABI_VERSION, LIB_PATH, lib, parse_header

    protos = parse_header()
    assert len(protos) >= 29
    cdll = ctypes.CDLL(LIB_PATH)
    for name in protos:
        assert hasattr(cdll, name), f"{name} declared in include/sfb200.h but not exported by libsfb200.so"
    out = subprocess.run(["nm", "-D", "--defined-only", LIB_PATH], capture_output=True, text=True).stdout
    exported = {line.split()[-1] for line in out.splitlines() if " T " in line}
    assert {n for n in exported if n.startswith("sfb200_")} == set(protos), "exported ABI != declared ABI"
    # value-returning queries are safe without a GPU
    l = lib()
    assert l.query("sfb200_abi_version") == ABI_VERSION
    assert l.query("sfb200_moments_workspace_bytes", 64) > 0
    assert l.query("sfb200_loss_workspace_bytes", 32768) > 0
    assert l.query("sfb200_heads_backward_workspace_bytes", 512, 8) > 0
    assert l.query("sfb200_linear_backward_workspace_bytes", 32768, 512, 512) > 0


def test_sass_is_sm100a_only():
    from sample_factory_b200._lib import LIB_PATH

    out = subprocess.run(["cuobjdump", "-lelf", LIB_PATH], capture_output=True, text=True).stdout
    archs = {tok for line in out.splitlines() for tok in line.replace(".", " ").split() if tok.startswith("sm_")}
    assert archs == {"sm_100a"}, archs


def test_tc_objects_are_blackwell_native_by_instruction_mix():
    """Not just the arch tag: the GEMM engine's and the persistent rollout kernel's SASS must contain the 5th-gen tensor-core
    path -- UTCHMMA (tcgen05.mma), UTMALDG (TMA), LDTM / STTM (tcgen05.ld / st), UTCBAR (tcgen05.commit) -- and no legacy HMMA
    (mma.sync); the fp16 operand split shows up as F2FP packs.  (profiles/r02_sass_mix.md is the full table, tools/sass_mix.py.)"""
    csrc = os.path.join(ROOT, "sample_factory_b200", "csrc")
    for obj, need_f2fp in (("gemm_tc.o", True), ("rollout_fused.o", True)):
        path = os.path.join(csrc, obj)
        if not os.path.isfile(path):
            pytest.skip(f"{obj} not in tree (objects are built by __graft_entry__.build() and do not travel to the GPU box)")
        sass = subprocess.run(["cuobjdump", "-sass", path], capture_output=True, text=True, timeout=600).stdout
        count = lambda op: sum(1 for ln in sass.splitlines() if f" {op}" in ln and "/*" in ln)   # noqa: E731
        assert count("UTCHMMA") > 0 and count("UTMALDG") > 0 and count("LDTM") > 0 and count("STTM") > 0 and count("UTCBAR") > 0, obj
        assert count("HMMA.") == 0, f"{obj}: legacy mma.sync instructions"
        if need_f2fp:
            assert count("F2FP") > 0, f"{obj}: no fp16 operand split"


def test_no_cpu_fallback():
    """The product path must fail loudly without a device, not silently compute on the CPU."""
    from sample_factory_b200 import ops

    with pytest.raises(RuntimeError):
        ops.normalize_obs(torch.zeros(4, 4), torch.zeros(4, 4), None, None)
    # and the product package never imports the oracle
    import ast

    pkg = os.path.join(ROOT, "sample_factory_b200")
    for fn in os.listdir(pkg):
        if fn.endswith(".py"):
            tree = ast.parse(open(os.path.join(pkg, fn)).read())
            for node in ast.walk(tree):
                names = []
                if isinstance(node, ast.Import):
                    names = [a.name for a in node.names]
                elif isinstance(node, ast.ImportFrom):
                    names = [node.module or ""]
                assert not any(n.split(".")[0] == "oracle" for n in names), f"{fn} imports the oracle"


def test_cfg_surface_matches_reference_flags():
    """Every reference flag (cfg/cfg.py) parses with the reference's default; two-pass parse records cli_args."""
    from sample_factory_b200.cfg import default_cfg, parse_full_cfg, parse_sf_args, preprocess_cfg

    cfg = default_cfg()
    assert cfg.gamma == 0.99 and cfg.rollout == 32 and cfg.batch_size == 1024 and cfg.adam_eps == 1e-6
    assert cfg.encoder_mlp_layers == [512, 512] and cfg.exploration_loss_coeff == 0.003 and cfg.use_rnn is True
    argv = ["--env=synthetic", "--use_rnn=False", "--encoder_mlp_layers", "64", "64", "--batch_size=4096",
            "--my_env_flag=3"]
    parser, partial = parse_sf_args(argv)
    assert partial.env == "synthetic"
    parser.add_argument("--my_env_flag", type=int, default=0)       # what sf_examples do between the two passes
    parser.set_defaults(lr_schedule="linear_decay")                 # mujoco_params.py-style default override
    cfg = parse_full_cfg(parser, argv)
    assert cfg.my_env_flag == 3 and cfg.lr_schedule == "linear_decay" and cfg.encoder_mlp_layers == [64, 64]
    assert set(cfg.cli_args) == {"env", "use_rnn", "encoder_mlp_layers", "batch_size", "my_env_flag"}
    assert preprocess_cfg(cfg) and cfg.recurrence == 1
    cfg.with_vtrace = True
    assert not preprocess_cfg(cfg)   # V-trace needs recurrence == rollout and no returns normalisation
    # the reference's other verify_cfg rules (cfg/arguments.py:123-127, 187-191)
    from sample_factory_b200.cfg import verify_cfg

    c = default_cfg()
    assert preprocess_cfg(c) and c.recurrence == c.rollout        # use_rnn default True: recurrence -1 -> rollout
    c.num_envs_per_worker, c.worker_num_splits = 3, 2
    assert not verify_cfg(c)
    c.num_envs_per_worker = 4
    assert verify_cfg(c)
    c.recurrence = 1
    assert not verify_cfg(c)                                      # an RNN needs recurrence > 1
    c.use_rnn = False
    assert verify_cfg(c)
    c.batch_size, c.num_batches_per_epoch, c.rollout, c.async_rl = 1000, 1, 32, False
    assert not verify_cfg(c, num_agents_total=7) and verify_cfg(c, num_agents_total=125)


def test_model_layout_and_checkpoint_names():
    from oracle import appo_oracle as O
    from sample_factory_b200.model import ModelSpec, PolicyModel

    spec = ModelSpec(64, 8)
    m = PolicyModel(spec, torch.device("cpu"))
    assert m.num_params == 300553                       # SURVEY section 8: cfg-2 model
    assert m.names == O.param_names(O.OracleCfg())      # == reference nn.Module.parameters() order
    sd = m.state_dict()
    st = O.init_state(O.OracleCfg(), seed=1)
    assert set(sd.keys()) == set(st.keys())             # reference state_dict keys incl. normalizer buffers
    m.load_state_dict(st)
    for k, v in st.items():
        assert torch.equal(m.state_dict()[k], v)
    for t in m.params.values():                         # 256-byte alignment of every tensor in the flat buffer
        assert t.data_ptr() % 256 == m.flat.data_ptr() % 256
    osd = m.optimizer_state_dict(step=3, lr=1e-4, betas=(0.9, 0.999), eps=1e-6)
    assert len(osd["state"]) == len(m.names) and osd["param_groups"][0]["params"] == list(range(len(m.names)))
    # orthogonal init (actor_critic.py:73-96): W W^T = I for the wide first layer, biases zero
    W = m2 = PolicyModel(spec, torch.device("cpu"), seed=0).params["encoder.encoders.obs.mlp_head.0.weight"]
    np.testing.assert_allclose((W.t() @ W).numpy(), np.eye(64), atol=1e-5)


def test_lr_schedulers():
    from sample_factory_b200.cfg import default_cfg
    from sample_factory_b200.learner import get_lr_scheduler

    cfg = default_cfg()
    cfg.lr_schedule = "kl_adaptive_epoch"
    cfg.num_batches_per_epoch = 2
    s = get_lr_scheduler(cfg)
    assert s.invoke_after_each_epoch() and not s.invoke_after_each_minibatch()
    assert s.update(1e-4, [0.1, 0.1]) == pytest.approx(1e-4 / 1.5)      # KL above 2x threshold
    assert s.update(1e-4, [0.0, 0.001]) == pytest.approx(1.5e-4)        # KL below 0.5x threshold
    assert s.update(1e-4, [0.008, 0.008]) == 1e-4
    cfg.lr_schedule = "linear_decay"
    cfg.train_for_env_steps, cfg.batch_size, cfg.num_epochs, cfg.learning_rate = 10240, 1024, 1, 1.0
    s = get_lr_scheduler(cfg)
    assert s.update(1.0, []) == pytest.approx(0.9) and s.update(0.9, []) == pytest.approx(0.8)


def test_trajectory_layout_matches_reference():
    from oracle import appo_oracle as O
    from sample_factory_b200.trajectory import alloc_trajectory_tensors, trajectory_bytes_per_env_step

    t = alloc_trajectory_tensors(64, 8, 10, 32, "cpu")
    ref = O.alloc_trajectories(O.OracleCfg(), 10)
    assert set(t) == set(ref)
    for k in t:
        assert t[k].shape == ref[k].shape and t[k].dtype == ref[k].dtype, k
    assert trajectory_bytes_per_env_step(64, 8) == 574   # SURVEY section 8d


_GLOO_WORKER = r"""
import os, sys, torch, torch.distributed as dist
sys.path.insert(0, sys.argv[1])
from sample_factory_b200.dist_utils import init_from_env, pooled_moments_, allreduce_sum_
rank, local_rank, world = init_from_env("gloo")
assert world == 2
g = torch.Generator().manual_seed(0)
full = torch.randn(2000, 7, generator=g) * 3 + 1          # the data one process holding all envs would see
mine = full[rank * 1000:(rank + 1) * 1000]                # this rank's env shard
bm, bv = mine.mean(0), mine.var(0)
total = pooled_moments_(bm, bv, 1000)
assert total == 2000
assert torch.allclose(bm, full.mean(0), atol=1e-6), (bm, full.mean(0))
assert torch.allclose(bv, full.var(0), atol=1e-5), (bv, full.var(0))
grad = torch.full((5,), float(rank + 1))
allreduce_sum_(grad)
assert torch.equal(grad, torch.full((5,), 3.0))
# advantage statistics: per-rank (count, sum, sumsq) partials add up to the global ones
adv = full[:, 0]; a = adv[rank * 1000:(rank + 1) * 1000].double()
part = torch.stack([torch.tensor(float(a.numel()), dtype=torch.float64), a.sum(), (a * a).sum()])
allreduce_sum_(part)
mean = part[1] / part[0]; std = torch.sqrt((part[2] - part[1] * mean) / (part[0] - 1))
assert abs(mean - adv.double().mean()) < 1e-9 and abs(std - adv.double().std()) < 1e-9
dist.barrier(); dist.destroy_process_group()
print("rank", rank, "ok")
"""


def test_data_parallel_host_logic_gloo_world2(tmp_path):
    script = tmp_path / "gloo_worker.py"
    script.write_text(_GLOO_WORKER)
    procs = []
    port = 29000 + (os.getpid() % 2000)
    for rank in range(2):
        env = dict(os.environ, RANK=str(rank), LOCAL_RANK=str(rank), WORLD_SIZE="2", MASTER_ADDR="127.0.0.1",
                   MASTER_PORT=str(port))
        procs.append(subprocess.Popen([sys.executable, str(script), ROOT], env=env, stdout=subprocess.PIPE,
                                      stderr=subprocess.STDOUT, text=True))
    for p in procs:
        out, _ = p.communicate(timeout=240)
        assert p.returncode == 0, out


_PBT_GLOO_WORKER = r"""
import os, random, sys
sys.path.insert(0, sys.argv[1])
from collections import deque
from types import SimpleNamespace
import torch.distributed as dist
from sample_factory_b200.multi_policy import MultiPolicyRunner
from sample_factory_b200.pbt import PopulationBasedTraining

rank = int(os.environ["RANK"])
dist.init_process_group("gloo", rank=rank, world_size=2)
random.seed(100 + rank)                 # the ranks' Python RNGs differ on purpose: only rank 0's draws may count
cfg = SimpleNamespace(num_policies=3, with_pbt=True, pbt_optimize_gamma=False, pbt_mutation_rate=1.0, pbt_perturb_min=1.1,
                      pbt_perturb_max=1.5, pbt_replace_fraction=0.3, pbt_replace_reward_gap=0.1, pbt_replace_reward_gap_absolute=1e-6,
                      pbt_target_objective="true_objective", pbt_period_env_steps=10, pbt_start_mutation=10, env="e",
                      learning_rate=1e-4, exploration_loss_coeff=0.003, value_loss_coeff=0.5, max_grad_norm=4.0,
                      ppo_clip_ratio=0.1, ppo_clip_value=1.0, gamma=0.99, batch_size=1024, rollout=32)
mp = MultiPolicyRunner.__new__(MultiPolicyRunner)          # the decision plumbing only: no device members on a CPU box
mp.cfg, mp.rank, mp.world_size, mp.writers = cfg, rank, 2, {}
applied = []
mp.update_policy_cfg = lambda p, c: applied.append(("cfg", p, dict(c)))
mp.update_reward_shaping = lambda p, s: None
mp.replace_policy = lambda p, donor: applied.append(("replace", p, donor))
mp.subs = [SimpleNamespace(env_steps=100) for _ in range(3)]
mp.policy_avg_stats = {"true_objective": [deque([1.0 + rank]), deque([-5.0]), deque([4.0 - rank])]}   # rank-local statistics differ too
mp.pbt = PopulationBasedTraining(cfg, mp, log=lambda *a: None)
mp.pbt.dir, mp.pbt.default_reward_shaping = sys.argv[2] + f"/r{rank}", None
os.makedirs(mp.pbt.dir, exist_ok=True)
if rank == 0:
    mp.pbt.on_init(mp.pbt.dir, None)
mp._pbt_broadcast_all()
mp.pbt.on_training_step()
box = [None, None]
dist.all_gather_object(box, (mp.pbt.policy_cfg, applied))
assert box[0] == box[1], box                 # same hyper-parameters, same replacements, same order on both ranks
assert ("replace", 1, 2) in applied, applied
dist.barrier()
print("PBT_GLOO_OK")
"""


def test_pbt_decisions_are_rank0s_on_every_rank_gloo_world2(tmp_path):
    """data parallel + PBT: every rank must apply the SAME replacement and the SAME mutated hyper-parameters although their
    Python RNGs and local episode statistics differ (multi_policy.MultiPolicyRunner.pbt_decide: rank 0 decides, broadcast)"""
    script = tmp_path / "pbt_gloo_worker.py"
    script.write_text(_PBT_GLOO_WORKER)
    procs = []
    port = 31000 + (os.getpid() % 2000)
    for rank in range(2):
        env = dict(os.environ, RANK=str(rank), LOCAL_RANK=str(rank), WORLD_SIZE="2", MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
        procs.append(subprocess.Popen([sys.executable, str(script), ROOT, str(tmp_path)], env=env, stdout=subprocess.PIPE,
                                      stderr=subprocess.STDOUT, text=True))
    for p in procs:
        out, _ = p.communicate(timeout=240)
        assert p.returncode == 0 and "PBT_GLOO_OK" in out, out


# ------------------------------------------------------------------------------------ checkpoint compatibility (8f-2)
def _tiny_gae_model():
    from sample_factory_b200.model import ModelSpec, PolicyModel
    from tests.golden_utils import load_case

    z, meta, ocfg = load_case("tiny_gae")
    spec = ModelSpec(ocfg.obs_dim, ocfg.num_actions, list(ocfg.encoder_mlp_layers), list(ocfg.decoder_mlp_layers),
                     ocfg.nonlinearity, ocfg.normalize_input, ocfg.normalize_returns)
    return z, meta, ocfg, PolicyModel(spec, torch.device("cpu"))


def _ckpt_cfg(tmp_path, ocfg):
    from sample_factory_b200.cfg import default_cfg

    cfg = default_cfg()
    cfg.train_dir, cfg.experiment = str(tmp_path), "ck"
    cfg.adam_eps, cfg.adam_beta1, cfg.adam_beta2 = ocfg.adam_eps, ocfg.adam_beta1, ocfg.adam_beta2
    return cfg


def test_loads_checkpoint_written_by_the_reference(tmp_path):
    """tests/golden/tiny_gae_checkpoint.pth is the file the reference's own Learner.save() (learner.py:323-360) wrote
    after the last golden iteration: resume from it must restore weights, normaliser state, Adam moments, counters."""
    import shutil

    from sample_factory_b200.checkpoint import checkpoint_dir, load_checkpoint
    from tests.golden_utils import GOLDEN_DIR, state_from

    z, meta, ocfg, model = _tiny_gae_model()
    cfg = _ckpt_cfg(tmp_path, ocfg)
    shutil.copy(os.path.join(GOLDEN_DIR, "tiny_gae_checkpoint.pth"),
                os.path.join(checkpoint_dir(cfg, 0), "checkpoint_000000008_512.pth"))
    info = load_checkpoint(cfg, model, torch.device("cpu"))
    assert info["train_step"] == 8 and info["env_steps"] == 512 and info["opt_step"] == 8
    assert info["curr_lr"] == pytest.approx(ocfg.learning_rate)
    ref_state = state_from(z, f"it{meta['iters'] - 1}/state/")
    got = model.state_dict()
    assert set(got.keys()) == set(ref_state.keys())
    for k, v in ref_state.items():
        assert got[k].dtype == v.dtype and torch.equal(got[k].view(v.shape), v), k
    ref_ck = torch.load(os.path.join(GOLDEN_DIR, "tiny_gae_checkpoint.pth"), weights_only=False)
    osd = model.optimizer_state_dict(info["opt_step"], 1e-4, (0.9, 0.999), 1e-6)
    for i, st in ref_ck["optimizer"]["state"].items():
        assert torch.equal(osd["state"][i]["exp_avg"], st["exp_avg"])
        assert torch.equal(osd["state"][i]["exp_avg_sq"], st["exp_avg_sq"])


def test_checkpoint_we_write_has_the_reference_layout(tmp_path):
    """What the reference's loader does with a checkpoint (learner.py:257-310): torch.load -> actor_critic.load_state_dict
    (strict) -> optimizer.load_state_dict.  Ours must go through the same calls: same top-level keys / types as the
    reference's file, same model keys / shapes / dtypes, and torch.optim.Adam must accept the optimizer dict."""
    from types import SimpleNamespace

    from sample_factory_b200.checkpoint import get_checkpoints, load_checkpoint, save_checkpoint
    from tests.golden_utils import GOLDEN_DIR, state_from

    z, meta, ocfg, model = _tiny_gae_model()
    model.load_state_dict(state_from(z, "it0/state/"), strict=True)
    model.exp_avg.normal_(generator=torch.Generator().manual_seed(0))
    model.exp_avg_sq.uniform_(generator=torch.Generator().manual_seed(1))
    cfg = _ckpt_cfg(tmp_path, ocfg)
    learner = SimpleNamespace(policy_id=0, train_step=12, env_steps=768, opt_step=12, curr_lr=5e-5)
    path = save_checkpoint(cfg, model, learner)
    assert os.path.basename(path) == "checkpoint_000000012_768.pth"
    ours = torch.load(path, weights_only=False)
    ref = torch.load(os.path.join(GOLDEN_DIR, "tiny_gae_checkpoint.pth"), weights_only=False)
    assert list(ours.keys()) == list(ref.keys())
    assert {k: type(v) for k, v in ours.items() if k != "model"} == {k: type(v) for k, v in ref.items() if k != "model"}
    assert list(ours["model"].keys()) == list(ref["model"].keys())       # same ORDER: nn.Module.load_state_dict is by name,
    for k, v in ref["model"].items():                                    # optimizer state is by parameter index
        assert ours["model"][k].shape == v.shape and ours["model"][k].dtype == v.dtype, k
    assert set(ours["optimizer"]["param_groups"][0].keys()) == set(ref["optimizer"]["param_groups"][0].keys())
    params = [torch.nn.Parameter(v.clone()) for k, v in ours["model"].items() if "normalizer" not in k]
    opt = torch.optim.Adam(params, lr=1e-4, betas=(0.9, 0.999), eps=1e-6)
    opt.load_state_dict(ours["optimizer"])
    assert opt.param_groups[0]["lr"] == 5e-5 and float(opt.state[params[0]]["step"]) == 12.0
    # keep_checkpoints pruning (learner.py:353-358) and resume of our own file
    for step in (13, 14, 15):
        learner.train_step = learner.opt_step = step
        save_checkpoint(cfg, model, learner)
    assert len(get_checkpoints(os.path.dirname(path))) == cfg.keep_checkpoints
    z2, _, _, model2 = _tiny_gae_model()
    info = load_checkpoint(cfg, model2, torch.device("cpu"))
    assert info["train_step"] == 15 and info["opt_step"] == 15 and info["curr_lr"] == 5e-5
    a, b = model.optimizer_state_dict(15, 0, (0, 0), 0)["state"], model2.optimizer_state_dict(15, 0, (0, 0), 0)["state"]
    assert torch.equal(model2.flat, model.flat)
    assert all(torch.equal(a[i]["exp_avg"], b[i]["exp_avg"]) and torch.equal(a[i]["exp_avg_sq"], b[i]["exp_avg_sq"]) for i in a)


def test_training_info_interface_plumbing():
    """envs/env_utils.py:74-133: TrainingInfoInterface / RewardShapingInterface envs get the runner's training info"""
    from sample_factory_b200.envs import RewardShapingInterface, TrainingInfoInterface, set_training_info

    class Env(TrainingInfoInterface, RewardShapingInterface):
        num_agents = 5

        def __init__(self):
            TrainingInfoInterface.__init__(self)
            self.shaping = None

        def get_default_reward_shaping(self):
            return dict(kill=1.0)

        def set_reward_shaping(self, reward_shaping, agent_idx):
            self.shaping = (reward_shaping, agent_idx)

    e = Env()
    set_training_info(e, dict(approx_total_training_steps=123))
    assert e.training_info["approx_total_training_steps"] == 123 and e.shaping is None
    set_training_info(e, dict(approx_total_training_steps=456, reward_shaping=dict(kill=2.0)))
    assert e.training_info["approx_total_training_steps"] == 456 and e.shaping == (dict(kill=2.0), slice(0, 5))
    set_training_info(object(), dict(approx_total_training_steps=1))     # envs without the interfaces are left alone


def test_enjoy_load_from_checkpoint_cli_overrides(tmp_path):
    """cfg/arguments.py:227-260 semantics of enjoy's config loading: the saved file wins over defaults, explicitly passed
    flags win over the file, parameters the file does not know are taken from the current cfg; a missing file raises."""
    import json

    from sample_factory_b200.cfg import parse_full_cfg, parse_sf_args
    from sample_factory_b200.enjoy import cfg_file, load_from_checkpoint

    argv = ["--env=my_env", "--experiment=exp1", f"--train_dir={tmp_path}", "--eval_deterministic=True", "--rollout=16"]
    parser, _ = parse_sf_args(argv, evaluation=True)
    cfg = parse_full_cfg(parser, argv)
    assert cfg.cli_args["rollout"] == 16 and "gamma" not in cfg.cli_args
    with pytest.raises(Exception, match="Could not load saved parameters"):
        load_from_checkpoint(cfg)
    os.makedirs(os.path.dirname(cfg_file(cfg)), exist_ok=True)
    saved = dict(env="my_env", experiment="exp1", train_dir=str(tmp_path), rollout=64, gamma=0.9, batch_size=4096,
                 encoder_mlp_layers=[64, 64])
    with open(cfg_file(cfg), "w") as f:
        json.dump(saved, f)
    loaded = load_from_checkpoint(cfg)
    assert loaded.rollout == 16                      # passed on the command line: overrides the file
    assert loaded.gamma == 0.9 and loaded.batch_size == 4096 and loaded.encoder_mlp_layers == [64, 64]   # from the file
    assert loaded.eval_deterministic is True         # not in the file: from the current cfg
    assert loaded.max_num_episodes == cfg.max_num_episodes


def test_tensorboard_event_writer_roundtrip(tmp_path):
    """sample_factory_b200/tb_writer.py: TFRecord framing (masked crc32c) + hand-encoded Event protos read back intact"""
    from sample_factory_b200.tb_writer import SummaryWriter, crc32c, read_scalars

    assert crc32c(b"123456789") == 0xE3069283           # the CRC-32C check value
    w = SummaryWriter(str(tmp_path))
    w.add_scalar("perf/_fps", 40.4e6, 131072)
    w.add_scalar("reward/reward", -1.5, 2 ** 40)
    w.add_scalar("train/a_tag_longer_than_127_characters_" + "x" * 120, 3.0, 7)
    w.close()
    got = read_scalars(w.path)
    assert got[0] == (131072, "perf/_fps", np.float32(40.4e6)) and got[1] == (2 ** 40, "reward/reward", -1.5)
    assert got[2][0] == 7 and got[2][2] == 3.0 and len(got[2][1]) > 127
    assert os.path.basename(w.path).startswith("events.out.tfevents.")


def test_pbt_rules_match_the_reference_selection_and_mutation():
    """pbt.py on a fake runner: mutation range, the untouched best, policy 0 never mutated, replacement only across the reward
    gap, the reference's json files"""
    import json
    import random
    import tempfile
    from types import SimpleNamespace

    from sample_factory_b200.pbt import PopulationBasedTraining, perturb_exponential_decay, policy_cfg_file

    random.seed(11)
    cfg = SimpleNamespace(num_policies=4, with_pbt=True, pbt_optimize_gamma=True, pbt_mutation_rate=1.0, pbt_perturb_min=1.1,
                          pbt_perturb_max=1.5, pbt_replace_fraction=0.3, pbt_replace_reward_gap=0.1,
                          pbt_replace_reward_gap_absolute=1e-6, pbt_target_objective="true_objective", pbt_period_env_steps=10,
                          pbt_start_mutation=10, env="my_env", learning_rate=1e-4, exploration_loss_coeff=0.003,
                          value_loss_coeff=0.5, max_grad_norm=4.0, ppo_clip_ratio=0.1, ppo_clip_value=1.0, gamma=0.99,
                          batch_size=1024, rollout=32)
    calls = []
    runner = SimpleNamespace(update_policy_cfg=lambda p, c: calls.append(("cfg", p, dict(c))),
                             update_reward_shaping=lambda p, s: calls.append(("rew", p, s)),
                             replace_policy=lambda p, donor: calls.append(("replace", p, donor)),
                             policy_avg_stats={}, writers={}, env_steps_per_policy=[100] * 4)
    runner.pbt_decide = lambda pbt, p: (pbt.decide(p, pbt.objectives()) if pbt.objectives() is not None else None)
    pbt = PopulationBasedTraining(cfg, runner, log=lambda *a: None)
    with tempfile.TemporaryDirectory() as d:
        pbt.on_init(d, dict(delta=dict(health=(-1.0, 2.0)), kill=5.0))
        assert pbt.policy_cfg[0]["learning_rate"] == 1e-4 and set(pbt.policy_cfg[0]) == {
            "learning_rate", "exploration_loss_coeff", "value_loss_coeff", "max_grad_norm", "ppo_clip_ratio", "ppo_clip_value", "gamma"}
        for p in range(1, 4):       # mutation rate 1: every parameter moved by a factor in [1/1.5, 1/1.1] or [1.1, 1.5]
            ratio = pbt.policy_cfg[p]["learning_rate"] / 1e-4
            assert 1.1 - 1e-9 <= max(ratio, 1 / ratio) <= 1.5 + 1e-9
            assert 0.0 < pbt.policy_cfg[p]["gamma"] < 1.0 and pbt.policy_cfg[p]["gamma"] != 0.99
            assert pbt.policy_reward_shaping[p]["delta"]["health"] != (-1.0, 2.0)
        assert json.load(open(policy_cfg_file(d, 2))) == pbt.policy_cfg[2]
        pbt.on_start()
        assert [c[0] for c in calls].count("cfg") == 4
        # not enough data -> nothing happens
        calls.clear()
        pbt.on_training_step()
        assert not [c for c in calls if c[0] == "replace"] and pbt.last_update == [100] * 4
        # objectives: 3 best, 1 worst (big gap), 2 close to the best, 0 in between
        from collections import deque
        runner.policy_avg_stats["true_objective"] = [deque([2.0]), deque([-3.0]), deque([9.9]), deque([10.0])]
        runner.env_steps_per_policy = [200] * 4
        cfg2, cfg3 = dict(pbt.policy_cfg[2]), dict(pbt.policy_cfg[3])
        calls.clear()
        pbt.on_training_step()
        # ceil(0.3 * 4) = 2: best = {3, 2} (left alone), worst = {0, 1}: both clear the reward gap and take a best member's weights
        repl = {c[1]: c[2] for c in calls if c[0] == "replace"}
        assert set(repl) == {0, 1} and set(repl.values()) <= {2, 3}
        assert pbt.policy_cfg[3] == cfg3 and pbt.policy_cfg[2] == cfg2
        donors = {2: cfg2, 3: cfg3}
        assert pbt.policy_cfg[0] == donors[repl[0]]            # policy 0 is never MUTATED: it takes the donor's parameters as they are
        assert pbt.policy_cfg[1] != donors[repl[1]]            # everybody else gets a mutated copy
        assert json.load(open(policy_cfg_file(d, 1))) == pbt.policy_cfg[1]
        # a small gap: the worst keeps its weights (but still mutates its own parameters)
        runner.policy_avg_stats["true_objective"] = [deque([9.95]), deque([9.9]), deque([9.99]), deque([10.0])]
        runner.env_steps_per_policy = [300] * 4
        calls.clear()
        pbt.on_training_step()
        assert not [c for c in calls if c[0] == "replace"]
    g = [perturb_exponential_decay(0.99, None) for _ in range(200)]
    assert all(0.97 < x < 0.9992 for x in g) and min(g) < 0.99 < max(g)


def test_bench_clock_sampler_counts_only_complete_nvidia_smi_lines():
    """bench.ClockSampler: the median SM clock / throttle reasons come from complete query lines only; `num_samples` is what the
    bench waits on (it keeps the sampler's rollouts running until nvidia-smi has delivered a few samples -- N = 8 lines had none)"""
    import importlib.util

    spec = importlib.util.spec_from_file_location("bench_mod", os.path.join(ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    cs = bench.ClockSampler(0)
    cs.proc = type("P", (), dict(terminate=lambda self: None, wait=lambda self, timeout=None: 0, kill=lambda self: None))()
    cs.lines = ["0, 1965, 1965, 801.2, 0x0000000000000000, Not Active, Not Active, Not Active, Not Active",
                "0, 1950, 1965, 990.0, 0x0000000000000004, Not Active, Not Active, Not Active, Active",
                "garbage", ""]
    assert cs.num_samples() == 2
    info = cs.stop()
    assert info["samples"] == 2 and info["sm_mhz"] == 1957.5 and info["sm_max_mhz"] == 1965.0 and info["reasons"] == ["sw_power_cap"]
