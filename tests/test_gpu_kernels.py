"""Per-kernel parity tests: every libsfb200 entry point (called through the ctypes C ABI) against the CPU oracle
(oracle/appo_oracle.py, itself pinned to the reference by tests/test_oracle_golden.py) on identical seeded inputs.
Tolerances: bit-exact for integer / bool / index outputs and for the pure-elementwise normaliser; 1e-5 abs for fp32
reductions and GEMMs (BASELINE.json north_star)."""
import math

import numpy as np
import pytest
import torch

from oracle import appo_oracle as O

pytestmark = pytest.mark.gpu

TOL = 1e-5


@pytest.fixture(scope="module")
def dev():
    from sample_factory_b200 import ops

    d = torch.device("cuda", 0)
    ops.bind_device(d)
    return d


def _ops():
    from sample_factory_b200 import ops

    return ops


def g(seed):
    return torch.Generator().manual_seed(seed)


# ----------------------------------------------------------------------------------------------- normalizers
@pytest.mark.parametrize("rows,dim", [(1, 4), (257, 64), (1000, 27), (4096, 64)])
def test_normalize_obs_bit_exact(dev, rows, dim):
    ops = _ops()
    x = torch.randn(rows, dim, generator=g(0)) * 3 + 1
    mean = torch.randn(dim, generator=g(1), dtype=torch.float64)
    var = torch.rand(dim, generator=g(2), dtype=torch.float64) * 4 + 0.01
    ref = x.clone()
    O.rms_normalize_(ref, mean, var)
    out = torch.empty_like(x, device=dev)
    ops.normalize_obs(x.to(dev), out, mean.to(dev), var.to(dev))
    assert torch.equal(out.cpu(), ref)
    # sub-mean / scale path (normalize.py:62-67), e.g. Atari obs_scale=255
    ref2 = x.clone()
    ref2.sub_(0.5).mul_(1.0 / 255.0)
    O.rms_normalize_(ref2, mean, var)
    ops.normalize_obs(x.to(dev), out, mean.to(dev), var.to(dev), 0.5, 1.0 / 255.0)
    assert torch.equal(out.cpu(), ref2)


@pytest.mark.parametrize("rows,dim", [(33, 1), (1056, 16), (135168, 64), (5000, 27), (300, 300)])
def test_moments_and_merge(dev, rows, dim):
    ops = _ops()
    x = torch.randn(rows, dim, generator=g(3)) * 2 + 5
    mean = torch.zeros(dim, dtype=torch.float64)
    var = torch.ones(dim, dtype=torch.float64)
    count = torch.ones(1, dtype=torch.float64)
    md, vd, cd = mean.to(dev), var.to(dev), count.to(dev)
    bm = torch.empty(dim, device=dev)
    bv = torch.empty(dim, device=dev)
    ws = torch.empty(ops.moments_workspace_bytes(dim) // 4, device=dev)
    xd = x.to(dev)
    for _ in range(2):  # two successive updates exercise the merge with count > 1
        O.rms_update(mean, var, count, x)
        ops.batch_moments(xd, bm, bv, ws)
        ops.rms_merge(md, vd, cd, bm, bv, float(rows))
    np.testing.assert_allclose(bm.cpu().numpy(), x.mean(0).numpy(), rtol=2e-6, atol=2e-6)
    np.testing.assert_allclose(bv.cpu().numpy(), x.var(0).numpy(), rtol=2e-5, atol=1e-6)
    np.testing.assert_allclose(md.cpu().numpy(), mean.numpy(), rtol=1e-6, atol=2e-6)
    np.testing.assert_allclose(vd.cpu().numpy(), var.numpy(), rtol=2e-5, atol=1e-6)
    assert cd.item() == count.item()


def test_returns_normalizer_roundtrip(dev):
    """reference tests/algo/test_rms.py:11-68: normalize -> denormalize round trip (atol 1e-6 x scale)."""
    ops = _ops()
    x = torch.randn(100000, generator=g(4)) * 0.8 + 0.3
    mean = torch.tensor([0.25], dtype=torch.float64)
    var = torch.tensor([0.7], dtype=torch.float64)
    ref = x.clone()
    O.rms_normalize_(ref, mean, var)
    xd = x.to(dev)
    ops.rms_apply_scalar(xd, mean.to(dev), var.to(dev), denormalize=False)
    assert torch.equal(xd.cpu(), ref)
    ops.rms_apply_scalar(xd, mean.to(dev), var.to(dev), denormalize=True)
    np.testing.assert_allclose(xd.cpu().numpy(), x.numpy(), atol=2e-6)
    ref_d = ref.clone()
    O.rms_denormalize_(ref_d, mean, var)
    assert torch.equal(xd.cpu(), ref_d)


# ----------------------------------------------------------------------------------------------- GEMM layers
@pytest.mark.parametrize("M,N,K,act", [(1, 8, 4, "elu"), (300, 70, 37, "elu"), (4096, 512, 64, "elu"),
                                       (1000, 512, 512, "relu"), (513, 129, 256, "tanh"), (128, 64, 16, "none")])
@pytest.mark.parametrize("engine", ["simt", "3xtf32"])
def test_linear_act_forward(dev, M, N, K, act, engine):
    ops = _ops()
    if engine != "simt" and not ops.tc_available():
        pytest.skip("tcgen05 engine not built")
    x = torch.randn(M, K, generator=g(5))
    W = torch.randn(N, K, generator=g(6)) / math.sqrt(K)
    b = torch.randn(N, generator=g(7)) * 0.1
    cfg = O.OracleCfg(nonlinearity=act if act != "none" else "elu")
    z = torch.nn.functional.linear(x.double(), W.double(), b.double())
    ref = (O._act(cfg, z) if act != "none" else z).float()
    out = torch.empty(M, N, device=dev)
    ops.linear_act_forward(x.to(dev), W.to(dev), b.to(dev), out, ops.ACT[act], ops.ENGINES[engine])
    np.testing.assert_allclose(out.cpu().numpy(), ref.numpy(), atol=TOL, rtol=1e-5)


def test_tc_engine_precision_classes(dev):
    """tcgen05 engine: the 3xTF32 split must be fp32-grade (same error class as the exact-fp32 CUDA-core engine),
    the single-pass TF32 mode must be visibly coarser (proves the tensor-core path really ran and the split matters)."""
    ops = _ops()
    if not ops.tc_available():
        pytest.skip("tcgen05 engine not available")
    M, N, K = 2048, 512, 512
    x = torch.randn(M, K, generator=g(70))
    W = torch.randn(N, K, generator=g(71)) / math.sqrt(K)
    b = torch.zeros(N)
    ref = torch.nn.functional.linear(x.double(), W.double()).float()
    errs = {}
    for name in ("simt", "3xtf32", "tf32"):
        out = torch.empty(M, N, device=dev)
        ops.linear_act_forward(x.to(dev), W.to(dev), b.to(dev), out, ops.ACT["none"], ops.ENGINES[name])
        errs[name] = (out.cpu() - ref).abs().max().item()
    print("max abs error vs fp64 (|out| up to ~4.5):", errs)
    scale = ref.abs().max().item()
    assert errs["simt"] < 1e-5 and errs["3xtf32"] < 3e-6 * scale, errs   # fp32-grade: <= ~25 ulp of the largest output
    assert errs["tf32"] > 20 * errs["3xtf32"] and errs["tf32"] < 2e-2, errs


@pytest.mark.parametrize("M,N,K,amp", [(2048, 512, 512, 1.0), (4096, 512, 64, 1.0), (32768, 512, 512, 1.0), (2048, 256, 512, 1e-6),
                                        (1000, 384, 128, 300.0)])
def test_fp16_split_engine_is_fp32_grade(dev, M, N, K, amp):
    """The fp16-split form of the 3-pass engine (registered fp16 weight twins + a registered activation bound): same
    accuracy class as 3xTF32 against fp64 -- forward (with bias / ELU), and dX through the transposed twins -- for
    activations of very different magnitudes (the bound sets the power-of-two operand shift) and a loose bound."""
    ops = _ops()
    if not ops.tc_available():
        pytest.skip("tcgen05 engine not available")
    x = (torch.randn(M, K, generator=g(170)) * amp).to(dev)
    W = (torch.randn(N, K, generator=g(171)) / math.sqrt(K)).to(dev).contiguous()
    b = (torch.randn(N, generator=g(172)) * 0.1 * amp).to(dev)
    # (the epilogue's ELU is exp(z) - 1 with 2.4e-7 ABSOLUTE error: not the subject here, so tiny outputs go without it)
    act = "elu" if amp >= 1e-3 else "none"
    ref = torch.nn.functional.linear(x.double(), W.double(), b.double())
    if act == "elu":
        ref = torch.nn.functional.elu(ref)
    scale = max(ref.abs().max().item(), 1e-30)
    out_tf32 = torch.empty(M, N, device=dev)
    ops.linear_act_forward(x, W, b, out_tf32, ops.ACT[act], ops.GEMM_TC_3XTF32)
    err_tf32 = (out_tf32.double() - ref).abs().max().item()
    twins = torch.empty(2 * W.numel(), dtype=torch.float16, device=dev)
    twinsT = torch.empty(2 * W.numel(), dtype=torch.float16, device=dev)
    bound = torch.full((1,), float(x.abs().max().item()) * 3.0, device=dev)        # a loose bound is as good as a tight one
    n0 = ops.launch_count()
    ops.register_f16_twins(W.view(-1), twins)
    ops.register_f16_transposed(W, twinsT)
    ops.register_operand_bound(x, bound)
    try:
        # the twins are what they claim to be
        hi, lo = twins[: W.numel()].float().view(N, K), twins[W.numel():].float().view(N, K)
        np.testing.assert_allclose(((hi + lo / 2048.0) / 256.0).cpu().numpy(), W.cpu().numpy(), rtol=3e-7, atol=1e-12)
        hiT = twinsT[: W.numel()].float().view(K, N)
        assert torch.equal(hiT, hi.t())
        out = torch.empty(M, N, device=dev)
        ops.linear_act_forward(x, W, b, out, ops.ACT[act], ops.GEMM_TC_3XTF32)
        err = (out.double() - ref).abs().max().item()
        print(f"forward  max abs err vs fp64 (scale {scale:.3g}): fp16-split {err:.3e}   3xTF32 {err_tf32:.3e}")
        assert err < 3e-6 * scale, (err, scale)
        assert not torch.equal(out, out_tf32), "the fp16-split kernel did not run (bit-identical to the tf32 split)"
        # dX = dz . W (* act'(x)) with the transposed twins; dz carries its own bound
        dz = (torch.randn(M, N, generator=g(173)) * amp * 1e-3).to(dev)
        dbound = torch.full((1,), float(dz.abs().max().item()), device=dev)
        ops.register_operand_bound(dz, dbound)
        xa = torch.nn.functional.elu(torch.randn(M, K, generator=g(174))).to(dev)
        ws = torch.empty(ops.linear_backward_workspace_bytes(M, N, K) // 4 + 4, device=dev)
        dx = torch.empty(M, K, device=dev)
        ops.linear_backward(dz, xa, W, ops.ACT["elu"], None, dx, None, ops.GEMM_TC_3XTF32, ws)
        dref = (dz.double() @ W.double()) * torch.where(xa > 0, torch.ones_like(xa), xa + 1).double()
        derr = (dx.double() - dref).abs().max().item()
        dscale = dref.abs().max().item()
        print(f"dX       max abs err vs fp64 (scale {dscale:.3g}): fp16-split {derr:.3e}")
        assert derr < 3e-6 * dscale, (derr, dscale)
        ops.unregister_operand_bound(dz)
    finally:
        ops.unregister_operand_bound(x)
        ops.unregister_f16_transposed(W)
        ops.unregister_f16_twins(W.view(-1))
    assert ops.launch_count() > n0


def test_linear_out_bound(dev):
    ops = _ops()
    W = torch.randn(96, 40, generator=g(180)).to(dev)
    b = torch.randn(96, generator=g(181)).to(dev)
    inb = torch.full((1,), 5.0, device=dev)
    out = torch.zeros(4, device=dev)
    for _ in range(2):          # (second launch: the scratch words were left at zero)
        ops.linear_out_bound(W, b, inb, out, ops.ACT["elu"])
        expect = (5.0 * W.abs().sum(1) + b.abs()).max().item()
        assert expect <= out[0].item() <= expect * 1.001 and out[1:3].abs().sum().item() == 0
    x = (torch.rand(4096, 40, generator=g(182)) * 10 - 5).to(dev)
    assert torch.nn.functional.elu(torch.nn.functional.linear(x, W, b)).abs().max().item() <= out[0].item()
    ops.linear_out_bound(W, b, inb, out, ops.ACT["tanh"])
    assert out[0].item() == 1.0
    # the dz bound of heads_backward
    dl = torch.randn(5000, 6, generator=g(183)).to(dev) * 1e-4
    dv = torch.randn(5000, generator=g(184)).to(dev) * 1e-4
    Wv = torch.randn(1, 96, generator=g(185)).to(dev)
    Wa = torch.randn(6, 96, generator=g(186)).to(dev)
    zb = torch.zeros(4, device=dev)
    for _ in range(2):
        ops.heads_dz_bound(dl, dv, Wv, Wa, zb)
        expect = (dv.abs() + dl.abs().sum(1)).max().item() * max(Wv.abs().max().item(), Wa.abs().max().item())
        assert expect <= zb[0].item() <= expect * 1.001 and zb[1:3].abs().sum().item() == 0
    dz = (dv[:, None] * Wv + dl @ Wa)
    assert dz.abs().max().item() <= zb[0].item()


def test_linear_forward_strided_input(dev):
    """The learner feeds obs[:, T] rows in place: x row stride != K."""
    ops = _ops()
    base = torch.randn(64, 9, 32, generator=g(8))
    x = base[:, 8]
    W = torch.randn(48, 32, generator=g(9)) / 6
    b = torch.zeros(48)
    ref = torch.nn.functional.elu(torch.nn.functional.linear(x, W, b))
    bd = base.to(dev)
    out = torch.empty(64, 48, device=dev)
    ops.linear_act_forward(bd[:, 8], W.to(dev), b.to(dev), out, ops.ACT["elu"], ops.GEMM_SIMT)
    np.testing.assert_allclose(out.cpu().numpy(), ref.numpy(), atol=TOL)


@pytest.mark.parametrize("M,N,K,act_prev", [(64, 8, 4, "elu"), (1000, 70, 37, "elu"), (4096, 512, 512, "elu"),
                                            (2048, 512, 64, "none"), (777, 130, 260, "tanh"), (4096, 256, 256, "none"),
                                            (8192, 128, 384, "relu")])
@pytest.mark.parametrize("engine", ["simt", "3xtf32"])
def test_linear_backward(dev, M, N, K, act_prev, engine):
    ops = _ops()
    if engine != "simt" and not ops.tc_available():
        pytest.skip("tcgen05 engine not built")
    dz = torch.randn(M, N, generator=g(10)) / M
    # x is the previous layer's OUTPUT: make it a genuine activation output so act'(x) is well defined
    pre = torch.randn(M, K, generator=g(11))
    cfg = O.OracleCfg(nonlinearity=act_prev if act_prev != "none" else "elu")
    x = O._act(cfg, pre) if act_prev != "none" else pre
    W = torch.randn(N, K, generator=g(12)) / math.sqrt(K)
    dW_ref = (dz.double().t() @ x.double()).float()
    dxl = (dz.double() @ W.double())
    if act_prev == "elu":
        d = torch.where(pre > 0, torch.ones_like(pre), torch.exp(pre)).double()
    elif act_prev == "tanh":
        d = (1 - torch.tanh(pre) ** 2).double()
    elif act_prev == "relu":
        d = (pre > 0).double()
    else:
        d = torch.ones_like(pre).double()
    dx_ref = (dxl * d).float()
    db_ref = dx_ref.double().sum(0).float()
    dW = torch.empty(N, K, device=dev)
    dx = torch.empty(M, K, device=dev)
    dbp = torch.empty(K, device=dev)
    ws = torch.empty(ops.linear_backward_workspace_bytes(M, N, K) // 4 + 4, device=dev)
    ops.linear_backward(dz.to(dev), x.to(dev), W.to(dev), ops.ACT[act_prev], dW, dx, dbp, ops.ENGINES[engine], ws)
    np.testing.assert_allclose(dW.cpu().numpy(), dW_ref.numpy(), atol=TOL, rtol=1e-4)
    np.testing.assert_allclose(dx.cpu().numpy(), dx_ref.numpy(), atol=TOL, rtol=1e-4)
    np.testing.assert_allclose(dbp.cpu().numpy(), db_ref.numpy(), atol=TOL, rtol=1e-4)


# ----------------------------------------------------------------------------------------------- heads
@pytest.mark.parametrize("rows,H,A", [(5, 64, 8), (4096, 512, 8), (1001, 96, 3), (257, 128, 17), (64, 512, 31)])
def test_heads_forward_and_sampling(dev, rows, H, A):
    ops = _ops()
    h = torch.randn(rows, H, generator=g(13))
    Wv = torch.randn(1, H, generator=g(14)) / math.sqrt(H)
    bv = torch.randn(1, generator=g(15))
    Wa = torch.randn(A, H, generator=g(16)) / math.sqrt(H) * 2
    ba = torch.randn(A, generator=g(17)) * 0.1
    noise = torch.empty(rows, A).exponential_(generator=g(18))
    values_ref = torch.nn.functional.linear(h, Wv, bv).squeeze(-1)
    logits_ref = torch.nn.functional.linear(h, Wa, ba)

    T = 3  # write into strided "trajectory slots" like the sampler does
    values = torch.zeros(rows, T + 1, device=dev)
    logits = torch.zeros(rows, T, A, device=dev)
    actions = torch.zeros(rows, T, 1, device=dev)
    logp = torch.zeros(rows, T, device=dev)
    pv = torch.zeros(rows, T, device=dev)
    env_actions = torch.zeros(rows, dtype=torch.int32, device=dev)
    pvs = torch.tensor([7.0], device=dev)
    t = 1
    ops.heads_forward(h.to(dev), Wv.to(dev), bv.to(dev), Wa.to(dev), ba.to(dev), values[:, t], values.stride(0),
                      logits[:, t], logits.stride(0), noise.to(dev), 0, 0, None, actions[:, t], actions.stride(0),
                      env_actions, logp[:, t], logp.stride(0), pvs, pv[:, t], pv.stride(0))
    np.testing.assert_allclose(values[:, t].cpu().numpy(), values_ref.numpy(), atol=TOL)
    np.testing.assert_allclose(logits[:, t].cpu().numpy(), logits_ref.numpy(), atol=TOL)
    # sampling is checked on the DEVICE logits (feeding identical logits to both sides, SURVEY section 7 hard parts)
    dl = logits[:, t].cpu()
    a_ref = O.cat_sample(dl, noise)
    assert torch.equal(env_actions.cpu().long(), a_ref.view(-1)), "action indices must be bit-exact"
    assert torch.equal(actions[:, t, 0].cpu(), a_ref.view(-1).float())
    np.testing.assert_allclose(logp[:, t].cpu().numpy(), O.cat_log_prob(dl, a_ref).numpy(), atol=2e-6)
    assert torch.all(pv[:, t] == 7.0) and torch.all(pv[:, 0] == 0) and torch.all(values[:, 0] == 0)


@pytest.mark.parametrize("rows,H,A", [(257, 64, 7), (4096, 128, 8), (100, 96, 31)])
def test_heads_action_mask_and_deterministic(dev, rows, H, A):
    """masked_softmax / masked_log_softmax sampling (action_distributions.py:84-95,135-143) incl. rows that allow nothing,
    and deterministic (argmax) actions (enjoy.py:165-171), through both heads entry points."""
    ops = _ops()
    h = torch.randn(rows, H, generator=g(113))
    Wv = torch.randn(1, H, generator=g(114)) / math.sqrt(H)
    bv = torch.randn(1, generator=g(115))
    Wa = torch.randn(A, H, generator=g(116)) / math.sqrt(H) * 2
    ba = torch.randn(A, generator=g(117)) * 0.1
    noise = torch.empty(rows, A).exponential_(generator=g(118))
    mask = (torch.rand(rows, A, generator=g(119)) < 0.4)
    mask[::13] = False                       # nothing allowed -> the reference's uniform 1e-6 fallback
    mask[1::13] = True                       # everything allowed
    values = torch.zeros(rows, device=dev)
    logits = torch.zeros(rows, A, device=dev)
    actions = torch.zeros(rows, 1, device=dev)
    logp = torch.zeros(rows, device=dev)
    env_actions = torch.zeros(rows, dtype=torch.int32, device=dev)
    args = (h.to(dev), Wv.to(dev), bv.to(dev), Wa.to(dev), ba.to(dev), values, 1, logits, A, noise.to(dev), 0, 0, None,
            actions, 1, env_actions, logp, 1)
    mask_dev = mask.to(dev)

    def partials_call(noise_dev):
        # the same tail behind heads_from_partials: one "partial" holding the finished dot products, zero biases
        part = torch.zeros(rows, ops.HEAD_PART_PAD, device=dev)
        part[:, 0] = values
        part[:, 1:A + 1] = logits
        ops.heads_from_partials(part.view(-1), 1, rows, torch.zeros(1, device=dev), torch.zeros(A, device=dev), values, 1,
                                None, 0, noise_dev, 0, 0, None, actions, 1, env_actions, logp, 1)

    try:
        ops.set_sampling_mode(mask_dev, False)
        ops.heads_forward(*args)
        dl = logits.cpu()
        m64 = mask.to(torch.int64)
        a_ref = O.masked_cat_sample(dl, m64, noise)
        lp_ref = O.masked_cat_log_prob(dl, m64, a_ref)
        assert torch.equal(env_actions.cpu().long(), a_ref.view(-1)), "masked action indices must be bit-exact"
        allowed = mask.gather(1, a_ref) | ~mask.any(1, keepdim=True)
        assert bool(allowed.all())
        np.testing.assert_allclose(logp.cpu().numpy(), lp_ref.numpy(), atol=2e-6, rtol=1e-6)
        if A + 1 <= ops.HEAD_PART_PAD:
            env_actions.zero_(); logp.zero_()
            partials_call(noise.to(dev))
            assert torch.equal(env_actions.cpu().long(), a_ref.view(-1))
            np.testing.assert_allclose(logp.cpu().numpy(), lp_ref.numpy(), atol=2e-6, rtol=1e-6)
        # deterministic + mask: argmax of the masked probabilities; no noise consumed (Philox path would otherwise run)
        ops.set_sampling_mode(mask_dev, True)
        ops.heads_forward(*args[:9], None, 0, 0, None, *args[13:])
        p = O.masked_cat_probs(dl, m64)
        p = torch.where((p.sum(-1) == 0).unsqueeze(-1), torch.full_like(p, 1e-6), p)
        assert torch.equal(env_actions.cpu().long(), torch.argmax(p, -1))
        # deterministic, no mask
        ops.set_sampling_mode(None, True)
        ops.heads_forward(*args[:9], None, 0, 0, None, *args[13:])
        assert torch.equal(env_actions.cpu().long(), torch.argmax(O.cat_probs(dl), -1))
        np.testing.assert_allclose(logp.cpu().numpy(), O.cat_log_probs(dl).max(-1).values.numpy(), atol=2e-6)
    finally:
        ops.set_sampling_mode(None, False)
    # back to the default: plain sampling again
    ops.heads_forward(*args)
    assert torch.equal(env_actions.cpu().long(), O.cat_sample(logits.cpu(), noise).view(-1))


def test_heads_deterministic_continuous_and_mask_errors(dev):
    ops = _ops()
    rows, H, Ad = 300, 64, 5
    h = torch.randn(rows, H, generator=g(120)).to(dev)
    Wv = (torch.randn(1, H, generator=g(121)) / 8).to(dev)
    Wa = (torch.randn(2 * Ad, H, generator=g(122)) / 8).to(dev)
    bv, ba = torch.zeros(1, device=dev), torch.zeros(2 * Ad, device=dev)
    values = torch.zeros(rows, device=dev)
    params = torch.zeros(rows, 2 * Ad, device=dev)
    actions = torch.zeros(rows, Ad, device=dev)
    logp = torch.zeros(rows, device=dev)
    call = lambda: ops.heads_forward_continuous(h, Wv, bv, Wa, ba, Ad, True, None, 0.0, values, 1, params, 2 * Ad, None, 3, 0,
                                                None, actions, Ad, None, logp, 1)
    try:
        ops.set_sampling_mode(None, True)
        call()
        assert torch.equal(actions, params[:, :Ad]), "deterministic Gaussian actions are the means"
        np.testing.assert_allclose(logp.cpu().numpy(), O.gauss_log_prob(params.cpu(), actions.cpu()).numpy(), atol=1e-5, rtol=1e-5)
        ops.set_sampling_mode(torch.ones(rows, 2 * Ad, dtype=torch.bool, device=dev), False)
        with pytest.raises(Exception, match="plain Discrete"):
            call()
    finally:
        ops.set_sampling_mode(None, False)


def test_heads_philox_sampling_distribution(dev):
    """Production path: in-kernel Philox Exp(1) noise. Empirical action frequencies must match softmax(logits)."""
    ops = _ops()
    rows, H, A = 200000, 32, 8
    h = torch.zeros(rows, H)
    h[:, 0] = 1.0
    Wa = torch.zeros(A, H)
    Wa[:, 0] = torch.tensor([0.0, 0.5, 1.0, 1.5, -1.0, 2.0, 0.2, -0.3])
    p_ref = torch.softmax(Wa[:, 0], 0)
    values = torch.empty(rows, device=dev)
    actions = torch.empty(rows, device=dev)
    env_actions = torch.empty(rows, dtype=torch.int32, device=dev)
    cnt = torch.tensor([5], dtype=torch.int64, device=dev)
    z1 = torch.zeros(1, device=dev)
    for seed, off in [(1, None), (1, cnt), (2, None)]:
        ops.heads_forward(h.to(dev), torch.zeros(1, H, device=dev), z1, Wa.to(dev), torch.zeros(A, device=dev), values, 1,
                          None, 0, None, seed, 0, off, actions, 1, env_actions)
        freq = torch.bincount(env_actions.cpu().long(), minlength=A).float() / rows
        np.testing.assert_allclose(freq.numpy(), p_ref.numpy(), atol=5e-3)
        if seed == 1 and off is None:
            first = env_actions.clone()
        elif seed == 1:
            assert (env_actions != first).float().mean() > 0.3, "device-side offset must change the stream"


@pytest.mark.parametrize("rows,H,A,act", [(64, 64, 8, "elu"), (32768, 512, 8, "elu"), (1000, 96, 3, "relu"),
                                          (20011, 256, 8, "relu"), (16500, 128, 5, "tanh"), (16384, 512, 2, "elu"),
                                          (555, 300, 17, "tanh")])
def test_heads_backward(dev, rows, H, A, act):
    ops = _ops()
    cfg = O.OracleCfg(nonlinearity=act)
    pre = torch.randn(rows, H, generator=g(19))
    h = O._act(cfg, pre)
    Wv = torch.randn(1, H, generator=g(20)) / math.sqrt(H)
    Wa = torch.randn(A, H, generator=g(21)) / math.sqrt(H)
    dlogits = torch.randn(rows, A, generator=g(22)) / rows
    dvalues = torch.randn(rows, generator=g(23)) / rows
    dh = dlogits.double() @ Wa.double() + dvalues.double()[:, None] * Wv.double()
    if act == "elu":
        d = torch.where(pre > 0, torch.ones_like(pre), torch.exp(pre)).double()
    elif act == "relu":
        d = (pre > 0).double()
    else:
        d = (1 - torch.tanh(pre) ** 2).double()
    dz_ref = (dh * d).float()
    dz = torch.empty(rows, H, device=dev)
    dWv = torch.empty(H, device=dev)
    dbv = torch.empty(1, device=dev)
    dWa = torch.empty(A, H, device=dev)
    dba = torch.empty(A, device=dev)
    dbp = torch.empty(H, device=dev)
    ws = torch.empty(ops.heads_backward_workspace_bytes(H, A) // 4 + 4, device=dev)
    ops.heads_backward(h.to(dev), Wv.to(dev).view(-1), Wa.to(dev), dlogits.to(dev), dvalues.to(dev), ops.ACT[act], dz,
                       dWv, dbv, dWa, dba, dbp, ws)
    np.testing.assert_allclose(dz.cpu().numpy(), dz_ref.numpy(), atol=TOL, rtol=1e-4)
    np.testing.assert_allclose(dWa.cpu().numpy(), (dlogits.double().t() @ h.double()).float().numpy(), atol=TOL, rtol=1e-4)
    np.testing.assert_allclose(dWv.cpu().numpy(), (dvalues.double() @ h.double()).float().numpy(), atol=TOL, rtol=1e-4)
    np.testing.assert_allclose(dba.cpu().numpy(), dlogits.double().sum(0).float().numpy(), atol=TOL, rtol=1e-4)
    np.testing.assert_allclose(dbv.cpu().numpy(), dvalues.double().sum().float().numpy(), atol=TOL, rtol=1e-4)
    np.testing.assert_allclose(dbp.cpu().numpy(), dz_ref.double().sum(0).float().numpy(), atol=TOL, rtol=1e-4)


# ----------------------------------------------------------------------------------------------- sampler steps
def test_sampler_pre_post_step_and_env(dev):
    ops = _ops()
    N, D, T, A = 300, 16, 5, 8
    obs = torch.randn(N, D, generator=g(24))
    mean = torch.randn(D, generator=g(25), dtype=torch.float64)
    var = torch.rand(D, generator=g(26), dtype=torch.float64) + 0.1
    traj_obs = torch.full((N, T + 1, D), -1.0, device=dev)
    traj_rnn = torch.full((N, T + 1, 1), -1.0, device=dev)
    rnn = torch.zeros(N, 1, device=dev)
    xn = torch.empty(N, D, device=dev)
    t = 2
    ops.sampler_pre_step(obs.to(dev), traj_obs[:, t], rnn, traj_rnn[:, t], xn, mean.to(dev), var.to(dev), 0.0, 1.0)
    ref = obs.clone()
    O.rms_normalize_(ref, mean, var)
    assert torch.equal(xn.cpu(), ref)
    assert torch.equal(traj_obs[:, t].cpu(), obs) and torch.all(traj_obs[:, t + 1] == -1) and torch.all(traj_obs[:, t - 1] == -1)
    assert torch.all(traj_rnn[:, t] == 0) and torch.all(traj_rnn[:, t + 1] == -1)

    # tape env vs the oracle's env, several steps, device-side step counter
    L = 7
    tape = torch.randn(L, N, D, generator=g(27))
    env_ref = O.TapeVecEnv(tape, A)
    env_ref.reset()
    from sample_factory_b200.envs import TapeVecEnv

    env = TapeVecEnv(tape.to(dev), A)
    assert torch.equal(env.reset().cpu(), tape[0])
    rew_t = torch.zeros(N, T, device=dev)
    done_t = torch.zeros(N, T, dtype=torch.bool, device=dev)
    to_t = torch.zeros(N, T, dtype=torch.bool, device=dev)
    pid_t = torch.full((N, T), -1, dtype=torch.int32, device=dev)
    ep_ret = torch.zeros(N, device=dev)
    ep_len = torch.zeros(N, dtype=torch.int32, device=dev)
    ep_min = torch.full((N,), float("inf"), device=dev)
    ep_max = torch.full((N,), float("-inf"), device=dev)
    stats = torch.zeros(8, dtype=torch.float64, device=dev)
    counter = torch.zeros(1, dtype=torch.int64, device=dev)
    ref_ret = torch.zeros(N)
    ref_len = torch.zeros(N)
    fin_cnt, fin_ret, fin_len = 0, 0.0, 0.0
    for step in range(T):
        a = torch.randint(0, A, (N,), generator=g(100 + step), dtype=torch.int32)
        o_ref, r_ref, tm_ref, tr_ref = env_ref.step(a)
        o, r, tm, tr = env.step(a.to(dev))
        assert torch.equal(o.cpu(), o_ref) and torch.equal(r.cpu(), r_ref)
        assert torch.equal(tm.cpu(), tm_ref) and torch.equal(tr.cpu(), tr_ref)
        ops.sampler_post_step(r, tm, tr, 0.7, 0.5, 0, rew_t[:, step], done_t[:, step], to_t[:, step], pid_t[:, step],
                              ep_ret, ep_len, ep_min, ep_max, 1, stats, counter)
        d_ref = tm_ref | tr_ref
        assert torch.equal(rew_t[:, step].cpu(), (r_ref * 0.7).clamp(-0.5, 0.5))
        assert torch.equal(done_t[:, step].cpu(), d_ref) and torch.equal(to_t[:, step].cpu(), tr_ref)
        ref_ret += r_ref
        ref_len += 1
        fin_cnt += int(d_ref.sum())
        fin_ret += float(ref_ret[d_ref].sum())
        fin_len += float(ref_len[d_ref].sum())
        ref_ret[d_ref] = 0
        ref_len[d_ref] = 0
    assert torch.all(pid_t == 0) and counter.item() == T and env.step_counter[0].item() == T
    assert env.step_counter[1].item() == 0
    s = stats.cpu()
    assert int(s[0]) == fin_cnt and abs(s[1].item() - fin_ret) < 1e-3 and abs(s[2].item() - fin_len) < 1e-6
    np.testing.assert_allclose(ep_ret.cpu().numpy(), ref_ret.numpy(), atol=1e-6)


def test_compute_valids(dev):
    ops = _ops()
    N, T = 200, 9
    pid = torch.randint(-1, 2, (N, T), generator=g(28), dtype=torch.int32)
    pver = torch.randint(0, 50, (N, T), generator=g(29)).float()
    valids = torch.zeros(N, T + 1, dtype=torch.bool, device=dev)
    ops.compute_valids(pid.to(dev), pver.to(dev), 0, 40, 25, valids)
    ref = torch.zeros(N, T + 1, dtype=torch.bool)
    ref[:, :-1] = (pid == 0) & (40 - pver < 25)
    ref[:, -1] = ref[:, -2]
    assert torch.equal(valids.cpu(), ref)


# ----------------------------------------------------------------------------------------------- time-axis scans
@pytest.mark.parametrize("N,T", [(7, 1), (257, 8), (4096, 32), (100, 50), (33, 128)])
@pytest.mark.parametrize("bootstrap,denorm", [(False, False), (True, True)])
def test_gae_returns(dev, N, T, bootstrap, denorm):
    ops = _ops()
    rewards = torch.randn(N, T, generator=g(30))
    dones = torch.rand(N, T, generator=g(31)) < 0.1
    time_outs = dones & (torch.rand(N, T, generator=g(32)) < 0.5)
    values = torch.randn(N, T + 1, generator=g(33))
    valids = torch.rand(N, T + 1, generator=g(34)) < 0.8
    mean = torch.tensor([0.3], dtype=torch.float64)
    var = torch.tensor([2.5], dtype=torch.float64)
    gamma, lam = 0.99, 0.95
    dv = values.clone()
    if denorm:
        O.rms_denormalize_(dv, mean, var)
    r = rewards.clone()
    if bootstrap:
        r.add_(gamma * dv[:, :-1] * time_outs * dones)
    adv_ref = O.gae_advantages(r, dones, dv, valids, gamma, lam)
    ret_ref = adv_ref + valids[:, :-1] * dv[:, :-1]
    rd = rewards.to(dev)
    adv = torch.empty(N, T, device=dev)
    ret = torch.empty(N, T, device=dev)
    ops.gae_returns(rd, dones.to(dev), time_outs.to(dev), values.to(dev), valids.to(dev), gamma, lam, bootstrap,
                    mean.to(dev) if denorm else None, var.to(dev) if denorm else None, adv, ret)
    assert torch.equal(rd.cpu(), r), "value-bootstrapped rewards must match bit for bit"
    np.testing.assert_allclose(adv.cpu().numpy(), adv_ref.numpy(), atol=TOL, rtol=1e-5)
    np.testing.assert_allclose(ret.cpu().numpy(), ret_ref.numpy(), atol=TOL, rtol=1e-5)


@pytest.mark.parametrize("n,R", [(5, 2), (300, 8), (1024, 32), (50, 40)])
def test_vtrace(dev, n, R):
    ops = _ops()
    cfg = O.OracleCfg(gamma=0.99, vtrace_rho=1.0, vtrace_c=0.9)
    ratio = torch.exp(torch.randn(n * R, generator=g(35)) * 0.3).clamp(0.05, 20)
    values = torch.randn(n * R, generator=g(36))
    rewards = torch.randn(n * R, generator=g(37))
    dones = torch.rand(n * R, generator=g(38)) < 0.1
    vs_ref, adv_ref = O.vtrace(cfg, ratio, values, rewards, dones.float(), R)
    vs = torch.empty(n * R, device=dev)
    adv = torch.empty(n * R, device=dev)
    ops.vtrace(ratio.to(dev), values.to(dev), rewards.to(dev), dones.to(dev), R, cfg.gamma, cfg.vtrace_rho, cfg.vtrace_c,
               vs, adv)
    np.testing.assert_allclose(vs.cpu().numpy(), vs_ref.numpy(), atol=TOL, rtol=1e-5)
    np.testing.assert_allclose(adv.cpu().numpy(), adv_ref.numpy(), atol=TOL, rtol=1e-5)


# ----------------------------------------------------------------------------------------------- loss
@pytest.mark.parametrize("expl", ["entropy", "symmetric_kl"])
@pytest.mark.parametrize("B,A,frac_invalid,kl_coeff", [(64, 8, 0.0, 0.0), (1000, 8, 0.2, 0.1), (32768, 8, 0.0, 0.0),
                                                       (777, 3, 0.3, 0.5), (513, 17, 0.1, 0.2)])
def test_ppo_loss_fwd_bwd(dev, B, A, frac_invalid, kl_coeff, expl):
    ops = _ops()
    cfg = O.OracleCfg(num_actions=A, kl_loss_coeff=kl_coeff, ppo_clip_ratio=0.1, ppo_clip_value=0.2, exploration_loss=expl,
                      exploration_loss_coeff=0.003 if expl == "entropy" else 0.02)
    logits = (torch.randn(B, A, generator=g(39)) * 1.5).requires_grad_(True)
    values = torch.randn(B, generator=g(40)).requires_grad_(True)
    logits_old = logits.detach() + torch.randn(B, A, generator=g(41)) * 0.3
    actions = torch.randint(0, A, (B, 1), generator=g(42)).float()
    lp_old = O.cat_log_prob(logits_old, actions) + torch.randn(B, generator=g(43)) * 0.05
    v_old = values.detach() + torch.randn(B, generator=g(44)) * 0.3
    adv = torch.randn(B, generator=g(45)) * 2 + 0.5
    targets = torch.randn(B, generator=g(46))
    valids = torch.rand(B, generator=g(47)) >= frac_invalid
    num_invalids = int((~valids).sum())

    # oracle losses with logits/values as autograd leaves (same formulas as O.calculate_losses :588-657)
    clip_hi = 1.0 + cfg.ppo_clip_ratio
    clip_lo = 1.0 / clip_hi
    lp = O.cat_log_prob(logits, actions)
    ratio = torch.clamp(torch.exp(lp - lp_old), 0.05, 20.0)
    adv_std, adv_mean = torch.std_mean(O._masked_select(adv, valids, num_invalids))
    advn = (adv - adv_mean) / torch.clamp_min(adv_std, 1e-7)
    pl = -O._masked_select(torch.min(ratio * advn, torch.clamp(ratio, clip_lo, clip_hi) * advn), valids, num_invalids).mean()
    if expl == "entropy":
        ent = O._masked_select(O.cat_entropy(logits), valids, num_invalids)
        el = -cfg.exploration_loss_coeff * ent.mean()
    else:   # learner.py:479-486
        skl = O._masked_select(O.cat_symmetric_kl_with_uniform_prior(logits), valids, num_invalids).mean()
        el = cfg.exploration_loss_coeff * torch.clamp(skl, max=30)
    kl_old = O._masked_select(O.cat_kl(logits, logits_old), valids, num_invalids)
    kl = cfg.kl_loss_coeff * kl_old.mean()
    vc = v_old + torch.clamp(values - v_old, -cfg.ppo_clip_value, cfg.ppo_clip_value)
    vl = O._masked_select(torch.max((values - targets) ** 2, (vc - targets) ** 2), valids, num_invalids).mean() * cfg.value_loss_coeff
    total = pl + el + kl + vl
    total.backward()

    stats = torch.zeros(ops.LS_SIZE, dtype=torch.float64, device=dev)
    ws = torch.empty(ops.loss_workspace_bytes(B) // 8 + 8, dtype=torch.float64, device=dev)
    dl = torch.empty(B, A, device=dev)
    dv = torch.empty(B, device=dev)
    ops.adv_stats(adv.to(dev), valids.to(dev), stats, None, ws)
    ops.ppo_loss_fwd_bwd(logits.detach().to(dev), values.detach().to(dev), actions.view(-1).to(dev), lp_old.to(dev),
                         v_old.to(dev), adv.to(dev), targets.to(dev), valids.to(dev), logits_old.to(dev),
                         cfg.ppo_clip_ratio, cfg.ppo_clip_value, cfg.exploration_loss_coeff, cfg.value_loss_coeff,
                         cfg.kl_loss_coeff, 1.0, dl, dv, stats, ws, exploration_loss=expl)
    s = stats.cpu()
    LS = ops.LS
    assert int(s[LS["num_valid"]]) == B - num_invalids
    for key, ref in [("adv_mean", adv_mean), ("adv_std", adv_std), ("policy_loss", pl), ("value_loss", vl),
                     ("exploration_loss", el), ("kl_loss", kl), ("kl_old_mean", kl_old.mean()),
                     ("kl_old_max", kl_old.max()), ("total_loss", total)]:
        assert abs(s[LS[key]].item() - float(ref)) < TOL, (key, s[LS[key]].item(), float(ref))
    vr = ratio.detach()[valids]
    assert abs(s[LS["ratio_min"]].item() - float(vr.min())) < TOL and abs(s[LS["ratio_max"]].item() - float(vr.max())) < TOL
    np.testing.assert_allclose(dl.cpu().numpy(), logits.grad.numpy(), atol=1e-7, rtol=2e-4)
    np.testing.assert_allclose(dv.cpu().numpy(), values.grad.numpy(), atol=1e-7, rtol=2e-4)
    # properties that hold at any size: softmax-gradient rows sum to zero, invalid rows get exactly zero gradient
    assert dl.sum(-1).abs().max().item() < 1e-6
    assert torch.all(dl.cpu()[~valids] == 0) and torch.all(dv.cpu()[~valids] == 0)


def test_action_ratio(dev):
    ops = _ops()
    B, A = 1000, 8
    logits = torch.randn(B, A, generator=g(48))
    actions = torch.randint(0, A, (B, 1), generator=g(49)).float()
    lp_old = torch.randn(B, generator=g(50)) - 2
    ref = torch.clamp(torch.exp(O.cat_log_prob(logits, actions) - lp_old), 0.05, 20.0)
    out = torch.empty(B, device=dev)
    ops.action_ratio(logits.to(dev), actions.view(-1).to(dev), lp_old.to(dev), out)
    np.testing.assert_allclose(out.cpu().numpy(), ref.numpy(), rtol=2e-6, atol=1e-6)


# ----------------------------------------------------------------------------------------------- optimizer
@pytest.mark.parametrize("n,max_norm", [(1000, 4.0), (300553, 4.0), (300553, 0.0), (4097, 1e-3)])
def test_clip_adam_step(dev, n, max_norm):
    ops = _ops()
    p = torch.randn(n, generator=g(51))
    m = torch.zeros(n)
    v = torch.zeros(n)
    pd, md, vd = p.to(dev), m.to(dev), v.to(dev)
    ws = torch.empty(1024, device=dev)
    gn = torch.zeros(1, device=dev)
    num = torch.tensor([900.0], dtype=torch.float64, device=dev)
    den = torch.tensor([1000.0], dtype=torch.float64, device=dev)
    lr, b1, b2, eps = 1e-3, 0.9, 0.999, 1e-6
    for step in range(1, 4):
        grad = torch.randn(n, generator=g(60 + step)) * (10.0 if step == 2 else 0.01)
        gref = grad.clone()
        total = torch.linalg.vector_norm(gref)
        if max_norm > 0:
            O.clip_grad_norm_([gref], max_norm)
        O.adam_step(p, gref, m, v, step, lr * 900.0 / 1000.0, b1, b2, eps)
        ops.clip_adam_step(pd, grad.to(dev), md, vd, step, lr, b1, b2, eps, max_norm, num, den, gn, ws)
        assert abs(gn.item() - total.item()) <= 1e-5 * max(1.0, total.item())
        np.testing.assert_allclose(pd.cpu().numpy(), p.numpy(), atol=1e-6, rtol=1e-5)
        np.testing.assert_allclose(md.cpu().numpy(), m.numpy(), atol=1e-7, rtol=1e-5)
        np.testing.assert_allclose(vd.cpu().numpy(), v.numpy(), atol=1e-9, rtol=1e-5)


# ----------------------------------------------------------------------------------------------- recurrent core
@pytest.mark.parametrize("rnn_type", ["gru", "lstm"])
@pytest.mark.parametrize("M,H,IN", [(64, 32, 48), (1024, 512, 512), (333, 96, 20)])
def test_rnn_cell_forward_backward(dev, rnn_type, M, H, IN):
    """One recurrent step (cell kernels + the two gate GEMMs) against the oracle's written-out nn.GRU / nn.LSTM cell
    (oracle.rnn_cell, pinned to the reference's PackedSequence path by the tiny_gru / tiny_lstm goldens) incl. autograd
    gradients, with a reset mask on the outgoing state and carried gradients from a fictitious next step."""
    ops = _ops()
    ocfg = O.OracleCfg(obs_dim=IN, num_actions=4, encoder_mlp_layers=[IN], use_rnn=True, rnn_type=rnn_type, rnn_size=H)
    st = O.init_state(ocfg, seed=2)
    G = 4 if rnn_type == "lstm" else 3
    S = O.rnn_state_size(ocfg)
    x = torch.randn(M, IN, generator=g(80)).requires_grad_(True)
    state = (torch.randn(M, S, generator=g(81)) * 0.5).requires_grad_(True)
    reset = torch.rand(M, generator=g(82)) < 0.3
    params = {k: st[k].clone().requires_grad_(True) for k in [O.RNN_W_IH, O.RNN_W_HH, O.RNN_B_IH, O.RNN_B_HH]}
    out, new_state = O.rnn_cell(ocfg, params, x, state)
    nxt = new_state * (1.0 - reset.float()).unsqueeze(-1)
    d_out = torch.randn(M, H, generator=g(83))
    d_next = torch.randn(M, S, generator=g(84))
    ((out * d_out).sum() + (nxt * d_next).sum()).backward()

    W_ih, W_hh, b_ih, b_hh = (st[k].to(dev) for k in [O.RNN_W_IH, O.RNN_W_HH, O.RNN_B_IH, O.RNN_B_HH])
    xd, sd = x.detach().to(dev), state.detach().to(dev)
    gi = torch.empty(M, G * H, device=dev)
    gh = torch.empty(M, G * H, device=dev)
    ops.linear_act_forward(xd, W_ih, b_ih, gi, ops.ACT["none"], ops.GEMM_SIMT)
    ops.linear_act_forward(sd[:, :H], W_hh, b_hh, gh, ops.ACT["none"], ops.GEMM_SIMT)
    s_out = torch.empty(M, S, device=dev)
    s_next = torch.empty(M, S, device=dev)
    gates = torch.empty(M, G * H, device=dev)
    rd = reset.to(dev)
    dgi = torch.empty(M, G * H, device=dev)
    dgh = torch.empty(M, G * H, device=dev)
    direct = torch.empty(M, H, device=dev)
    dnd = d_next.to(dev)
    if rnn_type == "lstm":
        ops.lstm_cell_forward(gi, gh, sd, s_out, s_next, rd, gates)
        # carries: gradient wrt next state's h part and c part (already "after the mask" in the oracle graph)
        ops.lstm_cell_backward(d_out.to(dev), dnd[:, :H].contiguous(), dnd[:, H:].contiguous(), rd, gates, sd, s_out, dgh, direct)
        dgi = dgh
    else:
        ops.gru_cell_forward(gi, gh, sd, s_out, s_next, rd, gates)
        ops.gru_cell_backward(d_out.to(dev), dnd, None, rd, gates, gh, sd, dgi, dgh, direct)
    np.testing.assert_allclose(s_out.cpu().numpy(), new_state.detach().numpy(), atol=TOL)
    np.testing.assert_allclose(s_next.cpu().numpy(), nxt.detach().numpy(), atol=TOL)
    # gradients: d x = dgi . W_ih ; d state_h = dgh . W_hh + direct ; d state_c (lstm) = direct
    dx = dgi.cpu().double() @ st[O.RNN_W_IH].double()
    dh = dgh.cpu().double() @ st[O.RNN_W_HH].double()
    np.testing.assert_allclose(dx.float().numpy(), x.grad.numpy(), atol=2e-5, rtol=1e-4)
    if rnn_type == "lstm":
        np.testing.assert_allclose(dh.float().numpy(), state.grad[:, :H].numpy(), atol=2e-5, rtol=1e-4)
        np.testing.assert_allclose(direct.cpu().numpy(), state.grad[:, H:].numpy(), atol=2e-5, rtol=1e-4)
    else:
        np.testing.assert_allclose((dh + direct.cpu().double()).float().numpy(), state.grad.numpy(), atol=2e-5, rtol=1e-4)
    np.testing.assert_allclose((dgi.cpu().double().t() @ x.detach().double()).float().numpy(), params[O.RNN_W_IH].grad.numpy(),
                               atol=2e-4, rtol=1e-4)
    np.testing.assert_allclose(dgh.cpu().double().sum(0).float().numpy(), params[O.RNN_B_HH].grad.numpy(), atol=2e-4, rtol=1e-4)
    # mask_rows + colsum helpers
    masked = torch.empty(M, S, device=dev)
    ops.mask_rows(s_out, masked, rd)
    assert torch.equal(masked, s_next)
    cs = torch.empty(G * H, device=dev)
    ops.colsum(dgh, cs, torch.empty(ops.colsum_workspace_bytes(G * H) // 4 + 4, device=dev))
    np.testing.assert_allclose(cs.cpu().numpy(), dgh.cpu().double().sum(0).float().numpy(), atol=1e-4, rtol=1e-4)


@pytest.mark.parametrize("engine_name", ["simt", "3xtf32"])
@pytest.mark.parametrize("rnn_type", ["gru", "lstm"])
@pytest.mark.parametrize("random_dones", [True, False])
@pytest.mark.parametrize("T,N,D", [(5, 1, 1), (5, 64, 10), (27, 1, 42), (27, 64, 10), (37, 64, 42)])
def test_bptt_matches_loopy_torch_rnn(dev, T, N, D, random_dones, rnn_type, engine_name):
    """The reference's own recurrent-core check (tests/algo/test_rnn.py:10-75: T in {5,27,37}, N in {1,64}, D in {1,10,42},
    dones every 7th step or random) against the device BPTT: a step-by-step torch nn.GRU / nn.LSTM loop that zeroes the
    state after a done is the ground truth for the forward outputs AND, through autograd, for every gradient."""
    ops = _ops()
    from sample_factory_b200.model import ModelSpec, PolicyModel
    from sample_factory_b200.rnn_core import RnnCore

    if engine_name != "simt" and not ops.tc_available():
        pytest.skip("tcgen05 engine not available")
    engine = ops.ENGINES[engine_name]
    gen = g(1000 + T * 131 + N * 7 + D)
    rnn = (torch.nn.GRU if rnn_type == "gru" else torch.nn.LSTM)(D, D, 1)
    B = N * T
    if random_dones:
        dones = torch.randint(0, 2, (B,), generator=gen).bool()
    else:
        dones = torch.zeros(B, dtype=torch.bool)
        dones[1::7] = True
    S = D if rnn_type == "gru" else 2 * D
    states = torch.rand(B, S, generator=gen)
    x = torch.randn(B, D, generator=gen, requires_grad=True)
    d_core = torch.randn(B, D, generator=gen)

    # loopy ground truth, env-major rows c*T + t (tests/algo/test_rnn.py:37-45)
    h = states[::T, :D].unsqueeze(0).contiguous()
    c = states[::T, D:].unsqueeze(0).contiguous() if rnn_type == "lstm" else None
    outs = []
    for t in range(T):
        if rnn_type == "gru":
            out, h = rnn(x[t::T].view(1, N, D), h)
        else:
            out, (h, c) = rnn(x[t::T].view(1, N, D), (h, c))
            c = c * (1 - dones[t::T].float().view(1, N, 1))
        outs.append(out.view(N, D))
        h = h * (1 - dones[t::T].float().view(1, N, 1))
    loopy = torch.stack(outs, dim=1).view(B, D)
    (loopy * d_core).sum().backward()

    spec = ModelSpec(D, 3, [D], [], "elu", False, False, use_rnn=True, rnn_type=rnn_type, rnn_size=D)
    model = PolicyModel(spec, dev)
    sd = {f"core.core.{k}": v.detach().clone() for k, v in rnn.state_dict().items()}
    model.load_state_dict(sd, strict=False)
    core = RnnCore(model, engine)
    b = core.alloc_bptt(B, T)
    valids = torch.ones(B, dtype=torch.bool, device=dev)
    got = core.forward_bptt(x.detach().to(dev), states.to(dev), dones.to(dev), valids, b)
    np.testing.assert_allclose(got.cpu().numpy(), loopy.detach().numpy(), atol=4e-6)      # the reference test's tolerance

    model.grad.zero_()
    lin_ws = torch.empty(core.lin_ws_bytes(B, T, D) // 4 + 4, device=dev)
    dgi = core.backward_bptt(d_core.to(dev), b, lin_ws).cpu().double()
    W_ih = rnn.weight_ih_l0.detach().double()
    np.testing.assert_allclose((dgi @ W_ih).float().numpy(), x.grad.numpy(), atol=2e-5, rtol=1e-4)
    np.testing.assert_allclose((dgi.t() @ x.detach().double()).float().numpy(), rnn.weight_ih_l0.grad.numpy(), atol=1e-4, rtol=1e-4)
    _, dW_hh, db_ih, db_hh = model.rnn_params(grads=True)
    np.testing.assert_allclose(dW_hh.cpu().numpy(), rnn.weight_hh_l0.grad.numpy(), atol=1e-4, rtol=1e-4)
    np.testing.assert_allclose(db_ih.cpu().numpy(), rnn.bias_ih_l0.grad.numpy(), atol=1e-4, rtol=1e-4)
    np.testing.assert_allclose(db_hh.cpu().numpy(), rnn.bias_hh_l0.grad.numpy(), atol=1e-4, rtol=1e-4)


def test_bad_arguments_raise(dev):
    """Error behaviour: argument violations surface as Python exceptions carrying the library message."""
    ops = _ops()
    from sample_factory_b200._lib import SfbError

    x = torch.zeros(4, 4, device=dev)
    with pytest.raises(SfbError):
        ops.heads_forward(x, x[0:1], x[0, :1], torch.zeros(40, 4, device=dev), torch.zeros(40, device=dev), x[:, 0], 4)
    with pytest.raises(RuntimeError):
        ops.normalize_obs(torch.zeros(4, 4), x, None, None)  # CPU tensor: there is no CPU path


# ----------------------------------------------------------------------------------------------- fused paths
@pytest.mark.parametrize("engine_name", ["3xtf32", "tf32"])
@pytest.mark.parametrize("M,K,N,A,act", [(4096, 512, 512, 8, "elu"), (1000, 64, 256, 5, "tanh"), (333, 96, 128, 1, "relu")])
def test_linear_heads_fused_matches_separate(dev, engine_name, M, K, N, A, act):
    """sfb200_linear_act_heads_forward + sfb200_heads_from_partials == sfb200_linear_act_forward + sfb200_heads_forward
    (same GEMM accumulators -> identical y; head dot products differ only in summation order) and == the oracle."""
    ops = _ops()
    engine = {"3xtf32": ops.GEMM_TC_3XTF32, "tf32": ops.GEMM_TC_TF32}[engine_name]
    P = ops.linear_heads_partials(N, A, engine)
    assert P == 2 * (N // 128), "fused path must cover these shapes on a B200"
    x = torch.randn(M, K, generator=g(60))
    W = torch.randn(N, K, generator=g(61)) / math.sqrt(K)
    b = torch.randn(N, generator=g(62)) * 0.1
    Wv = torch.randn(1, N, generator=g(63)) / math.sqrt(N)
    bv = torch.randn(1, generator=g(64))
    Wa = torch.randn(A, N, generator=g(65)) / math.sqrt(N)
    ba = torch.randn(A, generator=g(66)) * 0.1
    noise = torch.empty(M, A).exponential_(generator=g(67))
    xd, Wd, bd, Wvd, bvd, Wad, bad, nd = (t.to(dev).contiguous() for t in (x, W, b, Wv, bv, Wa, ba, noise))
    actc = ops.ACT[act]

    def outs():
        return dict(values=torch.empty(M, device=dev), logits=torch.empty(M, A, device=dev),
                    actions=torch.empty(M, device=dev), env_actions=torch.empty(M, dtype=torch.int32, device=dev),
                    lp=torch.empty(M, device=dev), pv=torch.empty(M, device=dev))

    pvs = torch.full((1,), 7.0, device=dev)

    def kw(o):
        return dict(values=o["values"], values_stride=1, logits=o["logits"], logits_stride=A, noise=nd,
                    actions_f32=o["actions"], actions_stride=1, env_actions=o["env_actions"], log_prob=o["lp"],
                    log_prob_stride=1, policy_version_scalar=pvs, policy_version_out=o["pv"], pv_stride=1)

    # separate
    y_ref = torch.empty(M, N, device=dev)
    o1 = outs()
    ops.linear_act_forward(xd, Wd, bd, y_ref, actc, engine)
    ops.heads_forward(y_ref, Wvd, bvd, Wad, bad, **kw(o1))
    # fused, storing y
    part = torch.full((P * M * ops.HEAD_PART_PAD,), float("nan"), device=dev)
    y = torch.full((M, N), float("nan"), device=dev)
    o2 = outs()
    ops.linear_act_heads_forward(xd, Wd, bd, y, actc, engine, Wvd, Wad, part)
    ops.heads_from_partials(part, P, M, bvd, bad, **kw(o2))
    assert torch.equal(y, y_ref)
    # fused, not storing y (sampler mode)
    part3 = torch.full_like(part, float("nan"))
    o3 = outs()
    ops.linear_act_heads_forward(xd, Wd, bd, None, actc, engine, Wvd, Wad, part3)
    ops.heads_from_partials(part3, P, M, bvd, bad, **kw(o3))
    for k in o2:
        assert torch.equal(o2[k], o3[k]), k
    # heads finished inside the GEMM kernel (last-arriving CTA of every 128-row block): identical to the two-launch path
    counters = torch.zeros((M + 127) // 128, dtype=torch.int32, device=dev)
    for rep in range(2):          # twice: the arrival counters must be left at zero
        part4 = torch.full_like(part, float("nan"))
        o4 = outs()
        y4 = torch.full((M, N), float("nan"), device=dev)
        ops.linear_act_heads_forward_fused(xd, Wd, bd, y4 if rep == 0 else None, actc, engine, Wvd, bvd, Wad, bad, part4,
                                           counters, **kw(o4))
        for k in o2:
            assert torch.equal(o2[k], o4[k]), (k, rep)
        assert rep == 1 or torch.equal(y4, y_ref)
        assert torch.all(counters == 0)
    assert (o2["values"] - o1["values"]).abs().max().item() < TOL
    assert (o2["logits"] - o1["logits"]).abs().max().item() < TOL
    assert (o2["lp"] - o1["lp"]).abs().max().item() < 2 * TOL
    assert torch.all(o2["pv"] == 7.0)
    same = (o2["actions"] == o1["actions"]).float().mean().item()
    assert same >= 0.999, same       # identical up to argmax near-ties moved by 1e-7-level logit differences
    assert torch.equal(o2["actions"].to(torch.int32), o2["env_actions"])
    if engine_name == "3xtf32":      # fp32-grade engine: against the oracle (fp32 CPU)
        h = {"elu": torch.nn.functional.elu, "tanh": torch.tanh, "relu": torch.relu}[act](x @ W.t() + b)
        v_ref = (h @ Wv.t() + bv).squeeze(1)
        l_ref = h @ Wa.t() + ba
        assert (o2["values"].cpu() - v_ref).abs().max().item() < 2 * TOL
        assert (o2["logits"].cpu() - l_ref).abs().max().item() < 2 * TOL
        a_ref = torch.argmax(torch.softmax(l_ref, -1) / noise, dim=-1).float()
        assert (o2["actions"].cpu() == a_ref).float().mean().item() >= 0.999


def test_sampler_post_pre_step_fused_matches_separate(dev):
    """sfb200_sampler_post_pre_step == sfb200_sampler_post_step(t) then sfb200_sampler_pre_step(t+1), bit for bit."""
    ops = _ops()
    N, D, T = 1000, 64, 4
    mean = torch.randn(D, generator=g(70), dtype=torch.float64).to(dev)
    var = (torch.rand(D, generator=g(71), dtype=torch.float64) + 0.1).to(dev)

    def state():
        return dict(traj_obs=torch.full((N, T + 1, D), -1.0, device=dev), traj_rnn=torch.full((N, T + 1, 1), -1.0, device=dev),
                    xn=torch.full((N, D), -2.0, device=dev), rew_t=torch.zeros(N, T, device=dev),
                    done_t=torch.zeros(N, T, dtype=torch.bool, device=dev), to_t=torch.zeros(N, T, dtype=torch.bool, device=dev),
                    pid_t=torch.full((N, T), -1, dtype=torch.int32, device=dev), ep_ret=torch.zeros(N, device=dev),
                    ep_len=torch.zeros(N, dtype=torch.int32, device=dev), ep_min=torch.full((N,), float("inf"), device=dev),
                    ep_max=torch.full((N,), float("-inf"), device=dev), stats=torch.zeros(8, dtype=torch.float64, device=dev),
                    counter=torch.zeros(1, dtype=torch.int64, device=dev),
                    fin_ret=torch.full((N, T), float("nan"), device=dev), fin_len=torch.full((N, T), -1, dtype=torch.int32, device=dev))

    s1, s2 = state(), state()
    rnn = torch.zeros(N, 1, device=dev)
    for t in range(T):
        obs = torch.randn(N, D, generator=g(80 + t)).to(dev)
        r = torch.randn(N, generator=g(90 + t)).to(dev)
        tm = (torch.rand(N, generator=g(100 + t)) < 0.1).to(dev)
        tr = (torch.rand(N, generator=g(110 + t)) < 0.1).to(dev)
        last = t + 1 == T

        def post_args(s):
            return (r, tm, tr, 0.7, 0.5, 3, s["rew_t"][:, t], s["done_t"][:, t], s["to_t"][:, t], s["pid_t"][:, t], s["ep_ret"],
                    s["ep_len"], s["ep_min"], s["ep_max"], 2, s["stats"], s["counter"], s["fin_ret"][:, t], s["fin_len"][:, t])

        ops.sampler_post_step(*post_args(s1))
        ops.sampler_pre_step(obs, s1["traj_obs"][:, t + 1], rnn, s1["traj_rnn"][:, t + 1], None if last else s1["xn"], mean, var,
                             0.25, 0.5)
        ops.sampler_post_pre_step(*post_args(s2), obs=obs, traj_obs_next=s2["traj_obs"][:, t + 1], rnn=rnn,
                                  traj_rnn_next=s2["traj_rnn"][:, t + 1], x_norm=None if last else s2["xn"], mean=mean,
                                  var=var, sub_mean=0.25, inv_scale=0.5)
        for k in s1:
            a, b = s1[k], s2[k]
            if k == "stats":      # fp64 atomics: warp order is not fixed
                assert torch.allclose(a, b, rtol=1e-12, atol=1e-12), (k, t)
            elif a.dtype.is_floating_point:
                assert torch.equal(torch.nan_to_num(a, nan=12345.0), torch.nan_to_num(b, nan=12345.0)), (k, t)
            else:
                assert torch.equal(a, b), (k, t)
    assert s2["counter"].item() == T and s2["stats"][0].item() > 0


def test_presplit_weight_lo_matches_inline_split(dev):
    """A GEMM whose weight operand lies in a buffer registered with sfb200_register_tf32_lo (lo tile loaded by TMA) is
    bit-identical to the same GEMM on an unregistered copy (lo derived in shared memory); Adam keeps lo current."""
    ops = _ops()
    M, K, N = 4096, 512, 512
    eng = ops.GEMM_TC_3XTF32
    flat = (torch.randn(N * K + N, generator=g(120)) / math.sqrt(K)).to(dev)
    lo = torch.empty_like(flat)
    ops.register_tf32_lo(flat, lo)
    try:
        W, b = flat[: N * K].view(N, K), flat[N * K:]
        W2, b2 = W.clone(), b.clone()
        x = torch.randn(M, K, generator=g(121)).to(dev)
        y1, y2 = torch.empty(M, N, device=dev), torch.empty(M, N, device=dev)
        ops.linear_act_forward(x, W, b, y1, ops.ACT["elu"], eng)
        ops.linear_act_forward(x, W2, b2, y2, ops.ACT["elu"], eng)
        assert torch.equal(y1, y2)
        ref = torch.nn.functional.elu(x.double() @ W.double().t() + b.double()).float()
        assert (y1 - ref).abs().max().item() < 2e-5
        dz = torch.randn(M, N, generator=g(122)).to(dev)
        ws = torch.empty(ops.linear_backward_workspace_bytes(M, N, K) // 4 + 4, device=dev)
        dW1, dW2 = torch.empty(N, K, device=dev), torch.empty(N, K, device=dev)
        dx1, dx2 = torch.empty(M, K, device=dev), torch.empty(M, K, device=dev)
        ops.linear_backward(dz, x, W, ops.ACT["elu"], dW1, dx1, None, eng, ws)
        ops.linear_backward(dz, x, W2, ops.ACT["elu"], dW2, dx2, None, eng, ws)
        assert torch.equal(dx1, dx2) and torch.equal(dW1, dW2)
        # Adam on the registered buffer refreshes lo in the same kernel
        grad = torch.randn_like(flat) * 0.01
        m, v = torch.zeros_like(flat), torch.zeros_like(flat)
        ops.clip_adam_step(flat, grad, m, v, 1, 1e-3, 0.9, 0.999, 1e-6, 4.0, None, None, None,
                           torch.empty(1024, device=dev))
        lo_adam = lo.clone()
        ops.refresh_tf32_lo(flat)
        assert torch.equal(lo_adam, lo)
        hi = (flat.view(torch.int32) & -8192).view(torch.float32)
        assert torch.equal(lo, ((flat - hi).view(torch.int32) & -8192).view(torch.float32))
    finally:
        ops.unregister_tf32_lo(flat)


# ----------------------------------------------------------------------------------------------- continuous actions
@pytest.mark.parametrize("adaptive,tanh_scale", [(True, 0.0), (False, 0.0), (False, 1.5)])
@pytest.mark.parametrize("rows,H,Ad", [(300, 64, 6), (4096, 512, 8), (37, 48, 1)])
def test_heads_forward_continuous(dev, rows, H, Ad, adaptive, tanh_scale):
    """sfb200_heads_forward_continuous vs the oracle's ContinuousActionDistribution restatement (pinned to the reference
    by the tiny_gauss goldens): distribution parameters, sampled actions, log-probs."""
    ops = _ops()
    ocfg = O.OracleCfg(obs_dim=H, num_actions=Ad, encoder_mlp_layers=[], continuous=True, adaptive_stddev=adaptive,
                       continuous_tanh_scale=tanh_scale)
    n_lin = O.num_linear_action_outputs(ocfg)
    h = torch.randn(rows, H, generator=g(130))
    st = {O.CRITIC_W: torch.randn(1, H, generator=g(131)) / math.sqrt(H), O.CRITIC_B: torch.randn(1, generator=g(132)),
          O.ACTION_W: torch.randn(n_lin, H, generator=g(133)) / math.sqrt(H), O.ACTION_B: torch.randn(n_lin, generator=g(134)) * 0.3,
          O.LEARNED_STD: torch.randn(Ad, generator=g(135)) * 0.5}
    eps = torch.randn(rows, Ad, generator=g(136))
    v_ref, params_ref = O.tail_forward(ocfg, st, h)
    a_ref = O.gauss_sample(params_ref, eps)
    lp_ref = O.gauss_log_prob(params_ref, a_ref)

    d = {k: v.to(dev).contiguous() for k, v in st.items()}
    values = torch.empty(rows, device=dev)
    params = torch.full((rows, 2 * Ad), float("nan"), device=dev)
    actions = torch.empty(rows, Ad, device=dev)
    env_actions = torch.empty(rows, Ad, device=dev)
    lp = torch.empty(rows, device=dev)
    pv = torch.empty(rows, device=dev)
    ops.heads_forward_continuous(h.to(dev), d[O.CRITIC_W], d[O.CRITIC_B], d[O.ACTION_W], d[O.ACTION_B], Ad, adaptive,
                                 None if adaptive else d[O.LEARNED_STD], tanh_scale, values, 1, params, 2 * Ad,
                                 eps.to(dev), 0, 0, None, actions, Ad, env_actions, lp, 1,
                                 torch.full((1,), 3.0, device=dev), pv, 1)
    assert (values.cpu() - v_ref).abs().max().item() < TOL
    assert (params.cpu() - params_ref).abs().max().item() < TOL
    if not adaptive:
        assert torch.equal(params.cpu()[:, Ad:], st[O.LEARNED_STD].repeat(rows, 1))
    # a = eps*std + mean: std = exp(log_std) carries the 1e-6 RELATIVE difference of log_std, so compare relatively
    np.testing.assert_allclose(actions.cpu().numpy(), a_ref.numpy(), atol=2e-5, rtol=5e-5)
    assert torch.equal(actions, env_actions) and torch.all(pv == 3.0)
    # log-prob of the device's own action under the device's own parameters, evaluated by the oracle formula
    lp_self = O.gauss_log_prob(params.cpu(), actions.cpu())
    assert (lp.cpu() - lp_self).abs().max().item() < 2e-5
    assert (lp.cpu() - lp_ref).abs().max().item() < 1e-3   # (a - mean)/std amplifies 1e-6 differences for small std
    # parameters-only mode (learner minibatch forward) and the Philox path (statistics only)
    params2 = torch.empty_like(params)
    ops.heads_forward_continuous(h.to(dev), d[O.CRITIC_W], d[O.CRITIC_B], d[O.ACTION_W], d[O.ACTION_B], Ad, adaptive,
                                 None if adaptive else d[O.LEARNED_STD], tanh_scale, values, 1, params2, 2 * Ad)
    assert torch.equal(params2, params)
    if rows >= 4096:
        ops.heads_forward_continuous(h.to(dev), d[O.CRITIC_W], d[O.CRITIC_B], d[O.ACTION_W], d[O.ACTION_B], Ad, adaptive,
                                     None if adaptive else d[O.LEARNED_STD], tanh_scale, values, 1, params2, 2 * Ad,
                                     None, 1234, 0, None, actions, Ad, env_actions, lp, 1)
        mu, _, sd = O.gauss_split(params.cpu())
        zs = (actions.cpu() - mu) / sd
        assert abs(zs.mean().item()) < 0.02 and abs(zs.std().item() - 1.0) < 0.02


@pytest.mark.parametrize("B,Ad,adaptive,tanh_scale,frac_invalid,kl_coeff",
                         [(64, 6, True, 0.0, 0.0, 0.0), (1000, 6, False, 1.5, 0.2, 0.1), (4096, 8, False, 0.0, 0.0, 0.1),
                          (777, 3, True, 0.0, 0.3, 0.5), (513, 12, False, 2.0, 0.1, 0.2)])
def test_ppo_loss_fwd_bwd_continuous(dev, B, Ad, adaptive, tanh_scale, frac_invalid, kl_coeff):
    """Gaussian PPO loss forward + backward vs autograd through the oracle's distribution formulas; the leaves are the
    distribution_linear outputs z (and the learned log-stddev vector when adaptive_stddev=False)."""
    ops = _ops()
    cfg = O.OracleCfg(num_actions=Ad, kl_loss_coeff=kl_coeff, ppo_clip_ratio=0.2, ppo_clip_value=0.2, continuous=True,
                      exploration_loss_coeff=0.003)
    n_lin = 2 * Ad if adaptive else Ad
    z = (torch.randn(B, n_lin, generator=g(140)) * 0.8).requires_grad_(True)
    learned = (torch.randn(Ad, generator=g(141)) * 0.4).requires_grad_(True)
    if adaptive:
        z.data[:, Ad:] *= 0.5
        z.data[0, Ad] = -12.0     # std clamp (1e-4) active: zero gradient through the clamp
        z.data[1, Ad] = 11.0      # std clamp (1e4) active

    def params_of(zz, ll):
        if adaptive:
            return zz
        means = torch.tanh(zz / tanh_scale) * tanh_scale if tanh_scale > 0 else zz
        return torch.cat((means, ll.repeat(B, 1)), dim=1)

    params = params_of(z, learned)
    values = torch.randn(B, generator=g(142)).requires_grad_(True)
    params_old = params.detach() + torch.randn(B, 2 * Ad, generator=g(143)) * 0.2
    actions = O.gauss_sample(params_old, torch.randn(B, Ad, generator=g(144)))
    lp_old = O.gauss_log_prob(params_old, actions) + torch.randn(B, generator=g(145)) * 0.05
    v_old = values.detach() + torch.randn(B, generator=g(146)) * 0.3
    adv = torch.randn(B, generator=g(147)) * 2 + 0.5
    targets = torch.randn(B, generator=g(148))
    valids = torch.rand(B, generator=g(149)) >= frac_invalid
    num_invalids = int((~valids).sum())

    clip_hi = 1.0 + cfg.ppo_clip_ratio
    clip_lo = 1.0 / clip_hi
    lp = O.gauss_log_prob(params, actions)
    ratio = torch.clamp(torch.exp(lp - lp_old), 0.05, 20.0)
    adv_std, adv_mean = torch.std_mean(O._masked_select(adv, valids, num_invalids))
    advn = (adv - adv_mean) / torch.clamp_min(adv_std, 1e-7)
    pl = -O._masked_select(torch.min(ratio * advn, torch.clamp(ratio, clip_lo, clip_hi) * advn), valids, num_invalids).mean()
    ent = O._masked_select(O.gauss_entropy(params), valids, num_invalids)
    el = -cfg.exploration_loss_coeff * ent.mean()
    kl_old = O._masked_select(O.gauss_kl(params, params_old), valids, num_invalids)
    kl = cfg.kl_loss_coeff * kl_old.mean()
    vc = v_old + torch.clamp(values - v_old, -cfg.ppo_clip_value, cfg.ppo_clip_value)
    vl = O._masked_select(torch.max((values - targets) ** 2, (vc - targets) ** 2), valids, num_invalids).mean() * cfg.value_loss_coeff
    total = pl + el + kl + vl
    total.backward()

    stats = torch.zeros(ops.LS_SIZE, dtype=torch.float64, device=dev)
    ws = torch.empty(ops.loss_workspace_bytes(B) // 8 + 8, dtype=torch.float64, device=dev)
    dl = torch.empty(B, n_lin, device=dev)
    dls = None if adaptive else torch.empty(B, Ad, device=dev)
    dv = torch.empty(B, device=dev)
    ops.adv_stats(adv.to(dev), valids.to(dev), stats, None, ws)
    ops.ppo_loss_fwd_bwd_continuous(params.detach().to(dev).contiguous(), values.detach().to(dev), adaptive, tanh_scale,
                                    actions.to(dev).contiguous(), lp_old.to(dev), v_old.to(dev), adv.to(dev), targets.to(dev),
                                    valids.to(dev), params_old.to(dev).contiguous(), cfg.ppo_clip_ratio, cfg.ppo_clip_value,
                                    cfg.exploration_loss_coeff, cfg.value_loss_coeff, cfg.kl_loss_coeff, 1.0, dl, dls, dv,
                                    stats, ws)
    s = stats.cpu()
    LS = ops.LS
    for key, ref in [("policy_loss", pl), ("value_loss", vl), ("exploration_loss", el), ("kl_loss", kl),
                     ("kl_old_mean", kl_old.mean()), ("kl_old_max", kl_old.max()), ("total_loss", total)]:
        assert abs(s[LS[key]].item() - float(ref)) < TOL + 1e-5 * abs(float(ref)), (key, s[LS[key]].item(), float(ref))
    np.testing.assert_allclose(dl.cpu().numpy(), z.grad.numpy(), atol=2e-7, rtol=5e-4)
    np.testing.assert_allclose(dv.cpu().numpy(), values.grad.numpy(), atol=1e-7, rtol=2e-4)
    if not adaptive:
        np.testing.assert_allclose(dls.cpu().sum(0).numpy(), learned.grad.numpy(), atol=1e-6, rtol=5e-4)
    else:
        assert dl[0, Ad].item() == 0.0 and dl[1, Ad].item() == 0.0    # clamped stddev passes no gradient
    assert torch.all(dl.cpu()[~valids] == 0) and torch.all(dv.cpu()[~valids] == 0)
    # V-trace pre-pass
    out = torch.empty(B, device=dev)
    ops.action_ratio_continuous(params.detach().to(dev).contiguous(), actions.to(dev).contiguous(), lp_old.to(dev), out)
    np.testing.assert_allclose(out.cpu().numpy(), ratio.detach().numpy(), rtol=2e-5, atol=1e-6)


# ----------------------------------------------------------------------------------------------- conv encoder
@pytest.mark.parametrize("engine_name", ["simt", "3xtf32"])
@pytest.mark.parametrize("B,shape,arch", [(5, (4, 44, 44), "convnet_atari"), (3, (4, 84, 84), "convnet_atari"),
                                          (4, (3, 36, 36), "convnet_simple"), (6, (1, 30, 30), "convnet_impala")])
def test_conv_head_forward_backward(dev, B, shape, arch, engine_name):
    """ConvHead (im2col + GEMM engine + col2im) vs torch.nn.functional.conv2d + autograd on the CPU (the arithmetic the
    reference's ConvEncoderImpl executes, model/encoder.py:88-118): features, conv weight / bias gradients."""
    ops = _ops()
    if engine_name != "simt" and not ops.tc_available():
        pytest.skip("tcgen05 engine not available")
    from sample_factory_b200.conv_encoder import ConvHead
    from sample_factory_b200.model import ModelSpec, PolicyModel

    ocfg = O.OracleCfg(obs_dim=int(np.prod(shape)), num_actions=4, obs_shape=shape, encoder_conv_architecture=arch,
                       encoder_conv_mlp_layers=[32], nonlinearity="relu")
    st = O.init_state(ocfg, seed=5)
    spec = ModelSpec(ocfg.obs_dim, 4, nonlinearity="relu", obs_shape=shape, encoder_conv_architecture=arch,
                     encoder_conv_mlp_layers=[32])
    model = PolicyModel(spec, dev)
    model.load_state_dict(st, strict=False)
    head = ConvHead(model, ops.ENGINES[engine_name], B + 2, need_backward=True)
    x = torch.randn(B, ocfg.obs_dim, generator=g(150))
    # CPU reference with autograd
    params = {k: st[k].clone().requires_grad_(True) for k in st if "conv_head" in k}
    hcpu = x.view(B, *shape)
    for i, (_co, _k, s_) in enumerate(O.CONV_ARCH[arch]):
        hcpu = torch.relu(torch.nn.functional.conv2d(hcpu, params[O.conv_w(i)], params[O.conv_b(i)], stride=s_))
    feat_ref = hcpu.reshape(B, -1)
    gfeat = torch.randn(feat_ref.shape, generator=g(151))
    feat_ref.backward(gfeat)

    feat = head.forward(x.to(dev))
    tol = 2e-5
    assert (feat.cpu() - feat_ref.detach()).abs().max().item() < tol
    # the backward takes the gradient w.r.t. the PRE-activation of the last conv layer
    dpre = (gfeat * (feat_ref.detach() > 0).float()).to(dev).contiguous()
    model.grad.zero_()
    head.backward(dpre)
    for i in range(len(O.CONV_ARCH[arch])):
        gW, gb = model.conv_params(grads=True)[i]
        ref_w, ref_b = params[O.conv_w(i)].grad, params[O.conv_b(i)].grad
        scale = max(1.0, ref_w.abs().max().item())
        assert (gW.cpu() - ref_w).abs().max().item() < 5e-5 * scale, i
        assert (gb.cpu() - ref_b).abs().max().item() < 5e-5 * max(1.0, ref_b.abs().max().item()), i


def test_normalize_obs_uint8(dev):
    """uint8 observation rows: .float() -> scale -> running-mean-std (utils/normalize.py:40-67), bit-exact"""
    ops = _ops()
    rows, dim = 77, 4 * 12 * 12
    x = torch.randint(0, 256, (rows, dim), generator=g(160), dtype=torch.uint8)
    mean = torch.rand(dim, generator=g(161), dtype=torch.float64)
    var = torch.rand(dim, generator=g(162), dtype=torch.float64) * 0.1 + 0.01
    ref = x.float().mul_(1.0 / 255.0)
    staged = torch.empty(rows, dim, device=dev)
    ops.normalize_obs(x.to(dev), staged, None, None, 0.0, 1.0 / 255.0)
    assert torch.equal(staged.cpu(), ref)
    # IEEE restatement of running_mean_std.py:96-110 in numpy float32 (every op correctly rounded).  torch's CPU sqrt is
    # NOT correctly rounded (vectorised approximation: ~1 % of inputs are 1 ulp off), so the torch oracle is matched to
    # 1 ulp while the numpy pipeline -- which is what torch computes on a CUDA device -- is matched bit for bit.
    f = np.float32
    sig = np.sqrt((var.numpy().astype(f) + f(1e-5)).astype(f))
    ieee = ((ref.numpy() - mean.numpy().astype(f)).astype(f) * (f(1) / sig).astype(f)).astype(f).clip(-5, 5)
    O.rms_normalize_(ref, mean, var)
    out = torch.empty(rows, dim, device=dev)
    ops.normalize_obs(x.to(dev), out, mean.to(dev), var.to(dev), 0.0, 1.0 / 255.0)
    assert np.array_equal(out.cpu().numpy(), ieee)
    np.testing.assert_allclose(out.cpu().numpy(), ref.numpy(), rtol=2.5e-7, atol=1e-7)
    ref = torch.from_numpy(ieee)
    # sampler pre-step: raw uint8 copy into the trajectory + normalised float row
    T = 3
    traj = torch.zeros((rows, T + 1, dim), dtype=torch.uint8, device=dev)
    traj_rnn = torch.zeros((rows, T + 1, 1), device=dev)
    xn = torch.empty(rows, dim, device=dev)
    ops.sampler_pre_step(x.to(dev), traj[:, 1], torch.zeros(rows, 1, device=dev), traj_rnn[:, 1], xn, mean.to(dev),
                         var.to(dev), 0.0, 1.0 / 255.0)
    assert torch.equal(traj[:, 1].cpu(), x) and torch.all(traj[:, 0] == 0) and torch.equal(xn.cpu(), ref)


def test_clip_lamb_step(dev):
    """sfb200_clip_lamb_step vs the oracle's restatement of algo/utils/optimizers.py (pinned by the tiny_lamb golden):
    three steps on a padded flat buffer with tensors of very different norms (trust ratio clamped at both ends)."""
    ops = _ops()
    shapes = [(64, 16), (64,), (5, 64), (5,), (1, 64), (1,)]
    numels = [int(np.prod(sh)) for sh in shapes]
    offs, off = [], 0
    for n in numels:
        offs.append(off)
        off += (n + 63) // 64 * 64
    total = off
    scales = [1.0, 1e-4, 30.0, 0.0, 0.5, 2.0]     # |p| = 0 -> trust 1 ; |p| large -> min(|p|, 10) ; tiny |p| -> min_trust
    ps = [torch.randn(n, generator=g(170 + i)) * sc for i, (n, sc) in enumerate(zip(numels, scales))]
    ms = [torch.zeros(n) for n in numels]
    vs = [torch.zeros(n) for n in numels]
    flat = torch.zeros(total)
    for p_, o, n in zip(ps, offs, numels):
        flat[o: o + n] = p_
    pd = flat.to(dev)
    md, vd = torch.zeros(total, device=dev), torch.zeros(total, device=dev)
    seg_off = torch.tensor(offs, dtype=torch.int64, device=dev)
    seg_n = torch.tensor(numels, dtype=torch.int64, device=dev)
    ws = torch.empty(ops.lamb_workspace_bytes(len(shapes), max(numels)) // 4 + 4, device=dev)
    gn = torch.zeros(1, device=dev)
    lr, b1, b2, eps, max_norm = 3e-3, 0.9, 0.999, 1e-6, 0.7
    for step in range(1, 4):
        gs = [torch.randn(n, generator=g(180 + 10 * step + i)) * 0.3 for i, n in enumerate(numels)]
        gflat = torch.zeros(total)
        for g_, o, n in zip(gs, offs, numels):
            gflat[o: o + n] = g_
        gd = gflat.to(dev)
        ops.clip_lamb_step(pd, gd, md, vd, seg_off, seg_n, max(numels), step, lr, b1, b2, eps, 1e-4, 0.01, max_norm, None,
                           None, gn, ws)
        gl = [x.clone() for x in gs]
        total_norm = O.clip_grad_norm_(gl, max_norm)
        assert abs(gn.item() - float(total_norm)) < 1e-5 * max(1.0, float(total_norm))
        for p_, g_, m_, v_ in zip(ps, gl, ms, vs):
            O.lamb_step(p_, g_, m_, v_, step, lr, b1, b2, eps)
        got = pd.cpu()
        for p_, o, n in zip(ps, offs, numels):
            np.testing.assert_allclose(got[o: o + n].numpy(), p_.numpy(), atol=2e-6, rtol=2e-5)
    # padding between the tensors is never touched
    mask = torch.ones(total, dtype=torch.bool)
    for o, n in zip(offs, numels):
        mask[o: o + n] = False
    assert torch.all(pd.cpu()[mask] == 0) and torch.all(md.cpu()[mask] == 0)


# ----------------------------------------------------------------------------------------------- tuple action spaces
@pytest.mark.parametrize("expl", ["entropy", "symmetric_kl"])
@pytest.mark.parametrize("B,segs,frac_invalid,kl_coeff", [(64, [3, 2, 4], 0.0, 0.0), (1000, [8], 0.2, 0.1),
                                                          (4096, [3, 3, 3, 3, 3, 3, 3, 3], 0.1, 0.3), (513, [17, 2, 5], 0.3, 0.2)])
def test_ppo_loss_fwd_bwd_tuple(dev, B, segs, frac_invalid, kl_coeff, expl):
    """Tuple-of-Discretes PPO loss forward + backward vs autograd through the oracle's TupleActionDistribution formulas"""
    ops = _ops()
    A = sum(segs)
    cfg = O.OracleCfg(num_actions=A, action_segments=list(segs), kl_loss_coeff=kl_coeff, ppo_clip_ratio=0.1,
                      ppo_clip_value=0.2, exploration_loss=expl, exploration_loss_coeff=0.003 if expl == "entropy" else 0.02)
    logits = (torch.randn(B, A, generator=g(190)) * 1.5).requires_grad_(True)
    values = torch.randn(B, generator=g(191)).requires_grad_(True)
    logits_old = logits.detach() + torch.randn(B, A, generator=g(192)) * 0.3
    noise = torch.empty(B, A).exponential_(generator=g(193))
    actions = O.tuple_sample(cfg, logits_old, noise).float()
    lp_old = O.tuple_log_prob(cfg, logits_old, actions) + torch.randn(B, generator=g(194)) * 0.05
    v_old = values.detach() + torch.randn(B, generator=g(195)) * 0.3
    adv = torch.randn(B, generator=g(196)) * 2 + 0.5
    targets = torch.randn(B, generator=g(197))
    valids = torch.rand(B, generator=g(198)) >= frac_invalid
    num_invalids = int((~valids).sum())

    clip_hi = 1.0 + cfg.ppo_clip_ratio
    clip_lo = 1.0 / clip_hi
    lp = O.dist_log_prob(cfg, logits, actions)
    ratio = torch.clamp(torch.exp(lp - lp_old), 0.05, 20.0)
    adv_std, adv_mean = torch.std_mean(O._masked_select(adv, valids, num_invalids))
    advn = (adv - adv_mean) / torch.clamp_min(adv_std, 1e-7)
    pl = -O._masked_select(torch.min(ratio * advn, torch.clamp(ratio, clip_lo, clip_hi) * advn), valids, num_invalids).mean()
    if expl == "entropy":
        el = -cfg.exploration_loss_coeff * O._masked_select(O.dist_entropy(cfg, logits), valids, num_invalids).mean()
    else:
        el = cfg.exploration_loss_coeff * torch.clamp(
            O._masked_select(O.dist_symmetric_kl(cfg, logits), valids, num_invalids).mean(), max=30)
    kl_old = O._masked_select(O.dist_kl(cfg, logits, logits_old), valids, num_invalids)
    kl = cfg.kl_loss_coeff * kl_old.mean()
    vc = v_old + torch.clamp(values - v_old, -cfg.ppo_clip_value, cfg.ppo_clip_value)
    vl = O._masked_select(torch.max((values - targets) ** 2, (vc - targets) ** 2), valids, num_invalids).mean() * cfg.value_loss_coeff
    total = pl + el + kl + vl
    total.backward()

    stats = torch.zeros(ops.LS_SIZE, dtype=torch.float64, device=dev)
    ws = torch.empty(ops.loss_workspace_bytes(B) // 8 + 8, dtype=torch.float64, device=dev)
    dl = torch.empty(B, A, device=dev)
    dv = torch.empty(B, device=dev)
    ops.adv_stats(adv.to(dev), valids.to(dev), stats, None, ws)
    ops.ppo_loss_fwd_bwd_tuple(logits.detach().to(dev), values.detach().to(dev), segs, actions.to(dev).contiguous(),
                               lp_old.to(dev), v_old.to(dev), adv.to(dev), targets.to(dev), valids.to(dev),
                               logits_old.to(dev), cfg.ppo_clip_ratio, cfg.ppo_clip_value, cfg.exploration_loss_coeff,
                               cfg.value_loss_coeff, cfg.kl_loss_coeff, 1.0, dl, dv, stats, ws, exploration_loss=expl)
    s = stats.cpu()
    LS = ops.LS
    for key, ref in [("policy_loss", pl), ("value_loss", vl), ("exploration_loss", el), ("kl_loss", kl),
                     ("kl_old_mean", kl_old.mean()), ("total_loss", total)]:
        assert abs(s[LS[key]].item() - float(ref)) < TOL, (key, s[LS[key]].item(), float(ref))
    np.testing.assert_allclose(dl.cpu().numpy(), logits.grad.numpy(), atol=1e-7, rtol=3e-4)
    np.testing.assert_allclose(dv.cpu().numpy(), values.grad.numpy(), atol=1e-7, rtol=2e-4)
    assert torch.all(dl.cpu()[~valids] == 0)
    out = torch.empty(B, device=dev)
    ops.action_ratio_tuple(logits.detach().to(dev), segs, actions.to(dev).contiguous(), lp_old.to(dev), out)
    np.testing.assert_allclose(out.cpu().numpy(), ratio.detach().numpy(), rtol=3e-6, atol=1e-6)


def test_heads_forward_tuple(dev):
    """Tuple heads: per-head sampling / log-prob sums vs the oracle, both the dot-product kernel and the from-partials one"""
    ops = _ops()
    rows, H, segs = 777, 96, [3, 2, 4]
    A = sum(segs)
    cfg = O.OracleCfg(num_actions=A, action_segments=segs)
    h = torch.randn(rows, H, generator=g(200))
    Wv = torch.randn(1, H, generator=g(201)) / math.sqrt(H)
    bv = torch.randn(1, generator=g(202))
    Wa = torch.randn(A, H, generator=g(203)) / math.sqrt(H) * 2
    ba = torch.randn(A, generator=g(204)) * 0.1
    noise = torch.empty(rows, A).exponential_(generator=g(205))
    logits_ref = torch.nn.functional.linear(h, Wa, ba)
    a_ref = O.tuple_sample(cfg, logits_ref, noise)
    lp_ref = O.tuple_log_prob(cfg, logits_ref, a_ref.float())
    values = torch.empty(rows, device=dev)
    logits = torch.empty(rows, A, device=dev)
    actions = torch.empty(rows, len(segs), device=dev)
    env_actions = torch.empty(rows, len(segs), dtype=torch.int32, device=dev)
    lp = torch.empty(rows, device=dev)
    ops.heads_forward_tuple(h.to(dev), Wv.to(dev), bv.to(dev), Wa.to(dev), ba.to(dev), segs, values, 1, logits, A,
                            noise.to(dev), 0, 0, None, actions, len(segs), env_actions, lp, 1)
    assert (logits.cpu() - logits_ref).abs().max().item() < TOL
    assert torch.equal(actions.cpu().long(), a_ref) and torch.equal(env_actions.cpu().long(), a_ref)
    assert (lp.cpu() - lp_ref).abs().max().item() < 2 * TOL
