"""Tensor-level wrappers over the C ABI (include/sfb200.h).

PyTorch is used here only as the owner of device memory and streams: every function takes CUDA tensors, checks
dtype / contiguity, and passes raw pointers + the current CUDA stream handle to libsfb200.  Nothing in this module
computes anything itself and there is no CPU path -- a CPU tensor raises.
"""
from __future__ import annotations

from typing import Optional

import torch
from torch import Tensor

from ._lib import lib

ACT = {"none": 0, "elu": 1, "relu": 2, "tanh": 3}
GEMM_SIMT, GEMM_TC_3XTF32, GEMM_TC_TF32 = 0, 1, 2
ENGINES = {"simt": GEMM_SIMT, "3xtf32": GEMM_TC_3XTF32, "tf32": GEMM_TC_TF32}

LS = dict(
    num_valid=0, adv_mean=1, adv_std=2, policy_loss=3, value_loss=4, exploration_loss=5, kl_loss=6, kl_old_mean=7,
    kl_old_max=8, entropy_mean=9, ratio_mean_abs_dev=10, ratio_min=11, ratio_max=12, fraction_clipped=13,
    value_mean=14, total_loss=15,
)
LS_SIZE = 16

_device_bound = {}


def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


def bind_device(device: torch.device) -> None:
    """cudaSetDevice for libsfb200's (statically linked) CUDA runtime on this thread."""
    idx = device.index if device.index is not None else torch.cuda.current_device()
    lib().call("sfb200_set_device", idx)


def _p(t: Optional[Tensor], dtype=None) -> Optional[int]:
    if t is None:
        return None
    if not t.is_cuda:
        raise RuntimeError("sample_factory_b200 ops need CUDA tensors (there is no CPU path)")
    if dtype is not None and t.dtype != dtype:
        raise TypeError(f"expected {dtype}, got {t.dtype}")
    if t.dim() > 0 and t.stride(-1) != 1 and t.shape[-1] != 1:
        raise ValueError("last dimension must be dense")
    return t.data_ptr()


F32, F64, U8, I32, I64 = torch.float32, torch.float64, torch.bool, torch.int32, torch.int64
BYTE = torch.uint8   # image observations


def _obs_entry(name: str, obs: Tensor):
    """(entry point, dtype) for an observation tensor: uint8 rows go to the *_u8 twin of the entry point"""
    if obs.dtype == BYTE:
        return name + "_u8", BYTE
    return name, F32


def sm_count() -> int:
    return lib().query("sfb200_sm_count")


def launch_count() -> int:
    """Kernels launched by libsfb200 in this process so far (counted inside the library)."""
    return lib().query("sfb200_launch_count")


def tc_available() -> bool:
    return bool(lib().query("sfb200_tc_available"))


# ------------------------------------------------------------------------------------------------ normalizers
def normalize_obs(x: Tensor, out: Tensor, mean: Optional[Tensor], var: Optional[Tensor], sub_mean: float = 0.0,
                  inv_scale: float = 1.0, eps: float = 1e-5, clip: float = 5.0) -> Tensor:
    """x, out: [rows, dim] (row strides free). utils/normalize.py:51-70."""
    rows, dim = x.shape
    entry, dt = _obs_entry("sfb200_normalize_obs", x)
    lib().call(entry, _p(x, dt), x.stride(0), _p(out, F32), out.stride(0), rows, dim,
               _p(mean, F64), _p(var, F64), sub_mean, inv_scale, eps, clip, _stream())
    return out


def moments_workspace_bytes(dim: int) -> int:
    return lib().query("sfb200_moments_workspace_bytes", dim)


def batch_moments(x: Tensor, batch_mean: Tensor, batch_var: Tensor, workspace: Tensor) -> None:
    rows, dim = x.shape
    assert workspace.numel() * workspace.element_size() >= moments_workspace_bytes(dim)
    lib().call("sfb200_batch_moments", _p(x, F32), x.stride(0), rows, dim, _p(batch_mean, F32), _p(batch_var, F32),
               workspace.data_ptr(), _stream())


def rms_merge(mean: Tensor, var: Tensor, count: Tensor, batch_mean: Tensor, batch_var: Tensor, batch_count: float):
    lib().call("sfb200_rms_merge", _p(mean, F64), _p(var, F64), _p(count, F64), _p(batch_mean, F32),
               _p(batch_var, F32), float(batch_count), mean.numel(), _stream())


def rms_apply_scalar(x: Tensor, mean: Tensor, var: Tensor, denormalize: bool, eps: float = 1e-5, clip: float = 5.0):
    assert x.is_contiguous()
    lib().call("sfb200_rms_apply_scalar", _p(x, F32), x.numel(), _p(mean, F64), _p(var, F64), eps, clip,
               int(denormalize), _stream())


# ------------------------------------------------------------------------------------------------ model forward
def linear_act_forward(x: Tensor, W: Tensor, b: Optional[Tensor], out: Tensor, act: int, engine: int) -> Tensor:
    M, K = x.shape
    N = W.shape[0]
    assert W.shape[1] == K and W.is_contiguous() and out.shape == (M, N)
    lib().call("sfb200_linear_act_forward", _p(x, F32), x.stride(0), _p(W, F32), _p(b, F32), _p(out, F32),
               out.stride(0), M, N, K, act, engine, _stream())
    return out


def heads_forward(h: Tensor, Wv: Tensor, bv: Tensor, Wa: Tensor, ba: Tensor, values: Tensor, values_stride: int,
                  logits: Optional[Tensor] = None, logits_stride: int = 0, noise: Optional[Tensor] = None,
                  philox_seed: int = 0, philox_offset: int = 0, philox_offset_dev: Optional[Tensor] = None,
                  actions_f32: Optional[Tensor] = None,
                  actions_stride: int = 0, env_actions: Optional[Tensor] = None, log_prob: Optional[Tensor] = None,
                  log_prob_stride: int = 0, policy_version_scalar: Optional[Tensor] = None,
                  policy_version_out: Optional[Tensor] = None, pv_stride: int = 0) -> None:
    """Outputs are raw views (pointer = first element, explicit element strides) so they can be trajectory slots."""
    rows, H = h.shape
    A = Wa.shape[0]
    assert Wa.is_contiguous() and Wv.is_contiguous() and (noise is None or noise.is_contiguous())
    lib().call("sfb200_heads_forward", _p(h, F32), h.stride(0), rows, H, A, _p(Wv, F32), _p(bv, F32), _p(Wa, F32),
               _p(ba, F32), values.data_ptr(), values_stride, None if logits is None else logits.data_ptr(),
               logits_stride, _p(noise, F32), philox_seed, philox_offset, _p(philox_offset_dev, I64),
               None if actions_f32 is None else actions_f32.data_ptr(), actions_stride, _p(env_actions, I32),
               None if log_prob is None else log_prob.data_ptr(), log_prob_stride, _p(policy_version_scalar, F32),
               None if policy_version_out is None else policy_version_out.data_ptr(), pv_stride, _stream())


def set_sampling_mode(action_mask: Optional[Tensor] = None, deterministic: bool = False) -> None:
    """action_mask: bool / uint8 [rows, A] on the device (0 = action not allowed) or None; see sfb200_set_sampling_mode"""
    if action_mask is not None:
        assert action_mask.dtype in (torch.bool, torch.uint8) and action_mask.dim() == 2 and action_mask.stride(1) == 1
        lib().call("sfb200_set_sampling_mode", action_mask.data_ptr(), action_mask.stride(0), int(deterministic))
    else:
        lib().call("sfb200_set_sampling_mode", None, 0, int(deterministic))


def _seg_array(head_sizes):
    import ctypes

    return (ctypes.c_int32 * len(head_sizes))(*[int(n) for n in head_sizes])


def _cat_tail_args(values, values_stride, logits, logits_stride, noise, philox_seed, philox_offset, philox_offset_dev,
                   actions_f32, actions_stride, env_actions, log_prob, log_prob_stride, policy_version_scalar,
                   policy_version_out, pv_stride):
    assert noise is None or noise.is_contiguous()
    return (values.data_ptr(), values_stride, None if logits is None else logits.data_ptr(), logits_stride,
            _p(noise, F32), philox_seed, philox_offset, _p(philox_offset_dev, I64),
            None if actions_f32 is None else actions_f32.data_ptr(), actions_stride, _p(env_actions, I32),
            None if log_prob is None else log_prob.data_ptr(), log_prob_stride, _p(policy_version_scalar, F32),
            None if policy_version_out is None else policy_version_out.data_ptr(), pv_stride, _stream())


def heads_forward_tuple(h: Tensor, Wv: Tensor, bv: Tensor, Wa: Tensor, ba: Tensor, head_sizes, values: Tensor,
                        values_stride: int, logits: Optional[Tensor] = None, logits_stride: int = 0,
                        noise: Optional[Tensor] = None, philox_seed: int = 0, philox_offset: int = 0,
                        philox_offset_dev: Optional[Tensor] = None, actions_f32: Optional[Tensor] = None,
                        actions_stride: int = 0, env_actions: Optional[Tensor] = None,
                        log_prob: Optional[Tensor] = None, log_prob_stride: int = 0,
                        policy_version_scalar: Optional[Tensor] = None, policy_version_out: Optional[Tensor] = None,
                        pv_stride: int = 0) -> None:
    """Tuple(Discrete(n_0), ...) action space: `actions_f32` rows hold one index per head, env_actions int32 [rows, K]"""
    rows, H = h.shape
    A = Wa.shape[0]
    assert Wa.is_contiguous() and Wv.is_contiguous() and sum(head_sizes) == A
    lib().call("sfb200_heads_forward_tuple", _p(h, F32), h.stride(0), rows, H, A, len(head_sizes), _seg_array(head_sizes),
               _p(Wv, F32), _p(bv, F32), _p(Wa, F32), _p(ba, F32),
               *_cat_tail_args(values, values_stride, logits, logits_stride, noise, philox_seed, philox_offset,
                               philox_offset_dev, actions_f32, actions_stride, env_actions, log_prob, log_prob_stride,
                               policy_version_scalar, policy_version_out, pv_stride))


def heads_from_partials_tuple(head_partials: Tensor, P: int, rows: int, bv: Tensor, ba: Tensor, head_sizes,
                              values: Tensor, values_stride: int, logits: Optional[Tensor] = None,
                              logits_stride: int = 0, noise: Optional[Tensor] = None, philox_seed: int = 0,
                              philox_offset: int = 0, philox_offset_dev: Optional[Tensor] = None,
                              actions_f32: Optional[Tensor] = None, actions_stride: int = 0,
                              env_actions: Optional[Tensor] = None, log_prob: Optional[Tensor] = None,
                              log_prob_stride: int = 0, policy_version_scalar: Optional[Tensor] = None,
                              policy_version_out: Optional[Tensor] = None, pv_stride: int = 0) -> None:
    A = ba.shape[0]
    lib().call("sfb200_heads_from_partials_tuple", _p(head_partials, F32), P, rows, A, len(head_sizes),
               _seg_array(head_sizes), _p(bv, F32), _p(ba, F32),
               *_cat_tail_args(values, values_stride, logits, logits_stride, noise, philox_seed, philox_offset,
                               philox_offset_dev, actions_f32, actions_stride, env_actions, log_prob, log_prob_stride,
                               policy_version_scalar, policy_version_out, pv_stride))


def _cont_tail_args(values, values_stride, params, params_stride, noise, philox_seed, philox_offset, philox_offset_dev,
                    actions_f32, actions_stride, env_actions, log_prob, log_prob_stride, policy_version_scalar,
                    policy_version_out, pv_stride):
    assert noise is None or noise.is_contiguous()
    assert env_actions is None or (env_actions.dtype == F32 and env_actions.is_contiguous())
    return (values.data_ptr(), values_stride, None if params is None else params.data_ptr(), params_stride,
            _p(noise, F32), philox_seed, philox_offset, _p(philox_offset_dev, I64),
            None if actions_f32 is None else actions_f32.data_ptr(), actions_stride, _p(env_actions, F32),
            None if log_prob is None else log_prob.data_ptr(), log_prob_stride, _p(policy_version_scalar, F32),
            None if policy_version_out is None else policy_version_out.data_ptr(), pv_stride, _stream())


def heads_forward_continuous(h: Tensor, Wv: Tensor, bv: Tensor, Wa: Tensor, ba: Tensor, act_dim: int,
                             adaptive_stddev: bool, learned_log_std: Optional[Tensor], tanh_scale: float, values: Tensor,
                             values_stride: int, logits: Optional[Tensor] = None, logits_stride: int = 0,
                             noise: Optional[Tensor] = None, philox_seed: int = 0, philox_offset: int = 0,
                             philox_offset_dev: Optional[Tensor] = None, actions_f32: Optional[Tensor] = None,
                             actions_stride: int = 0, env_actions: Optional[Tensor] = None,
                             log_prob: Optional[Tensor] = None, log_prob_stride: int = 0,
                             policy_version_scalar: Optional[Tensor] = None, policy_version_out: Optional[Tensor] = None,
                             pv_stride: int = 0) -> None:
    """Box action space: `logits` receives the distribution parameters [means | log_std] (2*act_dim per row), actions
    are float vectors; `env_actions` is a dense float32 [rows, act_dim] copy for the env."""
    rows, H = h.shape
    assert Wa.shape[0] == (2 * act_dim if adaptive_stddev else act_dim) and Wa.is_contiguous() and Wv.is_contiguous()
    lib().call("sfb200_heads_forward_continuous", _p(h, F32), h.stride(0), rows, H, act_dim, int(adaptive_stddev),
               _p(Wv, F32), _p(bv, F32), _p(Wa, F32), _p(ba, F32), _p(learned_log_std, F32), float(tanh_scale),
               *_cont_tail_args(values, values_stride, logits, logits_stride, noise, philox_seed, philox_offset,
                                philox_offset_dev, actions_f32, actions_stride, env_actions, log_prob, log_prob_stride,
                                policy_version_scalar, policy_version_out, pv_stride))


def heads_from_partials_continuous(head_partials: Tensor, P: int, rows: int, bv: Tensor, ba: Tensor, act_dim: int,
                                   adaptive_stddev: bool, learned_log_std: Optional[Tensor], tanh_scale: float,
                                   values: Tensor, values_stride: int, logits: Optional[Tensor] = None,
                                   logits_stride: int = 0, noise: Optional[Tensor] = None, philox_seed: int = 0,
                                   philox_offset: int = 0, philox_offset_dev: Optional[Tensor] = None,
                                   actions_f32: Optional[Tensor] = None, actions_stride: int = 0,
                                   env_actions: Optional[Tensor] = None, log_prob: Optional[Tensor] = None,
                                   log_prob_stride: int = 0, policy_version_scalar: Optional[Tensor] = None,
                                   policy_version_out: Optional[Tensor] = None, pv_stride: int = 0) -> None:
    lib().call("sfb200_heads_from_partials_continuous", _p(head_partials, F32), P, rows, act_dim, int(adaptive_stddev),
               _p(bv, F32), _p(ba, F32), _p(learned_log_std, F32), float(tanh_scale),
               *_cont_tail_args(values, values_stride, logits, logits_stride, noise, philox_seed, philox_offset,
                                philox_offset_dev, actions_f32, actions_stride, env_actions, log_prob, log_prob_stride,
                                policy_version_scalar, policy_version_out, pv_stride))


# ------------------------------------------------------------------------------------------------ conv encoder
def im2col(x: Tensor, in_nchw: bool, B: int, C: int, H: int, W: int, kernel: int, stride: int, col: Tensor) -> None:
    """x: [B, C*H*W] rows in (C,H,W) order (in_nchw) or [B*H*W, C] NHWC rows; col: [B*OH*OW, C*kernel*kernel]"""
    assert x.is_contiguous() and col.is_contiguous()
    lib().call("sfb200_im2col", _p(x, F32), int(in_nchw), B, C, H, W, kernel, stride, _p(col, F32), _stream())


def col2im_act_backward(dcol: Tensor, x_act: Tensor, B: int, C: int, H: int, W: int, kernel: int, stride: int, act: int,
                        dx: Tensor) -> None:
    """dx [B*H*W, C] (NHWC) = col2im(dcol) * act'(x_act)"""
    assert dcol.is_contiguous() and x_act.is_contiguous() and dx.is_contiguous()
    lib().call("sfb200_col2im_act_backward", _p(dcol, F32), _p(x_act, F32), B, C, H, W, kernel, stride, act, _p(dx, F32),
               _stream())


def permute_bpc(src: Tensor, dst: Tensor, B: int, P: int, C: int, to_channel_major: bool) -> None:
    """[B, P, C] -> [B, C, P] (to_channel_major) or back"""
    assert src.is_contiguous() and dst.is_contiguous()
    lib().call("sfb200_permute_bpc", _p(src, F32), _p(dst, F32), B, P, C, int(to_channel_major), _stream())


def register_tf32_lo(base: Tensor, lo: Tensor) -> None:
    """Pair a flat weight buffer with its tf32 low-half twin (see include/sfb200.h) and fill the twin."""
    assert base.is_contiguous() and lo.is_contiguous() and base.numel() == lo.numel()
    lib().call("sfb200_register_tf32_lo", _p(base, F32), _p(lo, F32), base.numel())
    refresh_tf32_lo(base)


def unregister_tf32_lo(base: Tensor) -> None:
    lib().call("sfb200_unregister_tf32_lo", _p(base, F32))


def refresh_tf32_lo(base: Tensor) -> None:
    """Recompute the registered low halves after the weights were written by anything but clip_adam_step."""
    lib().call("sfb200_refresh_tf32_lo", _p(base, F32), _stream())


def register_f16_twins(base: Tensor, twins: Tensor) -> None:
    """Pair a flat weight buffer with its fp16 (hi, lo) twins [hi16[n] | lo16[n]] (include/sfb200.h) and fill them."""
    assert base.is_contiguous() and twins.is_contiguous() and twins.dtype == torch.float16 and twins.numel() == 2 * base.numel()
    lib().call("sfb200_register_f16_twins", _p(base, F32), twins.data_ptr(), base.numel())
    refresh_f16_twins(base)


def unregister_f16_twins(base: Tensor) -> None:
    lib().call("sfb200_unregister_f16_twins", _p(base, F32))


def refresh_f16_twins(base: Tensor) -> None:
    lib().call("sfb200_refresh_f16_twins", _p(base, F32), _stream())


def register_f16_transposed(W: Tensor, twinsT: Tensor) -> None:
    """Transposed fp16 twins [hiT[K][N] | loT[K][N]] of one weight matrix W[N][K] (the weight operand of dX = dz . W)."""
    N, K = W.shape
    assert W.is_contiguous() and twinsT.dtype == torch.float16 and twinsT.numel() == 2 * N * K
    lib().call("sfb200_register_f16_transposed", _p(W, F32), N, K, twinsT.data_ptr())
    refresh_f16_transposed(W)


def unregister_f16_transposed(W: Tensor) -> None:
    lib().call("sfb200_unregister_f16_transposed", _p(W, F32))


def refresh_f16_transposed(W: Tensor) -> None:
    lib().call("sfb200_refresh_f16_transposed", _p(W, F32), _stream())


def register_operand_bound(buf: Tensor, bound: Tensor) -> None:
    """`bound` (one device float) is an upper bound of |x| over `buf`: GEMMs reading an activation operand inside `buf`
    may use the fp16-split engine."""
    assert bound.dtype == torch.float32 and bound.numel() == 1 and bound.is_cuda
    lib().call("sfb200_register_operand_bound", buf.data_ptr(), buf.numel() * buf.element_size(), _p(bound, F32))


def unregister_operand_bound(buf: Tensor) -> None:
    lib().call("sfb200_unregister_operand_bound", buf.data_ptr())


def _drop_bounds(ptrs) -> None:
    try:
        for p in ptrs:
            lib().call("sfb200_unregister_operand_bound", p)
    except Exception:
        pass


def register_operand_bounds(owner, pairs) -> None:
    """register (buffer, bound) pairs for as long as `owner` lives: the registry is keyed by device address, so entries must
    not outlive the buffers (the allocator hands the address to somebody else)"""
    import weakref

    for buf, bound in pairs:
        register_operand_bound(buf, bound)
    weakref.finalize(owner, _drop_bounds, [buf.data_ptr() for buf, _ in pairs])


def linear_out_bound(W: Tensor, b: Optional[Tensor], in_bound: Tensor, out_bound: Tensor, act: int) -> None:
    """out_bound[0] = max_n (in_bound * sum_k |W[n][k]| + |b[n]|): an upper bound of |act(x W^T + b)| for |x| <= in_bound;
    out_bound = four floats [bound, scratch, counter, -], the middle two zero before and after"""
    N, K = W.shape
    assert out_bound.numel() >= 4
    lib().call("sfb200_linear_out_bound", _p(W, F32), _p(b, F32), N, K, _p(in_bound, F32), _p(out_bound, F32), act, _stream())


def heads_dz_bound(dlogits: Tensor, dvalues: Tensor, Wv: Tensor, Wa: Tensor, out_bound: Tensor) -> None:
    """out_bound = max_m (|dvalues[m]| + sum_a |dlogits[m][a]|) * max(|Wv|, |Wa|): bound of heads_backward's dz output"""
    rows, A = dlogits.shape
    H = Wv.numel()
    assert Wa.numel() == A * H and dlogits.is_contiguous() and Wa.is_contiguous() and out_bound.numel() >= 3
    lib().call("sfb200_heads_dz_bound", _p(dlogits, F32), _p(dvalues, F32), rows, A, _p(Wv, F32), _p(Wa, F32), H,
               _p(out_bound, F32), _stream())


def linear_heads_partials(N: int, A: int, engine: int) -> int:
    """Partials per row the fused last-layer + heads forward produces (0: not covered -> use the separate calls)."""
    return int(lib().query("sfb200_linear_heads_partials", N, A, engine))


HEAD_PART_PAD = 12   # floats per (partial, row) in the scratch buffer of the fused last-layer + heads forward


def linear_act_heads_forward(x: Tensor, W: Tensor, b: Tensor, out: Optional[Tensor], act: int, engine: int,
                             Wv: Tensor, Wa: Tensor, head_partials: Tensor) -> None:
    """out = act(x W^T + b) (not stored when out is None) and head_partials[p, m, :A+1] = partial out . [Wv ; Wa]."""
    M, K = x.shape
    N = W.shape[0]
    A = Wa.shape[0]
    assert W.shape[1] == K and W.is_contiguous() and Wa.is_contiguous() and Wv.is_contiguous()
    assert out is None or out.shape == (M, N)
    P = linear_heads_partials(N, A, engine)
    assert P > 0 and head_partials.numel() >= P * M * HEAD_PART_PAD and head_partials.is_contiguous()
    lib().call("sfb200_linear_act_heads_forward", _p(x, F32), x.stride(0), _p(W, F32), _p(b, F32), _p(out, F32),
               0 if out is None else out.stride(0), M, N, K, act, engine, _p(Wv, F32), _p(Wa, F32), A,
               _p(head_partials, F32), _stream())


def linear_act_heads_forward_fused(x: Tensor, W: Tensor, b: Tensor, out: Optional[Tensor], act: int, engine: int,
                                   Wv: Tensor, bv: Tensor, Wa: Tensor, ba: Tensor, head_partials: Tensor,
                                   finish_counters: Tensor, values: Tensor, values_stride: int,
                                   logits: Optional[Tensor] = None, logits_stride: int = 0,
                                   noise: Optional[Tensor] = None, philox_seed: int = 0, philox_offset: int = 0,
                                   philox_offset_dev: Optional[Tensor] = None, actions_f32: Optional[Tensor] = None,
                                   actions_stride: int = 0, env_actions: Optional[Tensor] = None,
                                   log_prob: Optional[Tensor] = None, log_prob_stride: int = 0,
                                   policy_version_scalar: Optional[Tensor] = None,
                                   policy_version_out: Optional[Tensor] = None, pv_stride: int = 0, *,
                                   head_sizes=None, act_dim: int = 0, adaptive_stddev: bool = True,
                                   learned_log_std: Optional[Tensor] = None, tanh_scale: float = 0.0,
                                   continuous: bool = False) -> None:
    """Last hidden layer + heads + distribution tail: linear_act_heads_forward, then the matching
    heads_from_partials{,_tuple,_continuous}.  This once was one launch that finished the heads inside the GEMM; that
    kernel measured slower (profiles/r01_l_heads_finish_in_gemm.md) and was removed.  `finish_counters` is no longer
    used (left untouched).  The function keeps its name and signature because existing callers look it up by name
    (bench.py times it alongside linear_act_heads_forward)."""
    linear_act_heads_forward(x, W, b, out, act, engine, Wv, Wa, head_partials)
    P = linear_heads_partials(W.shape[0], Wa.shape[0], engine)
    kw = dict(logits=logits, logits_stride=logits_stride, noise=noise, philox_seed=philox_seed, philox_offset=philox_offset,
              philox_offset_dev=philox_offset_dev, actions_f32=actions_f32, actions_stride=actions_stride,
              env_actions=env_actions, log_prob=log_prob, log_prob_stride=log_prob_stride,
              policy_version_scalar=policy_version_scalar, policy_version_out=policy_version_out, pv_stride=pv_stride)
    M = x.shape[0]
    if continuous:
        heads_from_partials_continuous(head_partials, P, M, bv, ba, act_dim=act_dim, adaptive_stddev=adaptive_stddev,
                                       learned_log_std=learned_log_std, tanh_scale=tanh_scale, values=values,
                                       values_stride=values_stride, **kw)
    elif head_sizes:
        heads_from_partials_tuple(head_partials, P, M, bv, ba, head_sizes, values=values, values_stride=values_stride, **kw)
    else:
        heads_from_partials(head_partials, P, M, bv, ba, values=values, values_stride=values_stride, **kw)


def heads_from_partials(head_partials: Tensor, P: int, rows: int, bv: Tensor, ba: Tensor, values: Tensor,
                        values_stride: int, logits: Optional[Tensor] = None, logits_stride: int = 0,
                        noise: Optional[Tensor] = None, philox_seed: int = 0, philox_offset: int = 0,
                        philox_offset_dev: Optional[Tensor] = None, actions_f32: Optional[Tensor] = None,
                        actions_stride: int = 0, env_actions: Optional[Tensor] = None,
                        log_prob: Optional[Tensor] = None, log_prob_stride: int = 0,
                        policy_version_scalar: Optional[Tensor] = None, policy_version_out: Optional[Tensor] = None,
                        pv_stride: int = 0) -> None:
    """Second half of the fused path: same outputs / sampling semantics as heads_forward."""
    A = ba.shape[0]
    assert noise is None or noise.is_contiguous()
    lib().call("sfb200_heads_from_partials", _p(head_partials, F32), P, rows, A, _p(bv, F32), _p(ba, F32),
               values.data_ptr(), values_stride, None if logits is None else logits.data_ptr(), logits_stride,
               _p(noise, F32), philox_seed, philox_offset, _p(philox_offset_dev, I64),
               None if actions_f32 is None else actions_f32.data_ptr(), actions_stride, _p(env_actions, I32),
               None if log_prob is None else log_prob.data_ptr(), log_prob_stride, _p(policy_version_scalar, F32),
               None if policy_version_out is None else policy_version_out.data_ptr(), pv_stride, _stream())


# ------------------------------------------------------------------------------------------------ sampler
def sampler_pre_step(obs: Tensor, traj_obs_t: Tensor, rnn: Optional[Tensor], traj_rnn_t: Optional[Tensor],
                     x_norm: Optional[Tensor], mean: Optional[Tensor], var: Optional[Tensor], sub_mean: float,
                     inv_scale: float, eps: float = 1e-5, clip: float = 5.0) -> None:
    """obs [N, D] dense; traj_obs_t = traj['obs'][:, t] view ([N, D], row stride (T+1)*D)."""
    n, dim = obs.shape
    assert obs.is_contiguous() and (x_norm is None or x_norm.is_contiguous())
    rnn_dim = 0 if rnn is None else rnn.shape[1]
    entry, dt = _obs_entry("sfb200_sampler_pre_step", obs)
    assert traj_obs_t.dtype == obs.dtype
    lib().call(entry, _p(obs, dt), n, dim, traj_obs_t.data_ptr(), traj_obs_t.stride(0),
               _p(rnn, F32), rnn_dim, None if traj_rnn_t is None else traj_rnn_t.data_ptr(),
               0 if traj_rnn_t is None else traj_rnn_t.stride(0), _p(x_norm, F32), _p(mean, F64), _p(var, F64),
               sub_mean, inv_scale, eps, clip, _stream())


def sampler_post_step(rew: Tensor, terminated: Tensor, truncated: Tensor, reward_scale: float, reward_clip: float,
                      policy_id: int, traj_rewards_t: Tensor, traj_dones_t: Tensor, traj_time_outs_t: Tensor,
                      traj_policy_id_t: Tensor, ep_return: Optional[Tensor], ep_len: Optional[Tensor],
                      ep_min_raw: Optional[Tensor], ep_max_raw: Optional[Tensor], len_increment: int,
                      stats: Optional[Tensor], step_counter: Optional[Tensor] = None,
                      fin_return_t: Optional[Tensor] = None, fin_len_t: Optional[Tensor] = None) -> None:
    n = rew.numel()
    stride = traj_rewards_t.stride(0)
    assert fin_return_t is None or (fin_return_t.stride(0) == stride and fin_len_t.stride(0) == stride)
    assert traj_dones_t.stride(0) == stride and traj_time_outs_t.stride(0) == stride
    assert traj_policy_id_t.stride(0) == stride
    lib().call("sfb200_sampler_post_step", _p(rew, F32), _p(terminated, U8), _p(truncated, U8), n, reward_scale,
               reward_clip, policy_id, traj_rewards_t.data_ptr(), traj_dones_t.data_ptr(),
               traj_time_outs_t.data_ptr(), traj_policy_id_t.data_ptr(), stride, _p(ep_return, F32), _p(ep_len, I32),
               _p(ep_min_raw, F32), _p(ep_max_raw, F32), len_increment, _p(stats, F64), _p(step_counter, I64),
               None if fin_return_t is None else fin_return_t.data_ptr(),
               None if fin_len_t is None else fin_len_t.data_ptr(), _stream())



def sampler_post_pre_step(rew: Tensor, terminated: Tensor, truncated: Tensor, reward_scale: float, reward_clip: float,
                          policy_id: int, traj_rewards_t: Tensor, traj_dones_t: Tensor, traj_time_outs_t: Tensor,
                          traj_policy_id_t: Tensor, ep_return: Optional[Tensor], ep_len: Optional[Tensor],
                          ep_min_raw: Optional[Tensor], ep_max_raw: Optional[Tensor], len_increment: int,
                          stats: Optional[Tensor], step_counter: Optional[Tensor] = None,
                          fin_return_t: Optional[Tensor] = None, fin_len_t: Optional[Tensor] = None, *,
                          obs: Tensor, traj_obs_next: Tensor, rnn: Optional[Tensor], traj_rnn_next: Optional[Tensor],
                          x_norm: Optional[Tensor], mean: Optional[Tensor], var: Optional[Tensor], sub_mean: float,
                          inv_scale: float, eps: float = 1e-5, clip: float = 5.0) -> None:
    """sampler_post_step(t) + sampler_pre_step(t+1) in one launch (x_norm None: record the observation only)."""
    n = rew.numel()
    stride = traj_rewards_t.stride(0)
    assert fin_return_t is None or (fin_return_t.stride(0) == stride and fin_len_t.stride(0) == stride)
    assert traj_dones_t.stride(0) == stride and traj_time_outs_t.stride(0) == stride
    assert traj_policy_id_t.stride(0) == stride
    n_obs, dim = obs.shape
    assert n_obs == n and obs.is_contiguous() and (x_norm is None or x_norm.is_contiguous())
    rnn_dim = 0 if rnn is None else rnn.shape[1]
    entry, dt = _obs_entry("sfb200_sampler_post_pre_step", obs)
    assert traj_obs_next.dtype == obs.dtype
    lib().call(entry, _p(rew, F32), _p(terminated, U8), _p(truncated, U8), n, reward_scale,
               reward_clip, policy_id, traj_rewards_t.data_ptr(), traj_dones_t.data_ptr(),
               traj_time_outs_t.data_ptr(), traj_policy_id_t.data_ptr(), stride, _p(ep_return, F32), _p(ep_len, I32),
               _p(ep_min_raw, F32), _p(ep_max_raw, F32), len_increment, _p(stats, F64), _p(step_counter, I64),
               None if fin_return_t is None else fin_return_t.data_ptr(),
               None if fin_len_t is None else fin_len_t.data_ptr(),
               _p(obs, dt), dim, traj_obs_next.data_ptr(), traj_obs_next.stride(0), _p(rnn, F32), rnn_dim,
               None if traj_rnn_next is None else traj_rnn_next.data_ptr(),
               0 if traj_rnn_next is None else traj_rnn_next.stride(0), _p(x_norm, F32), _p(mean, F64), _p(var, F64),
               sub_mean, inv_scale, eps, clip, _stream())


def sampler_tail_tape_step(head_partials: Tensor, P: int, rows: int, bv: Tensor, ba: Tensor, *, values: Tensor,
                           values_stride: int, logits: Tensor, logits_stride: int, noise: Optional[Tensor], philox_seed: int,
                           sampler_step: Tensor, actions_f32: Tensor, actions_stride: int, env_actions: Tensor,
                           log_prob: Tensor, log_prob_stride: int, policy_version_scalar: Tensor, policy_version_out: Tensor,
                           pv_stride: int, env, reward_scale: float, reward_clip: float, policy_id: int, traj_rewards: Tensor,
                           traj_dones: Tensor, traj_time_outs: Tensor, traj_policy_id: Tensor, ep_return: Tensor,
                           ep_len: Tensor, ep_min_raw: Tensor, ep_max_raw: Tensor, len_increment: int, stats: Tensor,
                           fin_return: Optional[Tensor], fin_len: Optional[Tensor], traj_obs_next: Tensor, rnn: Tensor,
                           traj_rnn_next: Tensor, x_norm: Optional[Tensor], mean: Optional[Tensor], var: Optional[Tensor],
                           sub_mean: float, inv_scale: float, eps: float = 1e-5, clip: float = 5.0) -> None:
    """heads finish + sampling, the tape env's step, post-step(t) and pre-step(t+1) in ONE launch (csrc/heads.cu,
    sampler_tail_tape_kernel).  `env` is a sample_factory_b200.envs.TapeVecEnv (float32 obs, Discrete actions)."""
    A = ba.numel()
    # (the trajectory slots [:, t] are strided columns: element strides are passed explicitly)
    for t_ in (values, logits, actions_f32, log_prob, policy_version_out, traj_rewards, traj_dones, traj_time_outs, traj_policy_id):
        assert t_.is_cuda
    assert traj_dones.stride(0) == traj_rewards.stride(0) == traj_time_outs.stride(0) == traj_policy_id.stride(0)
    assert values.dtype == F32 and logits.dtype == F32 and traj_rewards.dtype == F32 and traj_policy_id.dtype == I32
    lib().call("sfb200_sampler_tail_tape_step", _p(head_partials, F32), P, rows, A, _p(bv, F32), _p(ba, F32),
               values.data_ptr(), values_stride, logits.data_ptr(), logits_stride, _p(noise, F32), philox_seed,
               _p(sampler_step, I64), actions_f32.data_ptr(), actions_stride, _p(env_actions, I32), log_prob.data_ptr(),
               log_prob_stride, _p(policy_version_scalar, F32), policy_version_out.data_ptr(), pv_stride,
               _p(env.tape, F32), env.tape_len, env.obs_dim, env.env_index_offset, env.term_period, env.trunc_period,
               _p(env.step_counter, I64), _p(env.obs, F32), _p(env.rew, F32), _p(env.terminated, U8), _p(env.truncated, U8),
               reward_scale, reward_clip, policy_id, traj_rewards.data_ptr(), traj_dones.data_ptr(), traj_time_outs.data_ptr(),
               traj_policy_id.data_ptr(), traj_rewards.stride(0), _p(ep_return, F32), _p(ep_len, I32), _p(ep_min_raw, F32),
               _p(ep_max_raw, F32), len_increment, _p(stats, F64), None if fin_return is None else fin_return.data_ptr(),
               None if fin_len is None else fin_len.data_ptr(),
               _p(traj_obs_next, F32), traj_obs_next.stride(0), _p(rnn, F32), rnn.shape[1], _p(traj_rnn_next, F32),
               traj_rnn_next.stride(0), _p(x_norm, F32), _p(mean, F64), _p(var, F64), sub_mean, inv_scale, eps, clip, _stream())


def rollout_mlp2_partials(W1: Tensor, W2: Tensor, A: int, engine: int) -> int:
    """head partials per row of the persistent whole-rollout kernel, 0 when the model is not covered"""
    H1, K1 = W1.shape
    H2 = W2.shape[0]
    if W2.shape[1] != H1 or not (W1.is_contiguous() and W2.is_contiguous()):
        return 0
    return lib().query("sfb200_rollout_mlp2_partials", _p(W1, F32), _p(W2, F32), K1, H1, H2, A, engine)


def rollout_mlp2_tape(T: int, W1: Tensor, b1: Tensor, W2: Tensor, b2: Tensor, act: int, engine: int, Wv: Tensor, bv: Tensor,
                      Wa: Tensor, ba: Tensor, h1_scratch: Tensor, head_partials: Tensor, x_norm: Tensor, traj, env,
                      noise: Optional[Tensor], philox_seed: int, sampler_step: Tensor, env_actions: Tensor,
                      policy_version_scalar: Tensor, reward_scale: float, reward_clip: float, policy_id: int,
                      ep_return: Tensor, ep_len: Tensor, ep_min_raw: Tensor, ep_max_raw: Tensor, len_increment: int,
                      stats: Tensor, fin_return: Optional[Tensor], fin_len: Optional[Tensor], rnn: Tensor,
                      mean: Optional[Tensor], var: Optional[Tensor], sub_mean: float, inv_scale: float, eps: float = 1e-5,
                      clip: float = 5.0) -> None:
    """One launch = a whole rollout (csrc/rollout_fused.cu).  `traj` is the trajectory dict ([N, T(+1), ...] tensors), `env` a
    sample_factory_b200.envs.TapeVecEnv; x_norm must hold the normalised observations of step 0 (sampler_pre_step)."""
    N, K1 = x_norm.shape
    H1, H2, A = W1.shape[0], W2.shape[0], ba.numel()
    tr = traj
    assert tr["rewards"].shape == (N, T) and tr["obs"].shape[1] == T + 1 and h1_scratch.shape[0] >= N and h1_scratch.shape[1] == H1
    assert all(tr[k].is_contiguous() for k in ("values", "action_logits", "actions", "log_prob_actions", "policy_version",
                                              "rewards", "dones", "time_outs", "policy_id", "obs", "rnn_states"))
    lib().call("sfb200_rollout_mlp2_tape", N, T, K1, _p(W1, F32), _p(b1, F32), H1, _p(W2, F32), _p(b2, F32), H2, act, engine,
               _p(Wv, F32), _p(bv, F32), _p(Wa, F32), _p(ba, F32), A, _p(h1_scratch, F32), _p(head_partials, F32), _p(x_norm, F32),
               tr["values"].data_ptr(), tr["values"].stride(0), tr["action_logits"].data_ptr(), tr["action_logits"].stride(0),
               _p(noise, F32), philox_seed, _p(sampler_step, I64), tr["actions"].data_ptr(), tr["actions"].stride(0),
               _p(env_actions, I32), tr["log_prob_actions"].data_ptr(), tr["log_prob_actions"].stride(0),
               _p(policy_version_scalar, F32), tr["policy_version"].data_ptr(), tr["policy_version"].stride(0),
               _p(env.tape, F32), env.tape_len, env.env_index_offset, env.term_period, env.trunc_period,
               _p(env.step_counter, I64), _p(env.obs, F32), _p(env.rew, F32), _p(env.terminated, U8), _p(env.truncated, U8),
               reward_scale, reward_clip, policy_id, tr["rewards"].data_ptr(), tr["dones"].data_ptr(), tr["time_outs"].data_ptr(),
               tr["policy_id"].data_ptr(), tr["rewards"].stride(0), _p(ep_return, F32), _p(ep_len, I32), _p(ep_min_raw, F32),
               _p(ep_max_raw, F32), len_increment, _p(stats, F64), None if fin_return is None else fin_return.data_ptr(),
               None if fin_len is None else fin_len.data_ptr(), tr["obs"].data_ptr(), tr["obs"].stride(0), _p(rnn, F32),
               rnn.shape[1], tr["rnn_states"].data_ptr(), tr["rnn_states"].stride(0), _p(mean, F64), _p(var, F64), sub_mean,
               inv_scale, eps, clip, _stream())


def gather_rows(src: Tensor, idx: Tensor, dst: Tensor) -> None:
    """dst[r] = src[idx[r]] along dim 0 (dense rows of any dtype) -- the shuffled-minibatch gather"""
    assert src.is_contiguous() and dst.is_contiguous() and src.dtype == dst.dtype and src.shape[1:] == dst.shape[1:]
    assert idx.dtype == torch.int32 and idx.is_contiguous() and idx.numel() == dst.shape[0]
    row_bytes = src.element_size() * (src.numel() // max(src.shape[0], 1))
    lib().call("sfb200_gather_rows", src.data_ptr(), row_bytes, _p(idx, I32), dst.shape[0], dst.data_ptr(), _stream())


def copy_rows_bytes(src: Tensor, dst: Tensor) -> None:
    """dst[r, :] = src[r, :] for 2-D tensors of any (equal) dtype with dense rows and free row strides"""
    assert src.dim() == 2 and dst.dim() == 2 and src.shape == dst.shape and src.dtype == dst.dtype
    assert src.is_cuda and dst.is_cuda and (src.shape[1] == 1 or (src.stride(1) == 1 and dst.stride(1) == 1))
    es = src.element_size()
    lib().call("sfb200_copy_rows_bytes", src.data_ptr(), src.stride(0) * es, dst.data_ptr(), dst.stride(0) * es, src.shape[0],
               src.shape[1] * es, _stream())


def copy_rows(src: Tensor, dst: Tensor) -> None:
    rows, dim = src.shape
    lib().call("sfb200_copy_rows", _p(src, F32), src.stride(0), dst.data_ptr(), dst.stride(0), rows, dim, _stream())


def tape_env_step(actions: Tensor, num_actions: int, env_index_offset: int, term_period: int, trunc_period: int,
                  step_counter: Optional[Tensor], step_host: int, tape: Optional[Tensor], obs_out: Optional[Tensor],
                  rew: Tensor, terminated: Tensor, truncated: Tensor) -> None:
    n = actions.numel()
    tape_len, dim = (tape.shape[0], tape.shape[2]) if tape is not None else (0, 0)
    lib().call("sfb200_tape_env_step", _p(actions, I32), n, num_actions, env_index_offset, term_period, trunc_period,
               _p(step_counter, I64), step_host, _p(tape, F32), tape_len, dim, _p(obs_out, F32), _p(rew, F32),
               _p(terminated, U8), _p(truncated, U8), _stream())


def tape_env_step_continuous(actions_f32: Tensor, env_index_offset: int, term_period: int, trunc_period: int,
                             step_counter: Optional[Tensor], step_host: int, tape: Optional[Tensor],
                             obs_out: Optional[Tensor], rew: Tensor, terminated: Tensor, truncated: Tensor) -> None:
    n, act_dim = actions_f32.shape
    assert actions_f32.is_contiguous()
    tape_len, dim = (tape.shape[0], tape.shape[2]) if tape is not None else (0, 0)
    lib().call("sfb200_tape_env_step_continuous", _p(actions_f32, F32), act_dim, n, env_index_offset, term_period,
               trunc_period, _p(step_counter, I64), step_host, _p(tape, F32), tape_len, dim, _p(obs_out, F32),
               _p(rew, F32), _p(terminated, U8), _p(truncated, U8), _stream())


# ------------------------------------------------------------------------------------------------ learner: prep
def compute_valids(policy_id: Tensor, policy_version: Tensor, this_policy: int, train_step: int, max_policy_lag: int,
                   valids: Tensor) -> None:
    n_traj, T = policy_id.shape
    assert policy_id.is_contiguous() and policy_version.is_contiguous() and valids.is_contiguous()
    assert valids.shape == (n_traj, T + 1)
    lib().call("sfb200_compute_valids", _p(policy_id, I32), _p(policy_version, F32), n_traj, T, this_policy,
               float(train_step), float(max_policy_lag), _p(valids, U8), _stream())


def gae_returns(rewards: Tensor, dones: Tensor, time_outs: Tensor, values: Tensor, valids: Tensor, gamma: float,
                lam: float, value_bootstrap: bool, ret_mean: Optional[Tensor], ret_var: Optional[Tensor], adv: Tensor,
                returns: Tensor, eps: float = 1e-5, clip: float = 5.0) -> None:
    n_traj, T = rewards.shape
    for t in (rewards, dones, time_outs, values, valids, adv, returns):
        assert t.is_contiguous()
    assert values.shape == (n_traj, T + 1) and valids.shape == (n_traj, T + 1)
    lib().call("sfb200_gae_returns", _p(rewards, F32), _p(dones, U8), _p(time_outs, U8), _p(values, F32),
               _p(valids, U8), n_traj, T, gamma, lam, int(value_bootstrap), _p(ret_mean, F64), _p(ret_var, F64), eps,
               clip, _p(adv, F32), _p(returns, F32), _stream())


def vtrace(ratio: Tensor, values: Tensor, rewards: Tensor, dones: Tensor, R: int, gamma: float, rho_hat: float,
           c_hat: float, vs: Tensor, adv: Tensor) -> None:
    n = ratio.numel() // R
    for t in (ratio, values, rewards, dones, vs, adv):
        assert t.is_contiguous()
    lib().call("sfb200_vtrace", _p(ratio, F32), _p(values, F32), _p(rewards, F32), _p(dones, U8), n, R, gamma, rho_hat,
               c_hat, _p(vs, F32), _p(adv, F32), _stream())


# ------------------------------------------------------------------------------------------------ learner: loss
def loss_workspace_bytes(batch: int) -> int:
    return lib().query("sfb200_loss_workspace_bytes", batch)


def action_ratio(logits: Tensor, actions_f32: Tensor, log_prob_old: Tensor, ratio: Tensor) -> None:
    B, A = logits.shape
    assert logits.is_contiguous()
    lib().call("sfb200_action_ratio", _p(logits, F32), A, _p(actions_f32, F32), _p(log_prob_old, F32), B,
               _p(ratio, F32), _stream())


def adv_stats(adv: Tensor, valids: Tensor, stats: Tensor, dp_partials: Optional[Tensor], workspace: Tensor) -> None:
    lib().call("sfb200_adv_stats", _p(adv, F32), _p(valids, U8), adv.numel(), _p(stats, F64), _p(dp_partials, F64),
               workspace.data_ptr(), _stream())


def adv_stats_finalize(dp_partials: Tensor, stats: Tensor) -> None:
    lib().call("sfb200_adv_stats_finalize", _p(dp_partials, F64), _p(stats, F64), _stream())


def ppo_loss_fwd_bwd(logits: Tensor, values: Tensor, actions_f32: Tensor, log_prob_old: Tensor, values_old: Tensor,
                     adv: Tensor, targets: Tensor, valids: Tensor, logits_old: Optional[Tensor], clip_ratio: float,
                     clip_value: float, exploration_coeff: float, value_coeff: float, kl_coeff: float,
                     grad_scale: float, dlogits: Tensor, dvalues: Tensor, stats: Tensor, workspace: Tensor,
                     exploration_loss: str = "entropy") -> None:
    B, A = logits.shape
    assert logits.is_contiguous() and dlogits.is_contiguous()
    assert workspace.numel() * workspace.element_size() >= loss_workspace_bytes(B)
    lib().call("sfb200_ppo_loss_fwd_bwd", _p(logits, F32), _p(values, F32), A, _p(actions_f32, F32),
               _p(log_prob_old, F32), _p(values_old, F32), _p(adv, F32), _p(targets, F32), _p(valids, U8),
               _p(logits_old, F32), B, clip_ratio, clip_value, exploration_coeff,
               {"entropy": 0, "symmetric_kl": 1}[exploration_loss], value_coeff, kl_coeff, grad_scale,
               _p(dlogits, F32), _p(dvalues, F32), _p(stats, F64), workspace.data_ptr(), _stream())


def action_ratio_tuple(logits: Tensor, head_sizes, actions_f32: Tensor, log_prob_old: Tensor, ratio: Tensor) -> None:
    B, A = logits.shape
    assert logits.is_contiguous() and actions_f32.is_contiguous()
    lib().call("sfb200_action_ratio_tuple", _p(logits, F32), A, len(head_sizes), _seg_array(head_sizes),
               _p(actions_f32, F32), _p(log_prob_old, F32), B, _p(ratio, F32), _stream())


def ppo_loss_fwd_bwd_tuple(logits: Tensor, values: Tensor, head_sizes, actions_f32: Tensor, log_prob_old: Tensor,
                           values_old: Tensor, adv: Tensor, targets: Tensor, valids: Tensor,
                           logits_old: Optional[Tensor], clip_ratio: float, clip_value: float,
                           exploration_coeff: float, value_coeff: float, kl_coeff: float, grad_scale: float,
                           dlogits: Tensor, dvalues: Tensor, stats: Tensor, workspace: Tensor,
                           exploration_loss: str = "entropy") -> None:
    """Tuple of Discretes: actions_f32 [B, K] (one index per head), logits / logits_old / dlogits [B, sum n_k]"""
    B, A = logits.shape
    assert logits.is_contiguous() and dlogits.is_contiguous() and actions_f32.is_contiguous()
    assert workspace.numel() * workspace.element_size() >= loss_workspace_bytes(B)
    lib().call("sfb200_ppo_loss_fwd_bwd_tuple", _p(logits, F32), _p(values, F32), A, len(head_sizes),
               _seg_array(head_sizes), _p(actions_f32, F32), _p(log_prob_old, F32), _p(values_old, F32), _p(adv, F32),
               _p(targets, F32), _p(valids, U8), _p(logits_old, F32), B, clip_ratio, clip_value, exploration_coeff,
               {"entropy": 0, "symmetric_kl": 1}[exploration_loss], value_coeff, kl_coeff, grad_scale,
               _p(dlogits, F32), _p(dvalues, F32), _p(stats, F64), workspace.data_ptr(), _stream())


def action_ratio_continuous(params: Tensor, actions_f32: Tensor, log_prob_old: Tensor, ratio: Tensor) -> None:
    B, A2 = params.shape
    assert params.is_contiguous() and actions_f32.is_contiguous()
    lib().call("sfb200_action_ratio_continuous", _p(params, F32), A2 // 2, _p(actions_f32, F32), _p(log_prob_old, F32),
               B, _p(ratio, F32), _stream())


def ppo_loss_fwd_bwd_continuous(params: Tensor, values: Tensor, adaptive_stddev: bool, tanh_scale: float,
                                actions_f32: Tensor, log_prob_old: Tensor, values_old: Tensor, adv: Tensor,
                                targets: Tensor, valids: Tensor, params_old: Optional[Tensor], clip_ratio: float,
                                clip_value: float, exploration_coeff: float, value_coeff: float, kl_coeff: float,
                                grad_scale: float, dlogits: Tensor, dlogstd: Optional[Tensor], dvalues: Tensor,
                                stats: Tensor, workspace: Tensor) -> None:
    """params / params_old [B, 2*Ad] = [means | log_std]; actions [B, Ad]; dlogits [B, 2*Ad] (adaptive) or [B, Ad]
    plus dlogstd [B, Ad] (learned stddev)."""
    B, A2 = params.shape
    Ad = A2 // 2
    assert params.is_contiguous() and dlogits.is_contiguous() and actions_f32.is_contiguous()
    assert dlogits.shape == (B, A2 if adaptive_stddev else Ad)
    assert params_old is None or params_old.is_contiguous()
    assert workspace.numel() * workspace.element_size() >= loss_workspace_bytes(B)
    lib().call("sfb200_ppo_loss_fwd_bwd_continuous", _p(params, F32), _p(values, F32), Ad, int(adaptive_stddev),
               float(tanh_scale), _p(actions_f32, F32), _p(log_prob_old, F32), _p(values_old, F32), _p(adv, F32),
               _p(targets, F32), _p(valids, U8), _p(params_old, F32), B, clip_ratio, clip_value, exploration_coeff,
               value_coeff, kl_coeff, grad_scale, _p(dlogits, F32), _p(dlogstd, F32), _p(dvalues, F32), _p(stats, F64),
               workspace.data_ptr(), _stream())


# ------------------------------------------------------------------------------------------------ learner: backward
def heads_backward_workspace_bytes(H: int, A: int) -> int:
    return lib().query("sfb200_heads_backward_workspace_bytes", H, A)


def heads_backward(h: Tensor, Wv: Tensor, Wa: Tensor, dlogits: Tensor, dvalues: Tensor, act: int, dz: Tensor,
                   dWv: Tensor, dbv: Tensor, dWa: Tensor, dba: Tensor, db_prev: Optional[Tensor],
                   workspace: Tensor) -> None:
    rows, H = h.shape
    A = Wa.shape[0]
    lib().call("sfb200_heads_backward", _p(h, F32), h.stride(0), rows, H, A, _p(Wv, F32), _p(Wa, F32),
               _p(dlogits, F32), _p(dvalues, F32), act, _p(dz, F32), dz.stride(0), _p(dWv, F32), _p(dbv, F32),
               _p(dWa, F32), _p(dba, F32), _p(db_prev, F32), workspace.data_ptr(), _stream())


def linear_backward_workspace_bytes(M: int, N: int, K: int) -> int:
    return lib().query("sfb200_linear_backward_workspace_bytes", M, N, K)


def linear_backward(dz: Tensor, x: Tensor, W: Tensor, act_prev: int, dW: Optional[Tensor], dx: Optional[Tensor],
                    db_prev: Optional[Tensor], engine: int, workspace: Tensor) -> None:
    M, N = dz.shape
    K = x.shape[1]
    assert W.shape == (N, K) and W.is_contiguous() and (dW is None or dW.is_contiguous())
    assert workspace.numel() * workspace.element_size() >= linear_backward_workspace_bytes(M, N, K)
    lib().call("sfb200_linear_backward", _p(dz, F32), dz.stride(0), _p(x, F32), x.stride(0), _p(W, F32), M, N, K,
               act_prev, _p(dW, F32), _p(dx, F32), 0 if dx is None else dx.stride(0), _p(db_prev, F32), engine,
               workspace.data_ptr(), _stream())


# ------------------------------------------------------------------------------------------------ optimizer
def clip_adam_step(p: Tensor, g: Tensor, m: Tensor, v: Tensor, step: int, lr: float, beta1: float, beta2: float,
                   eps: float, max_grad_norm: float, lr_scale_num: Optional[Tensor], lr_scale_den: Optional[Tensor],
                   grad_norm_out: Optional[Tensor], workspace: Tensor) -> None:
    for t in (p, g, m, v):
        assert t.is_contiguous() and t.dim() == 1
    assert workspace.numel() * workspace.element_size() >= 4096
    lib().call("sfb200_clip_adam_step", _p(p, F32), _p(g, F32), _p(m, F32), _p(v, F32), p.numel(), step, lr, beta1,
               beta2, eps, max_grad_norm, _p(lr_scale_num, F64), _p(lr_scale_den, F64), _p(grad_norm_out, F32),
               workspace.data_ptr(), _stream())


def lamb_workspace_bytes(num_tensors: int, max_numel: int) -> int:
    return lib().query("sfb200_lamb_workspace_bytes", num_tensors, max_numel)


def clip_lamb_step(p: Tensor, g: Tensor, m: Tensor, v: Tensor, seg_offsets: Tensor, seg_numel: Tensor, max_numel: int,
                   step: int, lr: float, beta1: float, beta2: float, eps: float, weight_decay: float, min_trust: float,
                   max_grad_norm: float, lr_scale_num: Optional[Tensor], lr_scale_den: Optional[Tensor],
                   grad_norm_out: Optional[Tensor], workspace: Tensor) -> None:
    """LAMB on the flat buffers; seg_offsets / seg_numel: int64 device tensors, one entry per parameter tensor"""
    for t in (p, g, m, v):
        assert t.is_contiguous() and t.dim() == 1
    T = seg_offsets.numel()
    assert seg_numel.numel() == T and workspace.numel() * workspace.element_size() >= lamb_workspace_bytes(T, max_numel)
    lib().call("sfb200_clip_lamb_step", _p(p, F32), _p(g, F32), _p(m, F32), _p(v, F32), p.numel(), _p(seg_offsets, I64),
               _p(seg_numel, I64), T, max_numel, step, lr, beta1, beta2, eps, weight_decay, min_trust, max_grad_norm,
               _p(lr_scale_num, F64), _p(lr_scale_den, F64), _p(grad_norm_out, F32), workspace.data_ptr(), _stream())


def compute_valids_dev(policy_id: Tensor, policy_version: Tensor, this_policy: int, train_step_dev: Tensor,
                       max_policy_lag: int, valids: Tensor) -> None:
    """compute_valids with the train-step counter in device memory (int64[1])"""
    n_traj, T = policy_id.shape
    assert policy_id.is_contiguous() and policy_version.is_contiguous() and valids.is_contiguous()
    assert valids.shape == (n_traj, T + 1)
    lib().call("sfb200_compute_valids_dev", _p(policy_id, I32), _p(policy_version, F32), n_traj, T, this_policy,
               _p(train_step_dev, I64), float(max_policy_lag), _p(valids, U8), _stream())


def clip_adam_step_dev(p: Tensor, g: Tensor, m: Tensor, v: Tensor, steps_done_dev: Tensor, lr_dev: Tensor, beta1: float,
                       beta2: float, eps: float, max_grad_norm: float, lr_scale_num: Optional[Tensor],
                       lr_scale_den: Optional[Tensor], grad_norm_out: Optional[Tensor], workspace: Tensor) -> None:
    """clip_adam_step with the step counter (int64[1], steps already taken) and the learning rate (float64[1]) in device
    memory -- every argument is then static, so the launch can be replayed from a CUDA graph"""
    for t in (p, g, m, v):
        assert t.is_contiguous() and t.dim() == 1
    assert workspace.numel() * workspace.element_size() >= 4096
    lib().call("sfb200_clip_adam_step_dev", _p(p, F32), _p(g, F32), _p(m, F32), _p(v, F32), p.numel(),
               _p(steps_done_dev, I64), _p(lr_dev, F64), beta1, beta2, eps, max_grad_norm, _p(lr_scale_num, F64),
               _p(lr_scale_den, F64), _p(grad_norm_out, F32), workspace.data_ptr(), _stream())


def advance_counters(a: Optional[Tensor], b: Optional[Tensor]) -> None:
    lib().call("sfb200_advance_counters", _p(a, I64), _p(b, I64), _stream())


# ------------------------------------------------------------------------------------------------ recurrent core
def _rs(t: Optional[Tensor]) -> int:
    return 0 if t is None else (t.stride(0) if t.dim() > 0 else 1)


def colsum_workspace_bytes(N: int) -> int:
    return lib().query("sfb200_colsum_workspace_bytes", N)


def colsum(x: Tensor, out: Tensor, workspace: Tensor) -> None:
    M, N = x.shape
    assert workspace.numel() * workspace.element_size() >= colsum_workspace_bytes(N)
    lib().call("sfb200_colsum", _p(x, F32), x.stride(0), M, N, _p(out, F32), workspace.data_ptr(), _stream())


def gru_cell_forward(gi: Tensor, gh: Tensor, h_in: Tensor, h_out: Tensor, h_next: Optional[Tensor] = None,
                     reset_next: Optional[Tensor] = None, gates: Optional[Tensor] = None) -> None:
    """All arguments are 2-D views with free row strides; reset_next is a 1-D bool view (any stride)."""
    M, H = h_in.shape
    lib().call("sfb200_gru_cell_forward", _p(gi, F32), gi.stride(0), _p(gh, F32), gh.stride(0), _p(h_in, F32),
               h_in.stride(0), _p(h_out, F32), h_out.stride(0), None if h_next is None else h_next.data_ptr(),
               _rs(h_next), None if reset_next is None else reset_next.data_ptr(), _rs(reset_next),
               None if gates is None else gates.data_ptr(), _rs(gates), M, H, _stream())


def gru_cell_backward(dh_out: Optional[Tensor], carry_a: Optional[Tensor], carry_b: Optional[Tensor],
                      reset: Optional[Tensor], gates: Tensor, gh: Tensor, h_in: Tensor, dgi: Tensor, dgh: Tensor,
                      dh_direct: Tensor) -> None:
    M, H = h_in.shape
    lib().call("sfb200_gru_cell_backward", None if dh_out is None else dh_out.data_ptr(), _rs(dh_out),
               None if carry_a is None else carry_a.data_ptr(), None if carry_b is None else carry_b.data_ptr(),
               _rs(carry_a), None if reset is None else reset.data_ptr(), _rs(reset), _p(gates, F32), gates.stride(0),
               _p(gh, F32), gh.stride(0), _p(h_in, F32), h_in.stride(0), _p(dgi, F32), dgi.stride(0), _p(dgh, F32),
               dgh.stride(0), _p(dh_direct, F32), dh_direct.stride(0), M, H, _stream())


def lstm_cell_forward(gi: Tensor, gh: Tensor, state_in: Tensor, state_out: Tensor, state_next: Optional[Tensor] = None,
                      reset_next: Optional[Tensor] = None, gates: Optional[Tensor] = None) -> None:
    M, H2 = state_in.shape
    lib().call("sfb200_lstm_cell_forward", _p(gi, F32), gi.stride(0), _p(gh, F32), gh.stride(0), _p(state_in, F32),
               state_in.stride(0), _p(state_out, F32), state_out.stride(0),
               None if state_next is None else state_next.data_ptr(), _rs(state_next),
               None if reset_next is None else reset_next.data_ptr(), _rs(reset_next),
               None if gates is None else gates.data_ptr(), _rs(gates), M, H2 // 2, _stream())


def lstm_cell_backward(dh_out: Optional[Tensor], dh_carry: Optional[Tensor], dc_carry: Optional[Tensor],
                       reset: Optional[Tensor], gates: Tensor, state_in: Tensor, state_out: Tensor, dgates: Tensor,
                       dc_in: Tensor) -> None:
    M, H2 = state_in.shape
    if dh_carry is not None and dc_carry is not None:
        assert dh_carry.stride(0) == dc_carry.stride(0)
    lib().call("sfb200_lstm_cell_backward", None if dh_out is None else dh_out.data_ptr(), _rs(dh_out),
               None if dh_carry is None else dh_carry.data_ptr(), None if dc_carry is None else dc_carry.data_ptr(),
               _rs(dh_carry if dh_carry is not None else dc_carry), None if reset is None else reset.data_ptr(), _rs(reset),
               _p(gates, F32), gates.stride(0), _p(state_in, F32), state_in.stride(0), _p(state_out, F32),
               state_out.stride(0), _p(dgates, F32), dgates.stride(0), _p(dc_in, F32), dc_in.stride(0), M, H2 // 2,
               _stream())


def mask_rows(src: Tensor, dst: Tensor, reset: Tensor) -> None:
    rows, dim = src.shape
    lib().call("sfb200_mask_rows", _p(src, F32), src.stride(0), _p(dst, F32), dst.stride(0), reset.data_ptr(),
               _rs(reset), rows, dim, _stream())


# ------------------------------------------------------------------------------------------------ data parallel (NVLink peers)
def ipc_export(t: Tensor):
    """(64-byte CUDA IPC handle of the allocation `t` lives in, byte offset of t inside it)"""
    import ctypes

    handle = ctypes.create_string_buffer(64)
    off = ctypes.c_int64(0)
    lib().call("sfb200_ipc_export", t.data_ptr(), ctypes.cast(handle, ctypes.c_void_p), ctypes.cast(ctypes.byref(off), ctypes.c_void_p))
    return bytes(handle.raw), int(off.value)


def ipc_import(handle: bytes, offset: int) -> int:
    """device address (in THIS process) of a peer's exported buffer"""
    import ctypes

    h = ctypes.create_string_buffer(handle, 64)
    out = ctypes.c_void_p(0)
    lib().call("sfb200_ipc_import", ctypes.cast(h, ctypes.c_void_p), offset, ctypes.cast(ctypes.byref(out), ctypes.c_void_p))
    return int(out.value)


def ipc_close(ptr: int, offset: int) -> None:
    lib().call("sfb200_ipc_close", ptr, offset)


def dp_header_bytes() -> int:
    return lib().query("sfb200_dp_header_bytes")


def dp_create(rank: int, world: int, peer_ptrs, scratch_bytes: int) -> int:
    import ctypes

    arr = (ctypes.c_uint64 * world)(*[int(p) for p in peer_ptrs])
    comm = lib().query("sfb200_dp_create", rank, world, ctypes.cast(arr, ctypes.c_void_p), scratch_bytes)
    if comm < 0:
        msg = lib().cdll.sfb200_last_error()
        raise RuntimeError(f"sfb200_dp_create failed: {msg.decode() if msg else '?'}")
    return comm


def dp_destroy(comm: int) -> None:
    lib().call("sfb200_dp_destroy", comm)


def dp_grad_allreduce(comm: int, g_out: Tensor, workspace: Tensor) -> None:
    assert workspace.numel() * workspace.element_size() >= 4096
    lib().call("sfb200_dp_grad_allreduce", comm, _p(g_out, F32), g_out.numel(), workspace.data_ptr(), _stream())


def dp_grad_allreduce_clip_adam(comm: int, g_out: Tensor, p: Tensor, m: Tensor, v: Tensor, step: int,
                                steps_done_dev: Optional[Tensor], lr: float, lr_dev: Optional[Tensor], beta1: float,
                                beta2: float, eps: float, max_grad_norm: float, lr_scale_num: Optional[Tensor],
                                lr_scale_den: Optional[Tensor], grad_norm_out: Optional[Tensor], workspace: Tensor) -> None:
    for t in (p, g_out, m, v):
        assert t.is_contiguous() and t.dim() == 1
    assert workspace.numel() * workspace.element_size() >= 4096
    lib().call("sfb200_dp_grad_allreduce_clip_adam", comm, _p(g_out, F32), _p(p, F32), _p(m, F32), _p(v, F32), p.numel(),
               step, _p(steps_done_dev, I64), lr, _p(lr_dev, F64), beta1, beta2, eps, max_grad_norm,
               _p(lr_scale_num, F64), _p(lr_scale_den, F64), _p(grad_norm_out, F32), workspace.data_ptr(), _stream())


def dp_allreduce_f64(comm: int, buf: Tensor, row_len: int = 0, max_mask: int = 0, min_mask: int = 0, keep_mask: int = 0,
                     avg_mask: int = 0) -> None:
    assert buf.is_contiguous()
    lib().call("sfb200_dp_allreduce_f64", comm, _p(buf, F64), buf.numel(), row_len, max_mask, min_mask, keep_mask, avg_mask,
               _stream())


def dp_pooled_moments(comm: int, batch_mean: Tensor, batch_var: Tensor, rows_per_rank: int) -> None:
    lib().call("sfb200_dp_pooled_moments", comm, _p(batch_mean, F32), _p(batch_var, F32), batch_mean.numel(),
               float(rows_per_rank), _stream())


def colsum_f64(src: Tensor, col: int, out: Tensor) -> None:
    """out[0] = src[:, col].sum() for a dense float64 [rows, stride] tensor"""
    assert src.dim() == 2 and src.is_contiguous()
    lib().call("sfb200_colsum_f64", _p(src, F64), src.shape[0], src.shape[1], col, _p(out, F64), _stream())
