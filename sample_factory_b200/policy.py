"""Forward pass of the actor-critic on the device: encoder MLP -> (recurrent core) -> decoder MLP -> heads
(reference: ActorCriticSharedWeights.forward_head / forward_core / forward_tail, model/actor_critic.py:160-195).

One function serves the three call sites of the hot path (sampler policy step, learner bootstrap value, learner
minibatch forward).  When the tensor feeding critic_linear / distribution_linear is the output of an MLP layer and the
tcgen05 engine covers the shape, that layer and the heads run as ONE GEMM whose epilogue leaves partial head dot
products (sfb200_linear_act_heads_forward) followed by a tiny finishing kernel (sfb200_heads_from_partials); the
activated layer output is stored only if the caller needs it (the learner's backward does, the sampler does not).
"""
from __future__ import annotations

from typing import Callable, Dict, List, Optional

import torch
from torch import Tensor

from . import ops
from .model import PolicyModel


class HeadsPlan:
    """Per call-site forward plan: decides once per (model, engine) whether the fused last-layer + heads path applies,
    owns its scratch, and owns the conv head's buffers for image observations."""

    def __init__(self, model: PolicyModel, engine: int, max_rows: int, need_backward: bool = False):
        spec = model.spec
        self.conv = None
        if spec.obs_shape is not None:
            from .conv_encoder import ConvHead

            self.conv = ConvHead(model, engine, max_rows, need_backward)
        self.tail_is_mlp = bool(spec.decoder_mlp_layers) or (not spec.use_rnn and bool(spec.fc_encoder_layers))
        # separate actor / critic weights: per-tower activations and ONE concatenated tail [rows, 2H] = [actor | critic]
        self.separate = not spec.share_weights
        if self.separate:
            f32 = dict(dtype=torch.float32, device=model.device)
            widths, H = spec.hidden, spec.tail_input_size
            assert len(widths) > 0, "separate actor / critic weights need at least one MLP layer per tower"
            self.tower_h = {tw: [torch.empty((max_rows, w), **f32) for w in widths[:-1]] for tw in ("actor_", "critic_")}
            self.tail_cat = torch.empty((max_rows, 2 * H), **f32)
            if need_backward:
                A = spec.num_linear_action_outputs
                self.tower_dz = {tw: [torch.empty((max_rows, w), **f32) for w in widths[:-1]] for tw in ("actor_", "critic_")}
                self.dz_cat = torch.empty((max_rows, 2 * H), **f32)
                self.gWv_cat = torch.empty((1, 2 * H), **f32)
                self.gWa_cat = torch.empty((A, 2 * H), **f32)
                self.db_cat = torch.empty(2 * H, **f32)
        self.P = 0
        if self.separate:
            return
        self.part: Optional[Tensor] = None
        if self.tail_is_mlp:
            self.P = ops.linear_heads_partials(spec.tail_input_size, spec.num_linear_action_outputs, engine)
        if self.P > 0:
            self.part = torch.empty(self.P * max_rows * ops.HEAD_PART_PAD, dtype=torch.float32, device=model.device)


def forward_policy(model: PolicyModel, x: Tensor, outs: List[Tensor], act: int, engine: int, plan: HeadsPlan,
                   heads_kwargs: Dict, rnn_fn: Optional[Callable[[Tensor], Tensor]] = None,
                   store_tail: bool = True, finish_fn: Optional[Callable] = None) -> Tensor:
    """x [M, D] (rows may be strided) -> heads outputs described by `heads_kwargs` (the keyword arguments of
    ops.heads_forward after the weights).  outs: one [>=M, h] buffer per MLP layer.  Returns the tensor that fed the
    heads (None if it was not stored)."""
    M = x.shape[0]
    if plan.separate:
        return _forward_separate(model, x, act, engine, plan, heads_kwargs)
    if plan.conv is not None:        # ConvEncoder: conv head first, its fully connected layers are `enc` below
        x = plan.conv.forward(x)
    enc, dec = model.encoder_layers(), model.decoder_layers()
    Wv, bv = model.critic
    Wa, ba = model.actor
    n_mlp = len(enc) + len(dec)
    fused = plan.P > 0
    k = 0
    tail: Optional[Tensor] = x
    for group, layers in (("enc", enc), ("dec", dec)):
        if group == "dec" and rnn_fn is not None:
            tail = rnn_fn(tail)
        for (W, b) in layers:
            last = fused and k == n_mlp - 1
            if last:
                out = outs[k][:M] if store_tail else None
                ops.linear_act_heads_forward(tail, W, b, out, act, engine, Wv, Wa, plan.part)
                tail = out
            else:
                ops.linear_act_forward(tail, W, b, outs[k][:M], act, engine)
                tail = outs[k][:M]
            k += 1
    if finish_fn is not None and fused:
        finish_fn(plan.part, plan.P, M, bv, ba)
    else:
        _heads(model, tail, Wv, bv, Wa, ba, fused, plan, M, heads_kwargs)
    return tail


def _forward_separate(model: PolicyModel, x: Tensor, act: int, engine: int, plan: HeadsPlan, heads_kwargs: Dict) -> Tensor:
    """ActorCriticSeparateWeights (model/actor_critic.py:283-318): two MLP towers on the same normalised observation; the
    towers' last layers write the two halves of one [M, 2H] tail, and the heads read it through zero-padded weights
    (PolicyModel.refresh_cat_heads), so value = critic half . Wv and logits = actor half . Wa^T."""
    M = x.shape[0]
    H = model.spec.tail_input_size
    for tw, col in (("actor_", 0), ("critic_", H)):
        t = x
        layers = model.tower_layers(tw)
        for k, (W, b) in enumerate(layers):
            out = plan.tail_cat[:M, col: col + H] if k == len(layers) - 1 else plan.tower_h[tw][k][:M]
            ops.linear_act_forward(t, W, b, out, act, engine)
            t = out
    _, bv = model.critic
    _, ba = model.actor
    tail = plan.tail_cat[:M]
    _heads(model, tail, model.Wv_cat, bv, model.Wa_cat, ba, False, plan, M, heads_kwargs)
    return tail


def _heads(model: PolicyModel, tail: Tensor, Wv: Tensor, bv: Tensor, Wa: Tensor, ba: Tensor, fused: bool, plan: HeadsPlan,
           M: int, heads_kwargs: Dict) -> None:
    if model.spec.continuous:   # Box action space: Gaussian heads (action_distributions.py:290-323)
        dk = model.dist_kwargs()
        if fused:
            ops.heads_from_partials_continuous(plan.part, plan.P, M, bv, ba, **dk, **heads_kwargs)
        else:
            ops.heads_forward_continuous(tail, Wv, bv, Wa, ba, **dk, **heads_kwargs)
    elif model.spec.action_segments:   # Tuple of Discretes: independent categorical heads (action_distributions.py:197-286)
        if fused:
            ops.heads_from_partials_tuple(plan.part, plan.P, M, bv, ba, model.spec.action_segments, **heads_kwargs)
        else:
            ops.heads_forward_tuple(tail, Wv, bv, Wa, ba, model.spec.action_segments, **heads_kwargs)
    elif fused:
        ops.heads_from_partials(plan.part, plan.P, M, bv, ba, **heads_kwargs)
    else:
        ops.heads_forward(tail, Wv, bv, Wa, ba, **heads_kwargs)
