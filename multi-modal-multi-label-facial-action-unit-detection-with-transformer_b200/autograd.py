"""torch.autograd bridges for the training step (train.py:206-236): every region of the hot path is one
``autograd.Function`` whose forward runs the tape-keeping CUDA forward and whose backward runs the hand-written
backward kernels, so ``loss.backward()`` in the reference's training loop works unchanged and the conv backbones
(plain torch) receive their input gradients.  Parameters are passed as Function inputs so that autograd accumulates
the returned gradients into ``p.grad`` like for any other module; when ``p.grad`` already exists as an fp32 buffer
(FusedAdam keeps them as views of its flat gradient bucket) the encoder kernels accumulate straight into it instead.

No arithmetic happens in torch here: tensors are allocated, viewed and handed to libavformer_b200.so.
"""
from __future__ import annotations

from typing import List

import torch

from . import functional as AF


# Listeners told which parameters' gradient kernels have just been enqueued on the current stream (optim.FusedAdam starts the
# all-reduce of a bucket segment as soon as the last of its parameters is reported).  Called at the END of each bridge's backward.
_GRAD_LISTENERS: List = []


def add_grad_listener(fn) -> None:
    if fn not in _GRAD_LISTENERS:
        _GRAD_LISTENERS.append(fn)


def remove_grad_listener(fn) -> None:
    if fn in _GRAD_LISTENERS:
        _GRAD_LISTENERS.remove(fn)


def _notify(params) -> None:
    for fn in _GRAD_LISTENERS:
        fn(params)


def _f32_dense(t: torch.Tensor) -> torch.Tensor:
    return t if (t.dtype == torch.float32 and t.is_contiguous()) else t.float().contiguous()


def direct_grad_ok(prm) -> bool:
    """May the kernels add this parameter's gradient straight into ``prm.grad``, bypassing autograd's AccumulateGrad?  Only when an
    optimiser asked for it (optim.FusedAdam marks the parameters whose .grad is a view of its flat bucket with ``_avf_direct_grad``)
    and nobody is listening on the normal path: tensor hooks and post-accumulate-grad hooks (torch DDP's reducer registers those)
    only fire when the gradient is returned to autograd.  torch.autograd.grad() / backward(inputs=...) on such parameters still
    see None — FusedAdam-managed parameters are meant for loss.backward() + optimizer.step(); torch DDP is not supported on
    them (dp.SegmentReducer / FusedAdam do the reduction)."""
    pg = prm.grad
    if pg is None or not getattr(prm, "_avf_direct_grad", False):
        return False
    if pg.dtype != torch.float32 or not pg.is_cuda or not pg.is_contiguous():
        return False
    if getattr(prm, "_backward_hooks", None) or getattr(prm, "_post_accumulate_grad_hooks", None):
        return False
    return True


def _direct_targets(params):
    return [p.grad if direct_grad_ok(p) else None for p in params]


def _hand_over(params, grads):
    """Gradient hand-over without one `add` launch per parameter: when every parameter that receives a gradient here already
    owns an fp32 ``.grad`` buffer of the right shape on the GPU (FusedAdam keeps them as views of its flat bucket), all the
    gradients are accumulated into those buffers with ONE multi-tensor launch and the Function returns None for them (autograd
    then has nothing to accumulate) — the AU_former front alone has 27 small parameters.  Otherwise the gradients are
    returned unchanged and autograd's AccumulateGrad does what it always does."""
    dst, src = [], []
    for prm, g in zip(params, grads):
        if g is None:
            continue
        pg = prm.grad
        if not direct_grad_ok(prm) or pg.shape != g.shape or not g.is_cuda:
            return list(grads)
        dst.append(pg)
        src.append(g if g.dtype == torch.float32 else g.float())
    if dst:
        torch._foreach_add_(dst, src)
    return [None] * len(grads)


class EncoderStackFn(torch.autograd.Function):
    """Transformer (models/heads.py:242-256) on an fp32 token matrix [n_seq*n_tok, dim]; ``keep`` [n_seq, n_tok] bool (or None) is
    the attention mask of every layer, a non-differentiable input."""

    @staticmethod
    def forward(ctx, x, tr, n_seq, n_tok, keep, *params):
        packed = tr.packed()
        shape = tr.shape(n_seq, n_tok)
        ctx.drop = tr.dropout_state()
        y, tape = AF.encoder_stack_fwd_train(_f32_dense(x.detach()), packed, shape, *ctx.drop, keep=keep)
        ctx.packed, ctx.shape_, ctx.tape, ctx.params, ctx.keep = packed, shape, tape, params, keep
        return y

    @staticmethod
    def backward(ctx, dy):
        needs = ctx.needs_input_grad
        dx = _f32_dense(dy).clone()
        dx, grads = AF.encoder_stack_bwd_(dx, ctx.packed, ctx.shape_, ctx.tape, list(needs[5:]), *ctx.drop, into=_direct_targets(ctx.params),
                                          keep=ctx.keep)
        ctx.tape = ctx.keep = None
        _notify(ctx.params)
        return (dx if needs[0] else None, None, None, None, None, *grads)


class SFormerFn(torch.autograd.Function):
    """models/vformer.py:245-259: NCHW map -> tokens + pos -> encoder -> NCHW map."""

    @staticmethod
    def forward(ctx, fmap, pos, tr, *params):
        F_, C, H, W = fmap.shape
        packed = tr.packed()
        shape = tr.shape(F_, H * W)
        x = AF.sformer_tokens_pack(fmap.detach(), pos.detach().reshape(-1, C)[: H * W])
        ctx.drop = tr.dropout_state()
        y, tape = AF.encoder_stack_fwd_train(x, packed, shape, *ctx.drop)
        ctx.packed, ctx.shape_, ctx.tape, ctx.fshape, ctx.fdtype, ctx.pos_shape = packed, shape, tape, (F_, C, H, W), fmap.dtype, pos.shape
        ctx.params = params
        ctx.pos_param = pos
        return AF.sformer_tokens_unpack(y, (F_, C, H, W), fmap.dtype)

    @staticmethod
    def backward(ctx, dout):
        needs = ctx.needs_input_grad
        F_, C, H, W = ctx.fshape
        dx = AF.sformer_tokens_pack(dout, None)
        dx, grads = AF.encoder_stack_bwd_(dx, ctx.packed, ctx.shape_, ctx.tape, list(needs[3:]), *ctx.drop, into=_direct_targets(ctx.params))
        ctx.tape = None
        dpos = None
        if needs[1]:
            dpos = torch.zeros(ctx.pos_shape, dtype=torch.float32, device=dx.device)
            dpos.view(-1, C)[: H * W] = AF.colsum(dx.view(F_, H * W * C)).view(H * W, C)
        dfmap = AF.sformer_tokens_unpack(dx, ctx.fshape, ctx.fdtype) if needs[0] else None
        (dpos,) = _hand_over((ctx.pos_param,), (dpos,))
        _notify(ctx.params + (ctx.pos_param,))
        return (dfmap, dpos, None, *grads)


class TFormerEmbedFn(torch.autograd.Function):
    """models/vformer.py:280-286: cat(cls, frames) + pos -> fp32 tokens [n_clips*(T+1), dim]."""

    @staticmethod
    def forward(ctx, frames, cls_token, pos, n_frames):
        ctx.meta = (frames.shape, frames.dtype, n_frames, cls_token.shape, pos.shape)
        ctx.params = (cls_token, pos)
        return AF.tformer_embed(frames.detach(), cls_token.detach().reshape(-1), pos.detach()[0], n_frames)

    @staticmethod
    def backward(ctx, dtok):
        fshape, fdtype, T, cshape, pshape = ctx.meta
        needs = ctx.needs_input_grad
        dtok = _f32_dense(dtok)
        dim = dtok.shape[1]
        n_clips = dtok.shape[0] // (T + 1)
        dframes = dcls = dpos = None
        if needs[0]:
            dframes = dtok.view(n_clips, T + 1, dim)[:, 1:].reshape(fshape).to(fdtype)
        if needs[1] or needs[2]:
            s = AF.colsum(dtok.view(n_clips, (T + 1) * dim))
            dpos = s.view(pshape) if needs[2] else None
            dcls = s[:dim].clone().view(cshape) if needs[1] else None
        dcls, dpos = _hand_over(ctx.params, (dcls, dpos))
        _notify(ctx.params)
        return dframes, dcls, dpos, None


class AUFrontFn(torch.autograd.Function):
    """models/heads.py:293-323: BatchNorm1d -> 12 x Linear(512,128) -> view [B,12,128] -> + pos."""

    @staticmethod
    def forward(ctx, emb, bn_w, bn_b, pos, head, n_clips, *wb):
        f = head._packed_front()
        bn = head.AU_BN1
        batch_stats = bool(bn.training)
        emb_d = emb.detach()
        if emb_d.dtype != torch.float32 or emb_d.stride(-1) != 1:
            emb_d = emb_d.float().contiguous()
        momentum = 0.1 if bn.momentum is None else bn.momentum
        x, tape = AF.au_former_front_train(emb_d, n_clips, bn_w.detach(), bn_b.detach(), bn.running_mean, bn.running_var, batch_stats, momentum,
                                           f.w, f.b, pos.detach()[0], f.mode)
        if batch_stats and bn.num_batches_tracked is not None:
            bn.num_batches_tracked += 1
        ctx.saved = (emb_d, f, bn, batch_stats, tape, n_clips, pos.shape, emb.shape, emb.dtype)
        ctx.save_for_backward(bn_w)
        ctx.params = (bn_w, bn_b, pos) + tuple(wb)
        return x

    @staticmethod
    def backward(ctx, dx):
        emb_d, f, bn, batch_stats, tape, n_clips, pos_shape, emb_shape, emb_dtype = ctx.saved
        (bn_w,) = ctx.saved_tensors
        needs = ctx.needs_input_grad
        want_w = any(needs[6:])
        demb, dg, db, dw, dbc = AF.au_former_front_bwd(emb_d, n_clips, bn_w.detach(), bn.running_mean, bn.running_var, batch_stats, f.w, tape,
                                                       _f32_dense(dx), f.mode, want_emb=needs[0], want_bn=needs[1] or needs[2], want_w=want_w)
        emb_dim = f.w.shape[0] // 12
        wb_grads: List = []
        for i in range(12):
            wb_grads.append(dw[i * emb_dim:(i + 1) * emb_dim] if (want_w and needs[6 + 2 * i]) else None)
            wb_grads.append(dbc[i * emb_dim:(i + 1) * emb_dim] if needs[7 + 2 * i] else None)
        if demb is not None:
            demb = demb.view(emb_shape).to(emb_dtype)
        pg = _hand_over(ctx.params, [dg if needs[1] else None, db if needs[2] else None, dbc.view(pos_shape).clone() if needs[3] else None] + wb_grads)
        _notify(ctx.params)
        return (demb, pg[0], pg[1], pg[2], None, None, *pg[3:])


class AddPosFn(torch.autograd.Function):
    """x[r,:] + pos[r % period,:] on an fp32 token matrix (models/tformer.py:387)."""

    @staticmethod
    def forward(ctx, x, pos, period):
        ctx.meta = (pos.shape, period)
        ctx.params = (pos,)
        y = _f32_dense(x.detach()).clone()
        return AF.add_row_periodic_(y, pos.detach().reshape(period, -1), period)

    @staticmethod
    def backward(ctx, dy):
        pshape, period = ctx.meta
        needs = ctx.needs_input_grad
        dpos = None
        if needs[1]:
            d = _f32_dense(dy)
            dpos = AF.colsum(d.view(d.shape[0] // period, period * d.shape[1])).view(pshape)
        (dpos,) = _hand_over(ctx.params, (dpos,))
        _notify(ctx.params)
        return (dy if needs[0] else None), dpos, None


class AULogitsFn(torch.autograd.Function):
    """models/tformer.py:389-401 + models/avformer.py:102-105: 12 per-token dots -> zero-padded [B,21]."""

    @staticmethod
    def forward(ctx, tokens, head, n_clips, *w12):
        last = head._packed_last()
        tok = _f32_dense(tokens.detach())
        ctx.saved = (tok, last, n_clips)
        ctx.params = tuple(w12)
        return AF.au_logits(tok, last.w, n_clips)

    @staticmethod
    def backward(ctx, dout21):
        tok, last, n_clips = ctx.saved
        needs = ctx.needs_input_grad
        d = dout21 if (dout21.dtype == torch.float32 and dout21.stride(-1) == 1) else dout21.float().contiguous()
        want_dw = any(needs[3:])
        dx, dw = AF.au_logits_bwd(d, tok, last.w, n_clips, want_dx=needs[0], want_dw=want_dw)
        pg = _hand_over(ctx.params, [(dw[i:i + 1] if needs[3 + i] else None) for i in range(12)])
        _notify(ctx.params)
        return (dx, None, None, *pg)
