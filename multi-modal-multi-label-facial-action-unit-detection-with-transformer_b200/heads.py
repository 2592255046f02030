"""AU-token encoders: the per-modality AU_former (models/heads.py:258-339) and the audio-visual fusion
head former_AU_head (== tformer_AU_head, models/tformer.py:362-403; models/avformer.py:19,87), with the
reference's parameter names (AU_BN1, AU_linear_p1..12, pos_embedding, corr_transformer, AU_linear_last1..12).
"""
from __future__ import annotations

from typing import Optional

import torch
from torch import nn

from . import functional as AF
from .encoder import Transformer, default_precision, needs_grad


class _PackedFront:
    """The 12 Linear(512,128) stacked to one [1536,512] operand (+ [1536] bias); re-packed when any source changes."""

    def __init__(self, linears, mode):
        self.mode = mode
        self.sources = [p for l in linears for p in (l.weight, l.bias)]
        w = torch.cat([l.weight.detach().float() for l in linears], dim=0).contiguous()
        self.w = AF.to_bf16(w) if mode == AF.AVF_BF16 else w
        self.b = torch.cat([l.bias.detach().float() for l in linears], dim=0).contiguous()
        self.versions = [AF._src_version(s) for s in self.sources]
        self.epoch = AF.WEIGHTS_EPOCH

    def stale(self):
        return self.epoch != AF.WEIGHTS_EPOCH or any(AF._src_version(s) != v for s, v in zip(self.sources, self.versions))


class _PackedLast:
    def __init__(self, linears):
        self.sources = [l.weight for l in linears]
        self.w = torch.cat([l.weight.detach().float() for l in linears], dim=0).contiguous()     # [12, dim]
        self.versions = [AF._src_version(s) for s in self.sources]
        self.epoch = AF.WEIGHTS_EPOCH

    def stale(self):
        return self.epoch != AF.WEIGHTS_EPOCH or any(AF._src_version(s) != v for s, v in zip(self.sources, self.versions))


class AU_former(nn.Module):
    """AU_former(input_dim=512, emb_dim=128, dropout=0.0); forward(emb[B,512]) -> (AU_out[B,12], tokens[B,12,128])."""

    def __init__(self, input_dim=512, emb_dim=128, dropout=0.0):
        super().__init__()
        self.emb_dim = input_dim                       # (sic) the reference stores the INPUT width here
        self.token_dim = emb_dim
        self.AU_BN1 = nn.BatchNorm1d(input_dim)
        for i in range(1, 13):
            setattr(self, f"AU_linear_p{i}", nn.Linear(input_dim, emb_dim))
        self.pos_embedding = nn.Parameter(torch.randn(1, 12, emb_dim))
        self.corr_transformer = Transformer(emb_dim, depth=2, heads=8, mlp_dim=256, dim_head=32, dropout=dropout)
        for i in range(1, 13):
            setattr(self, f"AU_linear_last{i}", nn.Linear(emb_dim, 1, bias=False))
        self._front: Optional[_PackedFront] = None
        self._last: Optional[_PackedLast] = None

    def _packed_front(self):
        mode = AF._mode(self.corr_transformer.precision or default_precision())
        if self._front is None or self._front.mode != mode or self._front.stale():
            self._front = _PackedFront([getattr(self, f"AU_linear_p{i}") for i in range(1, 13)], mode)
        return self._front

    def _packed_last(self):
        if self._last is None or self._last.stale():
            self._last = _PackedLast([getattr(self, f"AU_linear_last{i}") for i in range(1, 13)])
        return self._last

    def tokens_into(self, emb: torch.Tensor, ld_emb: int, n_clips: int, out: Optional[torch.Tensor] = None, ld_out: int = 0,
                    maps: bool = False):
        """BN -> 12 projections -> + pos -> 2 encoder layers.  ``emb`` may be a strided view (row stride
        ld_emb): the cls rows of a TFormer token matrix are consumed in place.  The last layer's result goes
        to ``out`` (row stride ld_out) when given — that is how the audio and video halves of the
        [B,12,256] fusion input get written side by side without a cat (models/avformer.py:100).  With
        BatchNorm in eval() the positional add is part of the encoder-stack launch.  ``maps``: run the stack kernel by kernel
        (Transformer.maps_) and return its attention maps [2, n_clips, 8, 12, 12] instead of the tokens, which still go to out / x."""
        stack = self.corr_transformer.maps_ if maps else self.corr_transformer.forward_
        f = self._packed_front()
        bn = self.AU_BN1
        if bn.training:
            # train() without gradients (a frozen sub-model inside a training loop): batch statistics, running ones updated
            view = torch.as_strided(emb, (n_clips, f.w.shape[1]), (ld_emb, 1))
            x, _ = AF.au_former_front_train(view, n_clips, bn.weight, bn.bias, bn.running_mean, bn.running_var, True,
                                            0.1 if bn.momentum is None else bn.momentum, f.w, f.b, self.pos_embedding[0], f.mode)
            bn.num_batches_tracked += 1
            return stack(x, n_clips, 12, out, ld_out)
        x = AF.au_former_front(emb, ld_emb, n_clips, (bn.weight, bn.bias, bn.running_mean, bn.running_var), f.w, f.b, None, f.mode)
        return stack(x, n_clips, 12, out, ld_out, pos=self.pos_embedding[0])

    def front_params(self):
        return [p for i in range(1, 13) for p in (getattr(self, f"AU_linear_p{i}").weight, getattr(self, f"AU_linear_p{i}").bias)]

    def tokens_train(self, emb: torch.Tensor, n_clips: int) -> torch.Tensor:
        """Autograd-visible version of tokens_into: emb [n_clips, 512] (any row stride) -> tokens [n_clips*12, emb_dim]."""
        from .autograd import AUFrontFn
        x = AUFrontFn.apply(emb, self.AU_BN1.weight, self.AU_BN1.bias, self.pos_embedding, self, n_clips, *self.front_params())
        return self.corr_transformer.forward_train(x, n_clips, 12)

    def relevance_fwd_(self, emb: torch.Tensor, n_clips: int):
        """tokens_train's forward (running statistics: eval()) without recording: (tokens [n_clips*12, emb_dim], ctx for relevance_bwd_);
        the tokens equal tokens_train's bit for bit."""
        f = self._packed_front()
        bn = self.AU_BN1
        emb_d = emb.detach()
        if emb_d.dtype != torch.float32 or emb_d.stride(-1) != 1:
            emb_d = emb_d.float().contiguous()
        x, ftape = AF.au_former_front_train(emb_d, n_clips, bn.weight.detach(), bn.bias.detach(), bn.running_mean, bn.running_var, False,
                                            0.1 if bn.momentum is None else bn.momentum, f.w, f.b, self.pos_embedding.detach()[0], f.mode)
        y, tape = self.corr_transformer.relevance_fwd_(x, n_clips, 12)
        return y, (emb_d, f, ftape, tape, n_clips)

    def relevance_bwd_(self, ctx, dy: torch.Tensor, maps: bool = True, want_emb: bool = False):
        """Backward of relevance_fwd_ from dy [n_clips*12, emb_dim] fp32 dense (used as scratch), activations only: (gradient maps
        [2, n_clips, 8, 12, 12] or None, dL/demb [n_clips, in_dim] or None)."""
        emb_d, f, ftape, tape, n_clips = ctx
        gmaps = self.corr_transformer.relevance_bwd_(dy, tape, n_clips, 12, maps=maps)
        demb = None
        if want_emb:
            bn = self.AU_BN1
            demb = AF.au_former_front_bwd(emb_d, n_clips, bn.weight.detach(), bn.running_mean, bn.running_var, False, f.w, ftape, dy, f.mode,
                                          want_emb=True, want_bn=False, want_w=False)[0]
        return gmaps, demb

    def forward(self, emb):
        AF._cuda(emb, "emb")
        bs = emb.shape[0]
        if needs_grad(self, emb):
            tok = self.tokens_train(emb, bs)
            with torch.no_grad():      # the per-modality AU logits are discarded by the AVFormer (models/avformer.py:53,70): no gradient path
                au_out = AF.au_logits(tok.detach(), self._packed_last().w, bs)[:, :12]
            return au_out, tok.view(bs, 12, -1)
        emb = emb.detach().float().contiguous()
        tok = self.tokens_into(emb, emb.shape[1], bs)
        au_out = AF.au_logits(tok, self._packed_last().w, bs)[:, :12]
        return au_out, tok.view(bs, 12, -1)


class former_AU_head(nn.Module):
    """former_AU_head(emb_dim=128, dropout=0.0); forward([B,12,emb_dim]) -> logits [B,12]."""

    def __init__(self, emb_dim=128, dropout=0.0):
        super().__init__()
        self.pos_embedding = nn.Parameter(torch.randn(1, 12, emb_dim))
        self.corr_transformer = Transformer(emb_dim, depth=3, heads=8, mlp_dim=256, dim_head=32, dropout=dropout)
        for i in range(1, 13):
            setattr(self, f"AU_linear_last{i}", nn.Linear(emb_dim, 1, bias=False))
        self._last: Optional[_PackedLast] = None

    def _packed_last(self):
        if self._last is None or self._last.stale():
            self._last = _PackedLast([getattr(self, f"AU_linear_last{i}") for i in range(1, 13)])
        return self._last

    def logits21_(self, tokens2d: torch.Tensor, n_clips: int, want_decisions: bool = False):
        """On fp32 tokens [n_clips*12, emb_dim] (used as scratch): + pos, 3 layers, 12 dots -> [B,21] zero-padded."""
        t = self.corr_transformer
        if t.training and t.dropout > 0.0:          # dropout: the tape-keeping kernels of forward_
            t.forward_(tokens2d, n_clips, 12, pos=self.pos_embedding[0])
            return AF.au_logits(tokens2d, self._packed_last().w, n_clips, want_decisions)
        return AF.token_stack_fwd_(tokens2d, t.packed(), t.shape(n_clips, 12), self.pos_embedding[0], w_last=self._packed_last().w,
                                   want_decisions=want_decisions)

    def logits21_maps_(self, tokens2d: torch.Tensor, n_clips: int):
        """logits21_ kernel by kernel with the attention maps of the three layers: ([B,21], maps [3, n_clips, 8, 12, 12]); the logits
        equal logits21_'s with set_fused_enabled(False) bit for bit (the same positional add, layers and logits launches)."""
        maps = self.corr_transformer.maps_(tokens2d, n_clips, 12, pos=self.pos_embedding[0])
        return AF.au_logits(tokens2d, self._packed_last().w, n_clips), maps

    def last_params(self):
        return [getattr(self, f"AU_linear_last{i}").weight for i in range(1, 13)]

    def logits21_train(self, tokens2d: torch.Tensor, n_clips: int) -> torch.Tensor:
        """Autograd-visible version of logits21_ on fp32 tokens [n_clips*12, emb_dim] -> [B,21]."""
        from .autograd import AddPosFn, AULogitsFn
        x = AddPosFn.apply(tokens2d, self.pos_embedding, 12)
        x = self.corr_transformer.forward_train(x, n_clips, 12)
        return AULogitsFn.apply(x, self, n_clips, *self.last_params())

    def relevance_fwd_(self, tokens2d: torch.Tensor, n_clips: int):
        """logits21_train's forward without recording: ([B,21] equal to logits21_train's bit for bit, ctx for relevance_bwd_)."""
        x = AF.add_row_periodic_(tokens2d.detach().float().contiguous().clone(), self.pos_embedding.detach().reshape(12, -1), 12)
        y, tape = self.corr_transformer.relevance_fwd_(x, n_clips, 12)
        last = self._packed_last()
        return AF.au_logits(y, last.w, n_clips), (y, tape, last, n_clips)

    def relevance_bwd_(self, ctx, weights: torch.Tensor, maps: bool = True):
        """Backward of relevance_fwd_ seeded with d out21[:, :12] = weights [n_clips, 12] fp32 (d out21[:, 12:] = 0), activations only:
        (gradient maps [3, n_clips, 8, 12, 12] or None, dL/dtokens [n_clips*12, emb_dim])."""
        y, tape, last, n_clips = ctx
        dx, _ = AF.au_logits_bwd(weights, y, last.w, n_clips, want_dx=True, want_dw=False)
        gmaps = self.corr_transformer.relevance_bwd_(dx, tape, n_clips, 12, maps=maps)
        return gmaps, dx

    def forward(self, input):
        AF._cuda(input, "input")
        bs = input.shape[0]
        if needs_grad(self, input):
            return self.logits21_train(input.reshape(bs * 12, -1), bs)[:, :12]
        tok = input.detach().float().reshape(bs * 12, -1).clone()
        return self.logits21_(tok, bs)[:, :12]


tformer_AU_head = former_AU_head     # the name the class carries in models/tformer.py:362


class VA_former(nn.Module):
    """VA_former(input_dim=512, emb_dim=128, dropout=0.0) (models/heads.py:341-372): BatchNorm1d -> 2 x Linear(512,128) -> 2 tokens + pos
    -> Transformer(128, depth 2, 8 x 32, mlp 128) -> 2 x Linear(128,1) -> (VA_out [B,2], tokens [B,2,128]).  One more (N, D, I, M) =
    (2, 128, 256, 128) instantiation of the stack the AU path uses (SURVEY.md section 8f-3); inference kernels only."""

    def __init__(self, input_dim=512, emb_dim=128, dropout=0.0):
        super().__init__()
        self.emb_dim = input_dim
        self.VA_BN1 = nn.BatchNorm1d(input_dim)
        self.VA_linear_p1 = nn.Linear(input_dim, emb_dim)
        self.VA_linear_p2 = nn.Linear(input_dim, emb_dim)
        self.pos_embedding = nn.Parameter(torch.randn(1, 2, emb_dim))
        self.corr_transformer = Transformer(emb_dim, depth=2, heads=8, mlp_dim=128, dim_head=32, dropout=dropout)
        self.VA_linear_last1 = nn.Linear(emb_dim, 1, bias=False)
        self.VA_linear_last2 = nn.Linear(emb_dim, 1, bias=False)
        self._front: Optional[_PackedFront] = None

    def _packed_front(self):
        mode = AF._mode(self.corr_transformer.precision or default_precision())
        if self._front is None or self._front.mode != mode or self._front.stale():
            self._front = _PackedFront([self.VA_linear_p1, self.VA_linear_p2], mode)
        return self._front

    @torch.no_grad()
    def forward(self, emb):
        AF._cuda(emb, "emb")
        if self.training:
            raise RuntimeError("VA_former: only the inference kernels are instantiated for this variant; call .eval()")
        bs = emb.shape[0]
        emb = emb.detach().float().contiguous()
        f = self._packed_front()
        bn = self.VA_BN1
        x = AF.token_front(emb, emb.shape[1], bs, 2, (bn.weight, bn.bias, bn.running_mean, bn.running_var), f.w, f.b, None, f.mode)
        tok = self.corr_transformer.forward_(x, bs, 2, pos=self.pos_embedding[0]).view(bs, 2, -1)
        w = torch.stack([self.VA_linear_last1.weight[0], self.VA_linear_last2.weight[0]]).float()       # [2, emb]
        va_out = (tok * w.unsqueeze(0)).sum(-1)      # two 128-wide dots per clip: output glue, not a kernel of the path
        return va_out, tok
