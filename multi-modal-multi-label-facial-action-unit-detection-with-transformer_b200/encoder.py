"""Pre-LN ViT encoder stack with the reference's module tree and state-dict names
(models/heads.py:164-256 and its byte-identical copies in vformer.py / tformer.py), executed by the
hand-written sm_100a kernels behind the C ABI.

The module tree exists to own parameters under the reference's names:

    layers.L.0.fn.norm.{weight,bias}      layers.L.0.fn.fn.to_qkv.weight
    layers.L.0.fn.fn.to_out.0.{weight,bias}
    layers.L.1.fn.norm.{weight,bias}      layers.L.1.fn.fn.net.{0,3}.{weight,bias}

``Transformer.forward`` does not walk that tree: it hands the whole stack to
``avf_encoder_stack_fwd``.  The sub-modules keep a working ``forward`` built from the library's
building blocks so that they can be called on their own like the reference's.
"""
from __future__ import annotations

from typing import Optional

import torch
from torch import nn

from . import functional as AF

_DEFAULT_PRECISION = "bf16"


def set_default_precision(precision: str) -> None:
    """'bf16' (tcgen05 tensor cores, fp32 residual/statistics) or 'fp32' (CUDA-core parity mode)."""
    global _DEFAULT_PRECISION
    AF._mode(precision)
    _DEFAULT_PRECISION = precision


def default_precision() -> str:
    return _DEFAULT_PRECISION


def _rank_salt() -> int:
    """0 on rank 0 / without a process group; otherwise a 62-bit hash of the data-parallel rank (murmur-style finaliser)."""
    import torch.distributed as dist
    if not (dist.is_available() and dist.is_initialized()):
        return 0
    h = (dist.get_rank() * 0x9E3779B97F4A7C15) & 0xFFFFFFFFFFFFFFFF
    h ^= h >> 31
    h = (h * 0xBF58476D1CE4E5B9) & 0xFFFFFFFFFFFFFFFF
    h ^= h >> 29
    return h & ((1 << 62) - 1)


def needs_grad(module: nn.Module, *inputs: torch.Tensor) -> bool:
    """True when autograd has to see this call: grad mode on and an input or a parameter of ``module`` requires grad.
    Such calls take the tape-keeping path (autograd.py); everything else takes the inference kernels."""
    if not torch.is_grad_enabled():
        return False
    return any(t is not None and t.requires_grad for t in inputs) or any(p.requires_grad for p in module.parameters())


class GELU(nn.Module):
    """tanh-GELU (models/heads.py:164-166); fused into the MLP1 epilogue when run through Transformer."""

    def forward(self, x):
        raise RuntimeError("GELU is fused into FeedForward's first linear; call FeedForward or Transformer")


class Residual(nn.Module):
    def __init__(self, fn):
        super().__init__()
        self.fn = fn

    def forward(self, x, **kw):
        return self.fn(x, **kw) + x


class PreNorm(nn.Module):
    def __init__(self, dim, fn):
        super().__init__()
        self.norm = nn.LayerNorm(dim)
        self.fn = fn

    def forward(self, x, **kw):
        prec = default_precision()
        y = AF.layernorm_fwd(x, self.norm.weight, self.norm.bias, prec)
        return self.fn(y.view(x.shape), **kw)


class FeedForward(nn.Module):
    def __init__(self, dim, hidden_dim, dropout=0.0):
        super().__init__()
        self.net = nn.Sequential(nn.Linear(dim, hidden_dim), GELU(), nn.Dropout(dropout), nn.Linear(hidden_dim, dim), nn.Dropout(dropout))

    def forward(self, x):
        prec = default_precision()
        cast = AF.to_bf16 if prec == "bf16" else (lambda t: t.detach().float())
        a = x.reshape(-1, x.shape[-1])
        a = a if a.dtype == (torch.bfloat16 if prec == "bf16" else torch.float32) else cast(a)
        h = AF.linear_fwd(a, cast(self.net[0].weight), self.net[0].bias, gelu=True, out_dtype=a.dtype, precision=prec)
        y = AF.linear_fwd(h, cast(self.net[3].weight), self.net[3].bias, out_dtype=torch.float32, precision=prec)
        return y.view(*x.shape[:-1], -1)


class Attention(nn.Module):
    def __init__(self, dim, heads=8, dim_head=64, dropout=0.0):
        super().__init__()
        inner = dim_head * heads
        self.heads, self.dim_head = heads, dim_head
        self.scale = dim_head ** -0.5
        self.to_qkv = nn.Linear(dim, inner * 3, bias=False)
        project_out = not (heads == 1 and dim_head == dim)
        self.to_out = nn.Sequential(nn.Linear(inner, dim), nn.Dropout(dropout)) if project_out else nn.Identity()

    def forward(self, x, mask=None):
        """x [b, n, dim]; ``mask`` (optional) bool [b, n - 1], True = keep: see Transformer.forward."""
        prec = default_precision()
        cast = AF.to_bf16 if prec == "bf16" else (lambda t: t.detach().float())
        b, n, _ = x.shape
        keep = None if mask is None else AF.keep_from_mask(mask, b, n)
        a = x.reshape(b * n, -1)
        a = a if a.dtype == (torch.bfloat16 if prec == "bf16" else torch.float32) else cast(a)
        qkv = AF.linear_fwd(a, cast(self.to_qkv.weight), out_dtype=a.dtype, precision=prec)
        o = AF.attention_fwd(qkv, b, n, self.heads, self.dim_head, keep)
        if isinstance(self.to_out, nn.Identity):
            return AF.to_f32(o).view(b, n, -1) if o.dtype != torch.float32 else o.view(b, n, -1)
        y = AF.linear_fwd(o, cast(self.to_out[0].weight), self.to_out[0].bias, out_dtype=torch.float32, precision=prec)
        return y.view(b, n, -1)


class Transformer(nn.Module):
    """Transformer(dim, depth, heads, dim_head, mlp_dim, dropout=0.) — models/heads.py:242-256."""

    def __init__(self, dim, depth, heads, dim_head, mlp_dim, dropout=0.0):
        super().__init__()
        self.dim, self.depth, self.heads, self.dim_head, self.mlp_dim, self.dropout = dim, depth, heads, dim_head, mlp_dim, dropout
        self.layers = nn.ModuleList([
            nn.ModuleList([Residual(PreNorm(dim, Attention(dim, heads=heads, dim_head=dim_head, dropout=dropout))),
                           Residual(PreNorm(dim, FeedForward(dim, mlp_dim, dropout=dropout)))])
            for _ in range(depth)])
        self.precision: Optional[str] = None       # None -> default_precision()
        self.fixed_dropout_seed: Optional[int] = None
        self.dropout_salt: Optional[torch.Tensor] = None
        self._packed: Optional[AF.PackedStack] = None

    # -- weights -------------------------------------------------------------------------------
    def _layer_tensors(self):
        for attn, ff in self.layers:
            a, f = attn.fn, ff.fn
            yield dict(ln1_gamma=a.norm.weight, ln1_beta=a.norm.bias, w_qkv=a.fn.to_qkv.weight,
                       w_out=a.fn.to_out[0].weight, b_out=a.fn.to_out[0].bias,
                       ln2_gamma=f.norm.weight, ln2_beta=f.norm.bias,
                       w_ff1=f.fn.net[0].weight, b_ff1=f.fn.net[0].bias, w_ff2=f.fn.net[3].weight, b_ff2=f.fn.net[3].bias)

    def packed(self) -> AF.PackedStack:
        mode = AF._mode(self.precision or default_precision())
        p = self._packed
        if p is None or p.mode != mode or p.stale():
            p = self._packed = AF.PackedStack(list(self._layer_tensors()), mode)
        return p

    def shape(self, n_seq: int, n_tok: int):
        return AF.make_shape(n_seq, n_tok, self.dim, self.heads, self.dim_head, self.mlp_dim, self.depth)

    def param_list(self):
        """Parameters in avf_layer_weights order, layer by layer (the order autograd.EncoderStackFn returns gradients in)."""
        names = [n for n, _ in AF.LayerWeights._fields_]
        return [lw[n] for lw in self._layer_tensors() for n in names]

    def dropout_state(self):
        """(p, seed, salt) of the next training forward: p = 0 in eval(); the seed is drawn from torch's default generator so
        that torch.manual_seed makes runs reproducible.  ``fixed_dropout_seed`` (tests) pins it.  ``dropout_salt`` is an optional
        one-element int32 CUDA tensor hashed into the seed on the device: graphs.GraphedTrainStep bumps it between replays."""
        if not self.training or self.dropout <= 0.0:
            return 0.0, 0, None
        seed = self.fixed_dropout_seed
        if seed is None:
            seed = int(torch.randint(0, 2 ** 62, (1,)).item())
            # Data parallel: every rank seeds torch identically (runner.py / train.py call manual_seed(seed) everywhere), so the draw
            # above is the same on all ranks.  Mix the rank in, or all shards of the global batch would share their dropout masks
            # (DDP and the single-GPU reference draw them independently per sample).
            seed ^= _rank_salt()
        return float(self.dropout), seed, self.dropout_salt

    # -- forward -------------------------------------------------------------------------------
    def forward_(self, x2d: torch.Tensor, n_seq: int, n_tok: int, out: Optional[torch.Tensor] = None, ld_out: int = 0,
                 pos: Optional[torch.Tensor] = None, keep: Optional[torch.Tensor] = None) -> torch.Tensor:
        """Inference kernels, in place on an fp32 residual stream [n_seq*n_tok, dim] (+ pos [n_tok, dim] first, if given).  In
        train() mode with dropout > 0 (a frozen sub-model inside a training loop, models/avformer.py:78-85 + train.py:327) the
        tape-keeping kernels run instead, because they are the ones that apply dropout.  ``keep`` [n_seq, n_tok] bool: attention
        mask of every layer (AF.keep_from_mask); a masked stack runs kernel by kernel, never as the fused kernel."""
        p, seed, salt = self.dropout_state()
        if p > 0.0:
            if pos is not None:
                AF.add_row_periodic_(x2d, pos, n_tok)
            y, _ = AF.encoder_stack_fwd_train(x2d, self.packed(), self.shape(n_seq, n_tok), p, seed, salt, keep=keep)
            if out is None:
                x2d.copy_(y)
                return x2d
            torch.as_strided(out, (y.shape[0], y.shape[1]), (ld_out, 1)).copy_(y)
            return out
        if keep is None:
            return AF.token_stack_fwd_(x2d, self.packed(), self.shape(n_seq, n_tok), pos, out, ld_out)
        if pos is not None:
            AF.add_row_periodic_(x2d, pos, n_tok)
        return AF.encoder_stack_fwd_(x2d, self.packed(), self.shape(n_seq, n_tok), out, ld_out, keep=keep)

    def forward_train(self, x2d: torch.Tensor, n_seq: int, n_tok: int, keep: Optional[torch.Tensor] = None) -> torch.Tensor:
        """Autograd-visible forward on an fp32 token matrix [n_seq*n_tok, dim] (activation tape kept for backward)."""
        from .autograd import EncoderStackFn
        return EncoderStackFn.apply(x2d, self, n_seq, n_tok, keep, *self.param_list())

    def forward(self, x: torch.Tensor, mask=None) -> torch.Tensor:
        """x [b, n, dim].  ``mask`` (optional): bool [b, n - 1] on x's device, True = keep; the first (cls) token is always kept.  Score
        (i, j) of every head of sequence b survives iff tokens i and j are both kept, in every layer: a kept token attends only to
        kept tokens, a dropped token attends uniformly to all n tokens (models/heads.py:225-234 in its ViT form).  Any other mask
        shape raises NotImplementedError, a non-bool mask TypeError, a mask off the input's CUDA device RuntimeError."""
        AF._cuda(x, "x")
        b, n, d = x.shape
        keep = None if mask is None else AF.keep_from_mask(mask, b, n)
        if needs_grad(self, x):
            return self.forward_train(x.reshape(b * n, d), b, n, keep).view(b, n, d)
        y = x.detach().float().reshape(b * n, d).clone()
        return self.forward_(y, b, n, keep=keep).view(b, n, d)

    # -- attention maps ------------------------------------------------------------------------
    def check_maps_allowed(self, who: str, *inputs: torch.Tensor) -> None:
        """Attention maps come from the inference kernels only: refuse a call autograd would record or one that would apply dropout."""
        if needs_grad(self, *inputs):
            raise RuntimeError(f"{who}: attention maps are inference only, and this call would be recorded by autograd; run it under "
                               f"torch.no_grad() (or with parameters and inputs that do not require grad)")
        if self.training and self.dropout > 0.0:
            raise RuntimeError(f"{who}: attention maps are inference only, and this stack applies dropout (train() with dropout "
                               f"{self.dropout}); call eval() first")

    def maps_(self, x2d: torch.Tensor, n_seq: int, n_tok: int, out: Optional[torch.Tensor] = None, ld_out: int = 0,
              pos: Optional[torch.Tensor] = None, keep: Optional[torch.Tensor] = None) -> torch.Tensor:
        """forward_ kernel by kernel (never the fused kernel) with the attention maps of every layer written by the attention launches:
        returns fp32 [depth, n_seq, heads, n_tok, n_tok]; x2d / out receive what forward_ writes with set_fused_enabled(False)."""
        return AF.encoder_stack_probs_(x2d, self.packed(), self.shape(n_seq, n_tok), keep, pos, out, ld_out)

    def attention_maps(self, x: torch.Tensor, mask=None):
        """(y, maps): y is ``forward(x, mask)`` as computed with set_fused_enabled(False), bit for bit, and maps fp32 [depth, b, heads, n,
        n] holds the softmax probabilities of every layer (p = exp(s - m) / l, the kernel's own values; INTEGRATION.md section 1).
        Inference only: RuntimeError under autograd or in train() with dropout > 0."""
        AF._cuda(x, "x")
        self.check_maps_allowed("Transformer.attention_maps", x)
        b, n, d = x.shape
        keep = None if mask is None else AF.keep_from_mask(mask, b, n)
        y = x.detach().float().reshape(b * n, d).clone()
        maps = self.maps_(y, b, n, keep=keep)
        return y.view(b, n, d), maps

    # -- attention relevance -------------------------------------------------------------------
    def check_relevance_allowed(self, who: str) -> None:
        """Relevance differentiates the eval() computation: refuse a stack in train() (dropout, and batch statistics in the model)."""
        if self.training:
            raise RuntimeError(f"{who}: attention relevance needs eval(); in train() dropout and BatchNorm batch statistics would couple "
                               f"the clips of a batch and BatchNorm would update its running statistics; call eval() first")

    def relevance_fwd_(self, x2d: torch.Tensor, n_seq: int, n_tok: int, keep: Optional[torch.Tensor] = None):
        """The tape-keeping forward without dropout of an fp32 token matrix [n_seq*n_tok, dim] (left untouched): (y, tape), y bit-equal
        to forward_train's."""
        return AF.encoder_stack_fwd_train(x2d, self.packed(), self.shape(n_seq, n_tok), keep=keep)

    def relevance_bwd_(self, d2d: torch.Tensor, tape: torch.Tensor, n_seq: int, n_tok: int, keep: Optional[torch.Tensor] = None,
                       maps: bool = True) -> Optional[torch.Tensor]:
        """Backward of relevance_fwd_ for the activations only, in place on d2d (dL/dy in, dL/dx out; no parameter gradient).  Returns
        the gradient maps fp32 [depth, n_seq, heads, n_tok, n_tok] (maps=True) or None."""
        shape = self.shape(n_seq, n_tok)
        if maps:
            return AF.encoder_stack_bwd_gradmaps_(d2d, self.packed(), shape, tape, keep)
        AF.encoder_stack_bwd_(d2d, self.packed(), shape, tape, [False] * (len(AF.LayerWeights._fields_) * self.depth), keep=keep)
        return None

    def attention_relevance(self, x: torch.Tensor, dy: torch.Tensor, mask=None):
        """(y, gmaps, R) for the target whose gradient wrt the output is ``dy`` [b, n, dim]: y is the tape-keeping forward's output
        (forward_train's, bit for bit), gmaps fp32 [depth, b, heads, n, n] the gradient maps G = P o dP of every layer from the
        attention backward kernels, and R fp32 [b, n, n] their rollout R = prod_l (I + mean_h max(G_l, 0)) (INTEGRATION.md section 1).
        No parameter gradient is computed or changed.  RuntimeError in train()."""
        AF._cuda(x, "x")
        AF._cuda(dy, "dy")
        self.check_relevance_allowed("Transformer.attention_relevance")
        b, n, d = x.shape
        if tuple(dy.shape) != (b, n, d):
            raise ValueError(f"Transformer.attention_relevance: dy must have the shape of x {(b, n, d)}, got {tuple(dy.shape)}")
        keep = None if mask is None else AF.keep_from_mask(mask, b, n)
        with torch.no_grad():
            y, tape = self.relevance_fwd_(x.detach().float().reshape(b * n, d).contiguous(), b, n, keep)
            dx = dy.detach().reshape(b * n, d).to(torch.float32, copy=True, memory_format=torch.contiguous_format)
            gmaps = self.relevance_bwd_(dx, tape, b, n, keep)
            return y.view(b, n, d), gmaps, AF.attention_rollout(gmaps)
