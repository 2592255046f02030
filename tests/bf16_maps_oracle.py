"""Attention maps of the encoder stack, in fp64 and with the bf16 rounding of the kernel-per-operation path.  TEST INFRASTRUCTURE
ONLY, next to tests/bf16_oracle.py, whose LayerNorm and feed-forward (with their rounding points) it reuses unchanged.

``stack_maps`` is bf16_oracle's stack with an attention that also returns its probabilities: the map value the kernels write,
exp2(s - m) / l with fp32 exp and row sum (avf_attention_mma.cu), taken before P is rounded to bf16 for the P V product.  The
layer output rounds exactly where bf16_oracle._attention's "per_op" path does, so the maps of layer l > 0 see the same rounded
residual stream as the kernel's."""
import math

import torch

import bf16_oracle as B


def _attention_maps(x, p, pre, heads, path, keep=None):
    Bn, N, _ = x.shape
    r = B.bf if path else (lambda t: t)
    wqkv = p[pre + "fn.fn.to_qkv.weight"]
    inner = wqkv.shape[0] // 3
    dh = inner // heads
    qkv = r(x @ r(wqkv).t())
    q, k, v = (t.reshape(Bn, N, heads, dh).permute(0, 2, 1, 3) for t in qkv.split(inner, dim=-1))
    s = torch.matmul(q, k.transpose(-1, -2))
    if keep is not None:                             # kept query: -inf on dropped keys; dropped query: the same score on every key
        s = s.masked_fill(~keep[:, None, None, :], -math.inf).masked_fill(~keep[:, None, :, None], 0.0)
    e = torch.exp2((s - s.amax(dim=-1, keepdim=True)) * (B.LOG2E * dh ** -0.5))
    probs = e / e.sum(dim=-1, keepdim=True)
    o = B.bf(torch.matmul(B.bf(e), v) / e.sum(dim=-1, keepdim=True)) if path else torch.matmul(e, v) / e.sum(dim=-1, keepdim=True)
    o = o.permute(0, 2, 1, 3).reshape(Bn, N, inner)
    return o @ r(p[pre + "fn.fn.to_out.0.weight"]).t() + p[pre + "fn.fn.to_out.0.bias"], probs


def stack_maps(x, p, pre, depth, heads, path=None, keep=None):
    """x [n_seq, n_tok, dim] fp64 -> (y, maps [depth, n_seq, heads, n_tok, n_tok]) in fp64 (path None) or with the rounding of the
    kernel-per-operation bf16 path (path "per_op").  ``keep`` [n_seq, n_tok] bool (True = kept), the mask of mask_score."""
    assert path in (None, "per_op")
    maps = []
    for l in range(depth):
        a, f = f"{pre}layers.{l}.0.", f"{pre}layers.{l}.1."
        y, m = _attention_maps(B._layer_norm(x, p[a + "fn.norm.weight"], p[a + "fn.norm.bias"], path), p, a, heads, path, keep)
        maps.append(m)
        x = x + y
        x = x + B._feed_forward(B._layer_norm(x, p[f + "fn.norm.weight"], p[f + "fn.norm.bias"], path), p, f, path)
    return x, torch.stack(maps)
