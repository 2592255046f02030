"""fp64 CPU restatement of the encoder stack WITH the attention mask of Transformer.forward (models/heads.py:225-232).  TEST
INFRASTRUCTURE ONLY, next to oracle/avformer_oracle.py, whose primitives (LayerNorm, feed-forward, the explicit dropout masks) it
reuses unchanged.

The reference's masked branch is dead code on the AVFormer path, so no run of the reference pins it.  What follows is the ViT form
that models/heads.py:164-256 is copied from (scaled dots at :224, mask branch at :225-232 with its shape assert at :229, softmax at
:234), written literally: ``keep`` is the module's ``mask``, bool [B, N-1], True = keep, padded with a kept first (cls) token; score
(i, j) of every head of sequence b is kept iff keep[b, i] and keep[b, j], the others are filled with -finfo.max before the softmax."""
import torch
import torch.nn.functional as F

from oracle import avformer_oracle as O


def attention(x, p, pre: str, heads: int, keep, drop=None):
    """O.attention with the mask (same operations, plus the masked_fill)."""
    B, N, _ = x.shape
    wqkv = p[pre + "fn.fn.to_qkv.weight"]
    inner = wqkv.shape[0] // 3
    dh = inner // heads
    qkv = x @ wqkv.t()
    q, k, v = (t.reshape(B, N, heads, dh).permute(0, 2, 1, 3) for t in qkv.split(inner, dim=-1))
    dots = torch.matmul(q, k.transpose(-1, -2)) * (dh ** -0.5)
    m = F.pad(keep, (1, 0), value=True)
    assert m.shape == (B, N), "mask has incorrect dimensions"
    dots = dots.masked_fill(~(m[:, None, :, None] & m[:, None, None, :]), -torch.finfo(dots.dtype).max)
    attn = torch.softmax(dots, dim=-1)
    out = torch.matmul(attn, v).permute(0, 2, 1, 3).reshape(B, N, inner)
    y = out @ p[pre + "fn.fn.to_out.0.weight"].t() + p[pre + "fn.fn.to_out.0.bias"]
    return y if drop is None else drop(0, y)


def transformer(x, p, pre: str, depth: int, heads: int, keep, masks=None):
    """O.transformer with the attention mask ``keep`` in every layer; ``masks`` are the explicit dropout masks of O.transformer."""
    for l in range(depth):
        drop = None
        if masks is not None:
            drop = (lambda site, t, l=l: t * masks[(l, site)].reshape(t.shape).to(t.dtype))
        a, f = f"{pre}layers.{l}.0.", f"{pre}layers.{l}.1."
        x = x + attention(O.layer_norm(x, p[a + "fn.norm.weight"], p[a + "fn.norm.bias"]), p, a, heads, keep, drop)
        x = x + O.feed_forward(O.layer_norm(x, p[f + "fn.norm.weight"], p[f + "fn.norm.bias"]), p, f, drop)
    return x


def tformer(frames, p, pre: str, n_frames: int, keep):
    """O.tformer with a frames-kept mask ``keep``, bool [B, T] (True = a real frame)."""
    x = frames.reshape(-1, n_frames, frames.shape[-1])
    B = x.shape[0]
    cls = p[pre + "cls_token"].expand(B, -1, -1)
    x = torch.cat([cls, x], dim=1) + p[pre + "pos_embedding"][:, : n_frames + 1]
    x = transformer(x, p, pre + "spatial_transformer.", O.STACKS["tformer"]["depth"], O.STACKS["tformer"]["heads"], keep)
    return x[:, 0]
