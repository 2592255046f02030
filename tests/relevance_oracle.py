"""fp64 references of the attention relevance (include/avformer_b200.h, "attention relevance"; INTEGRATION.md section 1).  TEST
INFRASTRUCTURE ONLY.

- ``gmap``: G = P o dP of one attention, restated (P = softmax of the masked scores, dP = dO V^T) with ``P.retain_grad()`` through
  autograd, so G is P times the gradient autograd gives P, not a second hand-written formula.
- ``oracle_gmaps``: runs any oracle function (oracle/avformer_oracle.py, tests/masked_oracle.py) with every ``torch.softmax`` output
  retained, back-propagates a seed from its result and returns the G of every softmax call in call order.
- ``stack_gmaps``: the gradient maps of tests/bf16_bwd_oracle.py's stack backward, exact (path None) or with bf16 rounding where the
  training path rounds (path "per_op"): G is formed from the same qkv and dob that backward feeds its attention backward.
- ``rollout``: R = prod_l (I + mean_h max(G_l, 0)), the last layer leftmost.
- ``bug``: one deliberate defect in the definition; tests/test_attention_relevance_cpu.py shows that each misses its check."""
import math
from unittest import mock

import torch

import bf16_bwd_oracle as BB

BUGS = ("g_from_unnormalised_e", "g_is_ds", "head_sum", "no_clamp", "r_times_a", "no_identity", "last_layer_cls_row_only")
G_BUGS = BUGS[:2]
R_BUGS = BUGS[2:6]


def gmap(qkv, dout, n_seq, n_tok, heads, dh, keep=None, bug=None):
    """qkv [n_seq*n_tok, 3*heads*dh] (q | k | v, head-major), dout [rows, heads*dh], fp64 -> G [n_seq, heads, n_tok, n_tok].  ``keep``
    [n_seq, n_tok] bool as mask_score: a kept query gets -inf on dropped keys, a dropped query score 0 on every key."""
    inner = heads * dh
    q, k, v = (t.reshape(n_seq, n_tok, heads, dh).permute(0, 2, 1, 3).detach() for t in qkv.split(inner, dim=-1))
    do = dout.reshape(n_seq, n_tok, heads, dh).permute(0, 2, 1, 3).detach()
    with torch.enable_grad():
        s = torch.matmul(q, k.transpose(-1, -2)) * dh ** -0.5
        if keep is not None:
            s = s.masked_fill(~keep[:, None, None, :], -math.inf).masked_fill(~keep[:, None, :, None], 0.0)
        s.requires_grad_(True)
        e = torch.exp(s - s.amax(-1, keepdim=True))
        p = e / e.sum(-1, keepdim=True)
        p.retain_grad()
        o = torch.matmul(p, v)
        o.backward(do)
    if bug == "g_from_unnormalised_e":
        return (e * p.grad).detach()
    if bug == "g_is_ds":
        return s.grad.detach()
    return (p * p.grad).detach()


def oracle_gmaps(fn, seed_fn, *args, **kw):
    """fn(*args, **kw) with every torch.softmax output retained; then seed_fn(result).backward(); returns (result, [G per softmax call])."""
    seen, real = [], torch.softmax

    def record(t, dim):
        out = real(t, dim=dim)
        if out.requires_grad:
            out.retain_grad()
        else:                                                 # nothing upstream requires grad: P becomes the leaf
            out = out.detach().requires_grad_(True)
        seen.append(out)
        return out
    with torch.enable_grad(), mock.patch.object(torch, "softmax", record):
        res = fn(*args, **kw)
        seed_fn(res).backward()
    return res, [(p * p.grad).detach() for p in seen]


def stack_gmaps(x, p, dy, depth, heads, keep=None, path=None):
    """(dx, G [depth, n_seq, heads, n_tok, n_tok]) of bf16_bwd_oracle.stack_bwd (fp64; path "per_op": bf16 rounding as the kernels)."""
    n_seq, n_tok, _ = x.shape
    maps, real = [], BB.attention_bwd

    def record(qkv, dout, n_seq_, n_tok_, heads_, dh, keep_=None, path_=None, bug=None):
        maps.append(gmap(qkv, dout, n_seq_, n_tok_, heads_, dh, keep_))
        return real(qkv, dout, n_seq_, n_tok_, heads_, dh, keep_, path_, bug)
    with mock.patch.object(BB, "attention_bwd", record):
        dx, _ = BB.stack_bwd(x, p, dy, depth, heads, keep=keep, path=path)
    return dx, torch.stack(maps[::-1])                      # the backward visits the layers last to first


def rollout(g, bug=None):
    """g [depth, n_seq, heads, n, n] fp64 -> R [n_seq, n, n]."""
    depth, n_seq, _, n, _ = g.shape
    a = g if bug == "no_clamp" else g.clamp(min=0)
    a = a.sum(2) if bug == "head_sum" else a.mean(2)
    eye = torch.eye(n, dtype=g.dtype, device=g.device).expand(n_seq, n, n)
    r = eye.clone()
    for l in range(depth):
        if bug == "r_times_a":
            r = r + torch.matmul(r, a[l])
        elif bug == "no_identity":
            r = torch.matmul(a[l], r) if l else a[l].clone()
        else:
            r = r + torch.matmul(a[l], r)
    return r


def cls_row_only(g):
    """The last layer's G with only the cls (first) query row kept: what a last layer run on the cls rows alone would give."""
    g = g.clone()
    g[-1, :, :, 1:] = 0.0
    return g


def rollout_bound(g64, r64):
    """Elementwise bound of an fp32 rollout against fp64: every term is non-negative, so each fp32 step (head sum of `heads` terms, an
    N-term dot product, one add) costs at most (heads + N + 3) units of 2^-24 relative to the exact value; over the layers they add
    up.  The test feeds both sides the same fp32 maps, so twice that is the bound the kernel is held to."""
    depth, _, heads, n, _ = g64.shape
    return 2 * depth * (heads + n + 3) * 2.0 ** -24 * r64.abs() + 1e-30
