"""bf16 error budgets for the training backward: the attention backward kernel and the encoder-stack gradients.  TEST
INFRASTRUCTURE ONLY, next to tests/bf16_oracle.py, whose rounding helper, per-op forward emulation and parameter draw it reuses.

A bf16 gradient differs from the fp64 gradient by its rounding.  A bound on a whole tensor's max-abs admits one missing query,
key or row at 33-64 tokens (each changes its elements by about 1 / n_tok).  Instead, every case gets its own budget: the same
backward in fp64 with bf16 rounding where the training path rounds (``path="per_op"``).  Errors are taken per unit, as RMS
against fp64: one token row of dx, one row of a weight gradient, one (token row, Q/K/V section, head) slice of the attention
backward's dqkv, the whole vector of a LayerNorm vector or bias gradient.  A case passes when the kernel's worst unit is within
``K_BWD`` times the emulation's worst unit (``unit_floor``: at least 1e-6 of the reference's RMS, since the top layer's db_ff2 is an
fp32 column sum of fp32 data and its emulated error is 0) and, for rows and slices, the median unit within [0.5, 2] times the
emulation's median.  ``bug`` is one deliberate backward bug in the fp64 computation; tests/test_bf16_bwd_budget_sensitivity.py
shows that each lands well outside every applicable case's budget.

Input choices that make the bugs show above bf16 noise: make_params keeps bf16_oracle's doubled Wq / Wk (peaked softmax rows, so
one query or key carries weight), and the incoming gradient dy has a per-row common offset (``make_dy``), so the mean term of the
LayerNorm backward and the row sums of dP matter.  Out of reach by nature, below bf16 rounding: a backward that takes gelu' of the
fp32 pre-activation instead of its bf16 copy (the bf16 tape is what the kernel has), and fp32 instead of fp64 statistics in the
LayerNorm backward (both far below the 2^-9 of one bf16 rounding).

Accumulation order is not modelled: fp32 sums of products of bf16 values sit far below bf16 rounding at these lengths.  The split-K
wgrad (K up to 50176 token rows) is checked against this at its own size."""
import math

import numpy as np
import torch

import bf16_oracle as B

# A case passes when worst_unit(kernel) <= K_BWD * worst_unit(emulation).  K_BWD = 1.5 x the largest kernel / emulation ratio over
# every case and tensor of tests/test_gpu_bf16_bwd_budget.py, measured on one B200 (1000 W limit, 1965 MHz max SM clock): 1.366
# (fusion-head, layer 0 w_qkv); median-unit ratios 0.94-1.06 (profiles/r08_bf16_bwd_budget_ratios.json).
K_BWD = 2.05
MEDIAN_RATIO = (0.5, 2.0)

NAMES = ("ln1_gamma", "ln1_beta", "w_qkv", "w_out", "b_out", "ln2_gamma", "ln2_beta", "w_ff1", "b_ff1", "w_ff2", "b_ff2")  # avf_layer_weights
KEYS = ("0.fn.norm.weight", "0.fn.norm.bias", "0.fn.fn.to_qkv.weight", "0.fn.fn.to_out.0.weight", "0.fn.fn.to_out.0.bias", "1.fn.norm.weight",
        "1.fn.norm.bias", "1.fn.fn.net.0.weight", "1.fn.fn.net.0.bias", "1.fn.fn.net.3.weight", "1.fn.fn.net.3.bias")
MATRICES = ("w_qkv", "w_out", "w_ff1", "w_ff2")

MUTANTS = ("dv_dk_skip_last_query", "delta_skip_last_key", "dq_skip_last_key", "masked_dropped_query_ds_kept", "ln_bwd_mean_term_dropped",
           "ln1_bwd_uses_ln2_gamma", "dx_last_row_not_written", "wgrad_skips_last_kblock", "colsum_skips_last_rows")
ATTENTION_MUTANTS = MUTANTS[:4]

BK = 64                      # avf_gemm_umma.cu:34: K block of the wgrad GEMM
SMS = B.SMS


# ---------------------------------------------------------------------------------------------------------------------------------
# attention backward (attention_bwd_mma_kernel, avf_attention_mma.cu:245-466)
# ---------------------------------------------------------------------------------------------------------------------------------
def attention_bwd(qkv, dout, n_seq, n_tok, heads, dh, keep=None, path=None, bug=None):
    """qkv [n_seq * n_tok, 3 * heads * dh] (columns q | k | v, head-major), dout [rows, heads * dh] -> dqkv like qkv, in fp64.
    ``keep`` [n_seq, n_tok] bool: the forward's mask (mask_score, avf_attention_mma.cu:48-52).  path="per_op" rounds like the kernel:
    S, P, dP and delta in fp32 from the bf16 operands (:354-407, not modelled), dS rounded to bf16 as an MMA operand and the
    1/sqrt(dh) applied to the fp32 product before the bf16 store: dQ = bf(scale bf(dS) K) (:409-419), dV = bf(bf(P)^T dO) (:461-462),
    dK = bf(scale bf(dS)^T Q) (:463-464)."""
    r = B.bf if path else (lambda t: t)
    inner = heads * dh
    q, k, v = (t.reshape(n_seq, n_tok, heads, dh).permute(0, 2, 1, 3) for t in qkv.split(inner, dim=-1))
    do = dout.reshape(n_seq, n_tok, heads, dh).permute(0, 2, 1, 3)
    scale = dh ** -0.5
    s = torch.matmul(q, k.transpose(-1, -2))
    if keep is not None:          # kept query: -inf on dropped keys (P = 0); dropped query: score 0 on every key (uniform P)
        s = s.masked_fill(~keep[:, None, None, :], -math.inf).masked_fill(~keep[:, None, :, None], 0.0)
    p = torch.softmax(s * scale, dim=-1)
    dp = torch.matmul(do, v.transpose(-1, -2))
    pdp = p * dp
    delta = (pdp[..., :-1] if bug == "delta_skip_last_key" else pdp).sum(dim=-1, keepdim=True)
    ds = p * (dp - delta)
    if keep is not None and bug != "masked_dropped_query_ds_kept":
        ds = ds * keep[:, None, :, None]               # every score of a dropped query was filled: dS = 0 (:412-415)
    if bug == "dq_skip_last_key":
        dq = r(scale * torch.matmul(r(ds[..., :-1]), k[..., :-1, :]))
    else:
        dq = r(scale * torch.matmul(r(ds), k))
    p2, ds2 = p, ds
    if bug == "dv_dk_skip_last_query":                 # pass 2 leaves the last query out of dV and dK
        p2, ds2 = p.clone(), ds.clone()
        p2[..., -1, :] = 0.0
        ds2[..., -1, :] = 0.0
    dv = r(torch.matmul(r(p2).transpose(-1, -2), do))
    dk = r(scale * torch.matmul(r(ds2).transpose(-1, -2), q))
    return torch.cat([t.permute(0, 2, 1, 3).reshape(n_seq * n_tok, inner) for t in (dq, dk, dv)], dim=-1)


# ---------------------------------------------------------------------------------------------------------------------------------
# encoder stack: forward with tape, hand-written backward (encoder_fwd_train / encoder_bwd, avf_train_api.cu:90-124, :162-215)
# ---------------------------------------------------------------------------------------------------------------------------------
def _ln_stats(x):
    mu = x.mean(dim=-1, keepdim=True)
    rstd = 1.0 / torch.sqrt(((x - mu) ** 2).mean(dim=-1, keepdim=True) + 1e-5)
    return (x - mu) * rstd, rstd


def _ln_bwd(x, gamma, dxn, dres, mean_term=True):
    """layernorm_bwd_kernel (avf_train.cu:143-248), fp32 there, fp64 here: dres + rstd (g - mean(g) - xhat mean(g xhat)), g = dxn gamma
    (:191-211); column sums of dxn xhat (dgamma), dxn (dbeta) and the incoming dres (the bias of the sub-layer's last linear)."""
    xhat, rstd = _ln_stats(x)
    g = dxn * gamma
    m1 = g.mean(dim=-1, keepdim=True) if mean_term else 0.0
    m2 = (g * xhat).mean(dim=-1, keepdim=True)
    dim = x.shape[-1]
    flat = (lambda t: t.reshape(-1, dim))
    return dres + rstd * (g - m1 - xhat * m2), flat(dxn * xhat).sum(0), flat(dxn).sum(0), flat(dres).sum(0)


def stack_bwd(x, p, dy, depth, heads, keep=None, path=None, bug=None):
    """x [n_seq, n_tok, dim] fp64 (the stack's fp32 input), p fp64 parameters (keys of A.Transformer.state_dict()), dy like x
    -> (dx, [11 * depth gradients in avf_layer_weights order]).  path=None is exact fp64; path="per_op" rounds to bf16 where the
    training path rounds:
      tape: xn1 = bf(LN1(x_in)) (avf_rowops.cu:46-54), qkv = bf(xn1 bf(Wqkv)^T) (avf_train_api.cu:110), o = bf(attention)
            (avf_attention_mma.cu:205), xn2 = bf(LN2(x_mid)), hpre = bf(h) (SAVE_PRE, avf_gemm_umma.cu:113-124), g = bf(gelu(h)) (:125-127);
            the residual streams x_in, x_mid are fp32 (not rounded here); GEMM weights are the bf16 packed copies;
      backward: dyb = bf(dy) (masked_copy, avf_train_api.cu:184); dh = bf((dyb W2) o gelu'(hpre)) (DGELU epilogue,
            avf_gemm_umma.cu:93-105); db_ff1 = column sum of bf16 dh (avf_train_api.cu:199); dxn = dh W1 in fp32 (:200); the LayerNorm
            backward in fp32, its bf16 copy of the new stream the next dyb (:201, avf_train.cu:213-227); dob = bf(dyb Wout) (:206);
            dqkv from attention_bwd (:207); dxn = dqkv Wqkv in fp32 (:209); every wgrad an fp32 sum of bf16 operands (:194-208)."""
    r = B.bf if path else (lambda t: t)
    n_seq, n_tok, dim = x.shape
    rows = n_seq * n_tok
    flat = (lambda t: t.reshape(rows, -1))
    tapes = []
    for l in range(depth):                                   # forward with tape (bf16_oracle's per-op emulation)
        a, f = f"layers.{l}.0.", f"layers.{l}.1."
        t = {"x_in": x}
        t["xn1"] = B._layer_norm(x, p[a + "fn.norm.weight"], p[a + "fn.norm.bias"], path)
        x = x + B._attention(t["xn1"], p, a, heads, path, None, keep=keep, tape=t)
        t["x_mid"] = x
        t["xn2"] = B._layer_norm(x, p[f + "fn.norm.weight"], p[f + "fn.norm.bias"], path)
        x = x + B._feed_forward(t["xn2"], p, f, path, tape=t)
        tapes.append(t)

    def wgrad(da, b):                                        # dW = da^T b over the token rows (K = rows)
        da, b = flat(da), flat(b)
        if bug == "wgrad_skips_last_kblock":
            keep_rows = (rows - 1) // BK * BK
            da, b = da[:keep_rows], b[:keep_rows]
        return da.t() @ b

    grads = [None] * (11 * depth)
    dx = dy
    dyb = r(dy)
    inner = p["layers.0.0.fn.fn.to_qkv.weight"].shape[0] // 3
    for l in reversed(range(depth)):
        t = tapes[l]
        a, f = f"layers.{l}.0.", f"layers.{l}.1."
        W = {n: p[f"layers.{l}.{k}"] for n, k in zip(NAMES, KEYS)}
        G = {}
        # MLP sub-layer
        G["w_ff2"] = wgrad(dyb, t["g"])
        hb = r(t["h"])
        hv = hb.detach().requires_grad_(True)                # gelu' of the (bf16) pre-activation
        with torch.enable_grad():
            gd, = torch.autograd.grad(B.O.gelu_tanh(hv).sum(), hv)
        dh = r(torch.matmul(dyb, r(W["w_ff2"])) * gd)
        G["w_ff1"] = wgrad(dh, t["xn2"])
        dhr = flat(dh)
        G["b_ff1"] = (dhr[:max(rows - 32, 0)] if bug == "colsum_skips_last_rows" else dhr).sum(0)
        dxn = torch.matmul(dh, r(W["w_ff1"]))
        mean_term = bug != "ln_bwd_mean_term_dropped"
        dx, G["ln2_gamma"], G["ln2_beta"], G["b_ff2"] = _ln_bwd(t["x_mid"], W["ln2_gamma"], dxn, dx, mean_term)
        dyb = r(dx)
        # attention sub-layer
        G["w_out"] = wgrad(dyb, t["o"])
        dob = r(torch.matmul(dyb, r(W["w_out"])))
        dqkv = attention_bwd(flat(t["qkv"]), flat(dob), n_seq, n_tok, heads, inner // heads, keep, path,
                             bug if bug in ATTENTION_MUTANTS else None).reshape(n_seq, n_tok, -1)
        G["w_qkv"] = wgrad(dqkv, t["xn1"])
        dxn = torch.matmul(dqkv, r(W["w_qkv"]))
        gamma1 = W["ln2_gamma"] if bug == "ln1_bwd_uses_ln2_gamma" else W["ln1_gamma"]
        dx, G["ln1_gamma"], G["ln1_beta"], G["b_out"] = _ln_bwd(t["x_in"], gamma1, dxn, dx, mean_term)
        dyb = r(dx)
        grads[11 * l:11 * (l + 1)] = [G[n] for n in NAMES]
    if bug == "dx_last_row_not_written":                     # the last token row keeps the incoming gradient
        dx = dx.clone()
        dx[-1, -1] = dy[-1, -1]
    return dx, grads


def mutant_applies(kind, case):
    """Bugs that are no bugs at a shape: one token has no other key to skip (and dS = 0 there), only a masked case has dropped
    queries, a stack-level bug needs a stack."""
    n_tok, stack = case["n_tok"], case["kind"] == "stack"
    if kind in ("delta_skip_last_key", "dq_skip_last_key"):
        return n_tok >= 2
    if kind == "masked_dropped_query_ds_kept":
        return case["masked"] and n_tok >= 2
    if kind in ATTENTION_MUTANTS:
        return True
    return stack


# ---------------------------------------------------------------------------------------------------------------------------------
# error units and budgets
# ---------------------------------------------------------------------------------------------------------------------------------
def units(name, t, heads=None):
    """Per-unit RMS of an error (or reference) tensor: dx -> token rows; dqkv -> (row, section, head) slices; matrices -> rows;
    vectors -> one unit."""
    t = t.double()
    if name == "dqkv":
        return t.reshape(t.shape[0], 3 * heads, -1).pow(2).mean(-1).sqrt().reshape(-1)
    if name == "dx" or name.split(".")[-1] in MATRICES:
        return t.reshape(-1, t.shape[-1]).pow(2).mean(-1).sqrt()
    return t.pow(2).mean().sqrt().reshape(1)


def unit_floor(ref):
    return 1e-6 * ref.double().pow(2).mean().sqrt().item()


def ratios(name, got, emu, ref, heads=None):
    """(worst-unit ratio, median-unit ratio or None) of ``got`` against the emulation's budget, both as RMS error per unit against
    fp64.  The median is taken over the units the emulation rounds (non-zero error); vectors have no median."""
    eg, ee = units(name, got - ref, heads), units(name, emu - ref, heads)
    worst = eg.max().item() / max(ee.max().item(), unit_floor(ref))
    if eg.numel() == 1:
        return worst, None
    nz = ee > 0
    if not bool(nz.any()):
        return worst, None
    return worst, (eg[nz].median() / ee[nz].median()).item()


def grad_names(depth):
    return [f"{l}.{n}" for l in range(depth) for n in NAMES]


# ---------------------------------------------------------------------------------------------------------------------------------
# the cases of tests/test_gpu_bf16_bwd_budget.py (shared with the sensitivity test)
# ---------------------------------------------------------------------------------------------------------------------------------
ATT_NTOK = (1, 2, 15, 16, 17, 31, 32, 33, 47, 48, 49, 63, 64)


def _att_cases():
    cases = []
    for masked in (False, True):
        for dh in (32, 64):
            for n_tok in ATT_NTOK:
                cases.append(dict(name=f"att-{'m' if masked else 'u'}-dh{dh}-t{n_tok}", kind="att", dh=dh, heads=8, n_tok=n_tok, n_seq=24,
                                  masked=masked))
            # an odd number of (sequence, head) problems: the second warp of the last 2-warp CTA idles (BwdCfg, :236-241)
            for n_tok in ((1, 17, 33, 64) if dh == 32 else (9, 31)):
                cases.append(dict(name=f"att-{'m' if masked else 'u'}-dh{dh}-t{n_tok}-h3", kind="att", dh=dh, heads=3, n_tok=n_tok, n_seq=25,
                                  masked=masked))
    return cases


def splitk_plan(m, n, k, sms):
    """(splits, K blocks of the last split, K blocks per split) of the wgrad C[m, n] = A^T B over K = k rows: avf_gemm_umma.cu:542-546."""
    bn = 128 if n % 128 == 0 else 64
    mn_tiles = -(-m // 128) * (n // bn)
    kblocks = -(-k // BK)
    splits = max(1, min(kblocks, sms // max(1, mn_tiles)))
    per = -(-kblocks // splits)
    splits = -(-kblocks // per)
    return splits, kblocks - (splits - 1) * per, per


def wgrad_shapes(case):
    d, i, m = case["dim"], 8 * case["dh"], case["mlp"]
    return ((d, m), (m, d), (d, i), (3 * i, d))          # w_ff2, w_ff1, w_out, w_qkv  (avf_train_api.cu:194,198,205,208)


def _first_n_seq(case, n_seq0, want):
    n = n_seq0
    while not all(want(*splitk_plan(mm, nn, n * case["n_tok"], SMS)) for mm, nn in wgrad_shapes(case)):
        n += 1
    return n


def _stack(name, dim, dh, depth, mlp, n_tok, n_seq, masked=False, splitk=None):
    return dict(name=name, kind="stack", dim=dim, dh=dh, depth=depth, mlp=mlp, n_tok=n_tok, n_seq=n_seq, masked=masked, splitk=splitk)


def _stack_cases():
    cases = [
        # every module of the training step (video.py:60,133, heads.py:54,118)
        _stack("sformer", 256, 32, 1, 512, 49, 24),
        _stack("tformer", 512, 64, 3, 1024, 17, 24),
        _stack("tformer-masked", 512, 64, 3, 1024, 17, 24, masked=True),
        _stack("au-former", 128, 32, 2, 256, 12, 24),
        _stack("fusion-head", 128, 32, 3, 256, 12, 24),
        # dim 384: LayerNorm backward VEC = 3
        _stack("d384-t20", 384, 32, 2, 384, 20, 24),
    ]
    for i, n_tok in enumerate((1, 2, 16, 33, 64)):
        cases.append(_stack(f"d256-t{n_tok}", 256, 32, 1 + i % 2, (256, 512)[i % 2], n_tok, 24))
    for i, n_tok in enumerate((1, 9, 48, 64)):
        cases.append(_stack(f"d512-t{n_tok}", 512, 64, 1 + i % 2, 1024, n_tok, 24 if n_tok > 1 else 40))
    # split-K: every wgrad in one K block (splits = 1), and every wgrad with a last split shorter than the others
    one = _stack("splitk1-d256-t12", 256, 32, 2, 512, 12, 5, splitk="one")
    cases.append(one)
    short = _stack("splitk-short-d128-t12", 128, 32, 2, 256, 12, 0, splitk="short")
    short["n_seq"] = _first_n_seq(short, 300, lambda s, last, per: s > 1 and last < per)
    cases.append(short)
    # the benchmarked training step's SFormer: 64 clips x 16 frames = 1024 sequences of 49 tokens (bench.py --mode train); every one
    # of the 50176 rows of dx and every weight gradient are compared
    cases.append(_stack("sformer-bench-1024x49", 256, 32, 1, 512, 49, 1024))
    return cases


ATT_CASES = _att_cases()
STACK_CASES = _stack_cases()


def _seed(case):
    return int(np.frombuffer(case["name"].encode(), dtype=np.uint8).astype(np.int64).sum()) * 7919 + case["n_tok"]


def make_keep(n_seq, n_tok, g):
    """Keep masks with sequence 0 fully dropped, sequence 1 keeping only its first token, the rest kept with probability 0.7."""
    keep = torch.rand(n_seq, n_tok, generator=g) < 0.7
    keep[0] = False
    keep[1] = False
    keep[1, 0] = True
    return keep


def make_dy(rows, dim, g):
    """The incoming gradient: 0.5 randn plus a per-row common offset of randn (the LayerNorm backward's mean term and the
    row sums of dP then matter)."""
    return 0.5 * torch.randn(rows, dim, generator=g) + torch.randn(rows, 1, generator=g)


def att_inputs(case):
    """(qkv bf16 [rows, 3I], dout bf16 [rows, I], keep bool | None).  Q and K are 2 randn (scores peaked like doubled Wq / Wk), dout
    carries a per-row offset like make_dy."""
    g = torch.Generator().manual_seed(_seed(case))
    n_seq, n_tok, inner = case["n_seq"], case["n_tok"], case["heads"] * case["dh"]
    rows = n_seq * n_tok
    qkv = torch.randn(rows, 3 * inner, generator=g)
    qkv[:, :2 * inner] *= 2.0
    dout = make_dy(rows, inner, g)
    keep = make_keep(n_seq, n_tok, g) if case["masked"] else None
    return qkv.bfloat16(), dout.bfloat16(), keep


def stack_inputs(case):
    """(params fp32, x fp32 [rows, dim], dy fp32 [rows, dim], keep bool | None).  Parameters as bf16_oracle.make_params (random
    LayerNorm vectors and biases, doubled Wq / Wk); x is randn."""
    seed = _seed(case)
    p = B.make_params(case, seed)
    g = torch.Generator().manual_seed(seed + 1)
    rows, dim = case["n_seq"] * case["n_tok"], case["dim"]
    x = torch.randn(rows, dim, generator=g)
    dy = make_dy(rows, dim, g)
    keep = make_keep(case["n_seq"], case["n_tok"], g) if case["masked"] else None
    return p, x, dy, keep


def att_references(case, device="cpu", bug=None):
    """(fp64 dqkv, emulated dqkv) of a kernel-level case; with ``bug`` the first is the mutant."""
    qkv, dout, keep = att_inputs(case)
    qkv, dout = qkv.double().to(device), dout.double().to(device)
    keep = keep.to(device) if keep is not None else None
    args = (case["n_seq"], case["n_tok"], case["heads"], case["dh"], keep)
    ref = attention_bwd(qkv, dout, *args, bug=bug)
    emu = attention_bwd(qkv, dout, *args, path="per_op") if bug is None else None
    return ref, emu


def stack_reference(case, path=None, bug=None, device="cpu"):
    """{"dx": [rows, dim], "l.name": gradient} of a stack case in fp64 (path None) or emulated (path "per_op"), or a mutant."""
    p, x, dy, keep = stack_inputs(case)
    n_seq, n_tok, dim = case["n_seq"], case["n_tok"], case["dim"]
    p64 = {k: v.double().to(device) for k, v in p.items()}
    x64 = x.double().to(device).view(n_seq, n_tok, dim)
    dy64 = dy.double().to(device).view(n_seq, n_tok, dim)
    keep = keep.to(device) if keep is not None else None
    dx, grads = stack_bwd(x64, p64, dy64, case["depth"], 8, keep, path, bug)
    out = {"dx": dx.reshape(-1, dim)}
    out.update(zip(grad_names(case["depth"]), grads))
    return out


def stack_ratios(got, emu, ref):
    """{tensor: (worst ratio, median ratio | None)} over every row of dx and every gradient."""
    return {k: ratios(k, got[k].double().to(ref[k].device), emu[k], ref[k]) for k in ref}
