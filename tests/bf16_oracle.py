"""bf16 error budgets for the encoder stacks.  TEST INFRASTRUCTURE ONLY, next to oracle/avformer_oracle.py, whose primitives
(LayerNorm, tanh-GELU, the stack itself as the fp64 reference) it reuses.

A bf16 stack differs from the fp64 oracle by its rounding.  A single max-abs bound over the whole output has to admit the worst
rounding anywhere, and a kernel that drops a key or kills a head stays under it at some shapes.  Instead, each case gets its own
budget: the same stack computed in fp64 with bf16 rounding at the points where the kernel rounds (``stack_emulated``).  A kernel
passes when its worst token row is within ``K`` times the emulation's worst token row, both in per-row RMS error against fp64
(``row_rms``).  ``mutant`` is the fp64 stack with one deliberate bug; tests/test_bf16_budget_sensitivity.py shows that every
mutant lands well outside the budget of every case tests/test_gpu_bf16_budget.py runs.

Parameters use the key names of ``avformer_b200.Transformer.state_dict()`` under ``pre`` ("layers.{l}.0.fn.norm.weight", ...)."""
import math

import numpy as np
import torch

from oracle import avformer_oracle as O

# A case passes when max_row row_rms(kernel - fp64) <= K * max_row row_rms(emulated - fp64).  K = 1.5 x the largest kernel /
# emulation ratio over every case of tests/test_gpu_bf16_budget.py, measured on one B200 (1000 W limit, 1965 MHz max SM clock):
# 1.159 (fused, rows-d256-t40); median-row ratios 0.99-1.045 (profiles/r06_bf16_budget_ratios.json).
K = 1.74

MUTANTS = ("drop_last_key", "neighbour_key_first_row", "extra_zero_key", "head_uniform", "ln1_ln2_swapped", "layer0_vectors",
           "b_ff1_chunk_rolled", "row_not_stored")

LOG2E = 1.4426950408889634
SMS = 148                    # B200: the fused kernel's grid is min(tiles, SMs); "wave boundary" tiles below are SMS - 1 and SMS


def bf(t):
    """Round to bf16 (nearest even) and return in t's dtype."""
    return t.to(torch.float32).to(torch.bfloat16).to(t.dtype)


def row_rms(err):
    """RMS error of each token row: err [..., dim] -> [...]."""
    return err.double().pow(2).mean(dim=-1).sqrt()


def budget(emulated, ref64):
    """The worst token row of the emulation: what a correct kernel may reach, up to K."""
    return row_rms(emulated - ref64).max().item()


# ---------------------------------------------------------------------------------------------------------------------------------
# the stack with optional bf16 rounding (path) or one bug (bug)
# ---------------------------------------------------------------------------------------------------------------------------------
def _layer_norm(x, g, b, path):
    if path == "fused":
        # avf_layer_fused.cu:269: (x - mean) * rstd in fp32 -> bf16, then fma.rn.bf16x2 with the bf16 gamma / beta (rounded when the
        # per-layer vectors are staged, :465-466): one rounding of the exact product-sum
        mu = x.mean(dim=-1, keepdim=True)
        var = ((x - mu) ** 2).mean(dim=-1, keepdim=True)
        return bf(bf((x - mu) / torch.sqrt(var + 1e-5)) * bf(g) + bf(b))
    y = O.layer_norm(x, g, b)
    return bf(y) if path == "per_op" else y          # avf_rowops.cu:46-54: fp32 LayerNorm, stored as bf16


def _gelu_fused(h):
    """gelu_bf16x2 (avf_fused_helpers.cuh:72-80) on bf16 inputs: every packed bf16x2 operation rounds, tanh.approx modelled as
    a rounded tanh."""
    c0, c1 = 0.796875, bf(torch.tensor(math.sqrt(2.0 / math.pi) * 0.044715, dtype=torch.float64)).item()
    x2 = bf(h * h)
    u = bf(h * bf(x2 * c1 + c0))
    hx = bf(h * 0.5)
    return bf(hx * bf(torch.tanh(u)) + hx)


def _attention(x, p, pre, heads, path, bug, keep=None, tape=None):
    """``keep`` [B, N] bool (True = kept): the mask of mask_score (avf_attention_mma.cu:48-52); ``tape`` (a dict) receives the
    bf16 qkv and merged-head o that the training forward stores (avf_train_api.cu:110-111)."""
    B, N, _ = x.shape
    r = bf if path else (lambda t: t)
    wqkv = p[pre + "fn.fn.to_qkv.weight"]
    inner = wqkv.shape[0] // 3
    dh = inner // heads
    # Q, K, V stored as bf16: avf_layer_fused.cu:494 (pack8u of the fp32 accumulator) / avf_api.cu:132 (GEMM with a bf16 output)
    qkv = r(x @ r(wqkv).t())
    q, k, v = (t.reshape(B, N, heads, dh).permute(0, 2, 1, 3) for t in qkv.split(inner, dim=-1))
    s = torch.matmul(q, k.transpose(-1, -2))
    if keep is not None:                             # kept query: -inf on dropped keys; dropped query: the same score on every key
        s = s.masked_fill(~keep[:, None, None, :], -math.inf).masked_fill(~keep[:, None, :, None], 0.0)
    if bug == "drop_last_key":
        s[..., -1] = -math.inf
    elif bug == "head_uniform":
        s[:, heads - 1] = 0.0
    elif bug == "extra_zero_key":                    # one more key with score 0 and a zero value row
        s = torch.cat([s, torch.zeros_like(s[..., :1])], dim=-1)
        v = torch.cat([v, torch.zeros_like(v[..., :1, :])], dim=-2)
    elif bug == "neighbour_key_first_row":           # token 0 of sequence b also sees key 0 of sequence b - 1
        extra = torch.full_like(s[..., :1], -math.inf)
        extra[:, :, 0, 0] = (q[:, :, 0] * k.roll(1, dims=0)[:, :, 0]).sum(-1)
        s = torch.cat([s, extra], dim=-1)
        v = torch.cat([v, v.roll(1, dims=0)[..., :1, :]], dim=-2)
    scale = LOG2E * dh ** -0.5                      # scores in exp2 units, like both kernels
    arg = (s - s.amax(dim=-1, keepdim=True)) * scale
    if path == "fused":
        # avf_layer_fused.cu:578 (and softmax_fixed, :328): the exp2 argument rounded to bf16, ex2.approx.bf16x2 returns bf16 P;
        # the row sum is taken over the rounded P (:579), O / l rounded to bf16 (:517)
        e = bf(torch.exp2(bf(arg)))
        o = bf(torch.matmul(e, v) / e.sum(dim=-1, keepdim=True))
    elif path == "per_op":
        # avf_attention_mma.cu:168-173: fp32 exp2 and row sum; P rounded to bf16 as the PV operand (:186-189); O / l -> bf16 (:205)
        e = torch.exp2(arg)
        o = bf(torch.matmul(bf(e), v) / e.sum(dim=-1, keepdim=True))
    else:
        e = torch.exp2(arg)
        o = torch.matmul(e, v) / e.sum(dim=-1, keepdim=True)
    o = o.permute(0, 2, 1, 3).reshape(B, N, inner)
    if tape is not None:
        tape.update(qkv=qkv, o=o)
    return o @ r(p[pre + "fn.fn.to_out.0.weight"]).t() + p[pre + "fn.fn.to_out.0.bias"]


def _feed_forward(x, p, pre, path, tape=None):
    """``tape`` (a dict) receives the fp32 pre-activation h (the training forward stores bf16(h), avf_gemm_umma.cu:113-124) and g."""
    r = bf if path else (lambda t: t)
    h = x @ r(p[pre + "fn.fn.net.0.weight"]).t() + p[pre + "fn.fn.net.0.bias"]
    if path == "fused":
        g = _gelu_fused(bf(h))                       # avf_layer_fused.cu:630: h + b1 rounded to bf16, packed bf16 GELU
    elif path == "per_op":
        g = bf(O.gelu_tanh(h))                       # avf_gemm_umma.cu:127: fp32 tanh-GELU in the epilogue, stored as bf16
    else:
        g = O.gelu_tanh(h)
    if tape is not None:
        tape.update(h=h, g=g)
    return g @ r(p[pre + "fn.fn.net.3.weight"]).t() + p[pre + "fn.fn.net.3.bias"]


_VECTORS = ("0.fn.norm.weight", "0.fn.norm.bias", "0.fn.fn.to_out.0.bias", "1.fn.norm.weight", "1.fn.norm.bias", "1.fn.fn.net.0.bias",
            "1.fn.fn.net.3.bias")


def _mutate_params(p, pre, depth, bug):
    q = dict(p)
    for l in range(depth):
        a, f = f"{pre}layers.{l}.0.fn.norm.", f"{pre}layers.{l}.1.fn.norm."
        if bug == "ln1_ln2_swapped":
            for s in ("weight", "bias"):
                q[a + s], q[f + s] = p[f + s], p[a + s]
        elif bug == "layer0_vectors":
            for k in _VECTORS:
                q[f"{pre}layers.{l}.{k}"] = p[f"{pre}layers.0.{k}"]
        elif bug == "b_ff1_chunk_rolled":                # chunk c of the hidden layer gets the bias of chunk c + 1
            k = f"{pre}layers.{l}.1.fn.fn.net.0.bias"
            q[k] = p[k].roll(-128)
    return q


def _stack(x, p, pre, depth, heads, path=None, bug=None):
    x0 = x
    if bug is not None:
        p = _mutate_params(p, pre, depth, bug)
    for l in range(depth):
        a, f = f"{pre}layers.{l}.0.", f"{pre}layers.{l}.1."
        x = x + _attention(_layer_norm(x, p[a + "fn.norm.weight"], p[a + "fn.norm.bias"], path), p, a, heads, path, bug)
        x = x + _feed_forward(_layer_norm(x, p[f + "fn.norm.weight"], p[f + "fn.norm.bias"], path), p, f, path)
    if bug == "row_not_stored":                          # the last token row of the last sequence keeps its input
        x = x.clone()
        x[-1, -1] = x0[-1, -1]
    return x


def stack_fp64(x, p, pre, depth, heads):
    """The same restatement with no rounding and no bug (equals O.transformer; pinned by the CPU tests)."""
    return _stack(x, p, pre, depth, heads)


def stack_emulated(x, p, pre, depth, heads, path):
    """x [n_seq, n_tok, dim] fp64 (the kernel's fp32 input, positional add included) -> the stack in fp64 with bf16 rounding where
    ``path`` rounds: "fused" (avf_layer_fused.cu) or "per_op" (the kernel-per-operation bf16 path of encoder_stack, avf_api.cu).
    Weights as bf16, biases fp32, the residual stream fp32 in both.  Accumulation order is not modelled: fp32 accumulation of
    products of bf16 values is far below bf16 rounding."""
    assert path in ("fused", "per_op")
    return _stack(x, p, pre, depth, heads, path=path)


def mutant(kind, x, p, pre, depth, heads):
    """The fp64 stack with one bug ``kind`` (see MUTANTS):
    drop_last_key            the last key of every sequence is left out of every softmax;
    neighbour_key_first_row  the first token row of each sequence also attends to the first key of the previous sequence;
    extra_zero_key           every softmax has one more key, with score 0 and a zero value row (a padding column counted);
    head_uniform             the last head attends uniformly (its scores are all 0);
    ln1_ln2_swapped          each layer's LN1 uses LN2's gamma / beta and vice versa;
    layer0_vectors           every layer uses layer 0's LayerNorm vectors and biases;
    b_ff1_chunk_rolled       the first MLP bias is rotated by one 128-wide chunk;
    row_not_stored           the last token row of the last sequence is never written (keeps its input)."""
    assert kind in MUTANTS, kind
    return _stack(x, p, pre, depth, heads, bug=kind)


def mutant_applies(kind, n_tok, depth, mlp):
    """Bugs that are no bugs at a shape: one token has nothing to drop and nothing to average over, one layer has no layer 0 to
    borrow from, one MLP chunk has nothing to rotate."""
    if kind in ("drop_last_key", "head_uniform"):
        return n_tok >= 2
    if kind == "layer0_vectors":
        return depth >= 2
    if kind == "b_ff1_chunk_rolled":
        return mlp >= 256
    return True


# ---------------------------------------------------------------------------------------------------------------------------------
# the cases of tests/test_gpu_bf16_budget.py (shared with the sensitivity test, which checks the mutants on the same inputs)
# ---------------------------------------------------------------------------------------------------------------------------------
ROWS_NTOK = (1, 2, 3, 7, 8, 9, 12, 15, 16, 17, 24, 31, 32, 33, 40, 48, 49, 57, 63, 64)
MLPS = (128, 256, 384, 512, 640, 1024)


def slot_of(n_tok):
    return 16 if n_tok <= 16 else (32 if n_tok <= 32 else 64)


def _rows_cases():
    cases = []
    for dim in (256, 128):
        for i, n_tok in enumerate(ROWS_NTOK):
            spt = 128 // slot_of(n_tok)
            cases.append(dict(name=f"rows-d{dim}-t{n_tok}", kind="rows", dim=dim, dh=32, n_tok=n_tok, depth=1 + i % 3,
                              mlp=MLPS[(i + (dim == 128)) % len(MLPS)], n_seq=_n_seq(spt), sample=None))
    # more tiles than SMs: 190 .. 301 tiles, the last one partial; static striding gives CTA b the tiles b, b + 148, ...
    for dim, n_tok, depth, mlp, tiles in ((256, 12, 2, 512, 301), (128, 33, 3, 256, 201), (256, 64, 1, 1024, 190)):
        spt = 128 // slot_of(n_tok)
        n_seq = (tiles - 1) * spt + 1
        cases.append(dict(name=f"rows-d{dim}-t{n_tok}-{tiles}tiles", kind="rows", dim=dim, dh=32, n_tok=n_tok, depth=depth, mlp=mlp,
                          n_seq=n_seq, sample=_sample_seqs(n_seq, spt)))
    return cases


def _n_seq(spt):
    """At least 24 sequences (a bug in the first row of a sequence gets 24 chances to show), the last tile partial."""
    return spt * -(-24 // spt) + (spt + 1) // 2


def _sample_seqs(n_seq, spt):
    """Sequences of the first tile, the two tiles at the wave boundary (SMS - 1, SMS) and the last tile."""
    n_tiles = (n_seq + spt - 1) // spt
    seqs = set()
    for t in (0, SMS - 1, SMS, n_tiles - 1):
        seqs.update(range(t * spt, min(n_seq, (t + 1) * spt)))
    return sorted(seqs)


NCHW_MAPS = ((1, 1), (2, 2), (3, 5), (4, 4), (6, 6), (8, 8), (7, 9))


def _nchw_cases():
    cases = [dict(name="nchw-resformer-7x7", kind="nchw", dim=256, dh=32, hw=(7, 7), n_tok=49, depth=1, mlp=512, num_patches=49, n_seq=_n_seq(2),
                  sample=None)]
    for i, hw in enumerate(NCHW_MAPS):
        n_tok = hw[0] * hw[1]
        spt = 128 // slot_of(n_tok)
        n_seq = _n_seq(spt)
        sample = None
        if hw == (4, 4):                             # 151 tiles on at most 148 CTAs (the NCHW form hands tiles out dynamically)
            n_seq = 150 * spt + 3
            sample = _sample_seqs(n_seq, spt)
        cases.append(dict(name=f"nchw-{hw[0]}x{hw[1]}", kind="nchw", dim=256, dh=32, hw=hw, n_tok=n_tok, depth=1 + i % 3, mlp=(512, 1024)[i % 2],
                          num_patches=64, n_seq=n_seq, sample=sample))
    return cases


def _tformer_cases():
    return [dict(name=f"rows-d512-t{n_tok}", kind="rows", dim=512, dh=64, n_tok=n_tok, depth=3, mlp=1024, n_seq=6, sample=None)
            for n_tok in (9, 17, 33, 64)]


FUSED_CASES = _rows_cases() + _nchw_cases()
PER_OP_CASES = FUSED_CASES + _tformer_cases()
ALL_CASES = PER_OP_CASES


def make_params(case, seed):
    """fp32 parameters like the module's, with the vectors a fresh module leaves at 1 / 0 drawn at random: LayerNorm gamma
    1 + 0.3 randn, beta 0.5 randn; Linear weights and biases uniform in +-1/sqrt(fan_in) (nn.Linear's initialisation).  Two
    departures make the attention bugs visible above bf16 rounding: LN1's beta is 1.0 randn (a common offset of V, which a
    zero-valued extra key pulls towards 0) and Wq / Wk are twice as large (scores peaked enough that one key matters to some rows,
    as in a trained model, instead of near-uniform weights of 1 / n_tok)."""
    g = torch.Generator().manual_seed(seed)
    dim, mlp, inner = case["dim"], case["mlp"], 8 * case["dh"]
    qk_gain = torch.ones(3 * inner, 1)
    qk_gain[:2 * inner] = 2.0

    def unif(*shape, fan_in):
        return (torch.rand(*shape, generator=g) * 2 - 1) / math.sqrt(fan_in)

    p = {}
    for l in range(case["depth"]):
        a, f = f"layers.{l}.0.fn.", f"layers.{l}.1.fn."
        p[a + "norm.weight"] = 1 + 0.3 * torch.randn(dim, generator=g)
        p[a + "norm.bias"] = 1.0 * torch.randn(dim, generator=g)
        p[a + "fn.to_qkv.weight"] = unif(3 * inner, dim, fan_in=dim) * qk_gain
        p[a + "fn.to_out.0.weight"] = unif(dim, inner, fan_in=inner)
        p[a + "fn.to_out.0.bias"] = unif(dim, fan_in=inner)
        p[f + "norm.weight"] = 1 + 0.3 * torch.randn(dim, generator=g)
        p[f + "norm.bias"] = 0.5 * torch.randn(dim, generator=g)
        p[f + "fn.net.0.weight"] = unif(mlp, dim, fan_in=dim)
        p[f + "fn.net.0.bias"] = unif(mlp, fan_in=dim)
        p[f + "fn.net.3.weight"] = unif(dim, mlp, fan_in=mlp)
        p[f + "fn.net.3.bias"] = unif(dim, fan_in=mlp)
    return p


def make_inputs(case):
    """(params fp32, kernel input, pos fp32 [n_tok, dim]).  The input is fp32 token rows [n_seq * n_tok, dim] (rows) or a bf16 NCHW
    map [n_seq, 256, h, w] (nchw; 0.6 randn: the bf16 rounding of the output, part of the budget, grows with the values)."""
    seed = int(np.frombuffer(case["name"].encode(), dtype=np.uint8).astype(np.int64).sum()) * 7919 + case["n_tok"]
    p = make_params(case, seed)
    g = torch.Generator().manual_seed(seed + 1)
    n_tok, dim = case["n_tok"], case["dim"]
    pos = 0.5 * torch.randn(n_tok, dim, generator=g)
    if case["kind"] == "rows":
        x = torch.randn(case["n_seq"] * n_tok, dim, generator=g)
    else:
        h, w = case["hw"]
        x = (0.6 * torch.randn(case["n_seq"], dim, h, w, generator=g)).bfloat16()
    return p, x, pos


def tokens64(case, x, pos, seqs=None):
    """The stack's fp64 input [n_seq, n_tok, dim]: token rows + pos (for an NCHW map: token n = position n of the map)."""
    n_tok, dim = case["n_tok"], case["dim"]
    if case["kind"] == "rows":
        t = x.double().view(-1, n_tok, dim)
    else:
        t = x.double().reshape(x.shape[0], dim, n_tok).permute(0, 2, 1)
    if seqs is not None:
        t = t[seqs]
    return t + pos.double()


def references(case, seqs=None):
    """(ref64, emulated fused, emulated per_op, fp64 input tokens) of a case on the sequences ``seqs`` (None: all).  The NCHW form
    stores bf16 maps: both emulations round the output too."""
    p, x, pos = make_inputs(case)
    p64 = {k: v.double() for k, v in p.items()}
    t = tokens64(case, x, pos, seqs)
    ref = stack_fp64(t, p64, "", case["depth"], 8)
    emu = {path: stack_emulated(t, p64, "", case["depth"], 8, path) for path in ("fused", "per_op")}
    if case["kind"] == "nchw":
        emu = {k: bf(v) for k, v in emu.items()}
    return ref, emu["fused"], emu["per_op"], t, p64
