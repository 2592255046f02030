"""Attention maps: the softmax probabilities every attention kernel family writes when asked (include/avformer_b200.h, "attention
maps"; INTEGRATION.md section 1).

1. one attention: dh 32 at 12 / 17 / 49 tokens, dh 64 at 17 / 64 / 65 / 129 / 256 tokens, fp32 and bf16, masked and not: out bit-equal
   to attention_fwd, probs against the fp64 softmax of the same q / k, rows summing to 1, dropped keys exactly 0, dropped queries
   uniform, an all-kept mask bit-equal to the unmasked maps;
2. stacks: Transformer.attention_maps bit-equal to the fused-off forward with the same launches, fp32 maps against the oracle's own
   per-layer ``attn`` (collected by recording torch.softmax, which leaves every returned value unchanged), bf16 maps within a per-row
   budget against the bf16 emulation of tests/bf16_maps_oracle.py;
3. the TFormer at T in {16, 64, 128, 255}: cls bit-equal to cls_features, the last map full, the indexed form bit-equal to the
   explicit gather;
4. the model: out21 bit-equal to the fused-off model(x) for any selection of stacks, maps independent of the selection, shapes, errors."""
import os
import sys
from unittest import mock

import pytest
import torch

import avformer_b200 as A
from oracle import avformer_oracle as O

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import bf16_maps_oracle as BM  # noqa: E402
import bf16_oracle as B  # noqa: E402
import masked_oracle as MO  # noqa: E402

pytestmark = pytest.mark.gpu
AF = A.functional
L = A._lib.lib
MEDIAN_RATIO = (0.5, 2.0)


@pytest.fixture(autouse=True)
def _deterministic():
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    old = torch.backends.cudnn.deterministic, torch.backends.cudnn.benchmark
    torch.backends.cudnn.deterministic, torch.backends.cudnn.benchmark = True, False
    yield
    torch.backends.cudnn.deterministic, torch.backends.cudnn.benchmark = old


class _FusedOff:
    def __enter__(self):
        self.prev = AF.set_fused_enabled(False)

    def __exit__(self, *exc):
        AF.set_fused_enabled(self.prev)


def _keep(n_seq, n_tok, seed):
    """Random keep rows (token 0 kept); sequence 1 keeps token 0 only, sequence 2 drops every token."""
    g = torch.Generator().manual_seed(seed)
    k = torch.rand(n_seq, n_tok, generator=g) < 0.6
    k[:, 0] = True
    k[1, 1:] = False
    k[2] = False
    return k


def _probs_ref(qkv, n_seq, n_tok, heads, dh, keep):
    """fp64 softmax of the same q / k, masked as mask_score: kept query -> 0 on dropped keys, dropped query -> uniform."""
    q, k, _ = (t.reshape(n_seq, n_tok, heads, dh).permute(0, 2, 1, 3) for t in qkv.double().cpu().chunk(3, dim=-1))
    s = q @ k.transpose(-1, -2) * dh ** -0.5
    if keep is not None:
        s = s.masked_fill(~keep[:, None, None, :], -float("inf")).masked_fill(~keep[:, None, :, None], 0.0)
    return torch.softmax(s, dim=-1)


def _module_keep(keep):
    """The keep rows a module mask ``keep[:, 1:]`` stands for: the first (cls) token is always kept (AF.keep_from_mask)."""
    k = keep.clone()
    k[:, 0] = True
    return k


def _check_map_invariants(probs, keep, n_tok):
    """Rows sum to 1 within fp32 rounding: p_j = rn(e_j / l) with l an fp32 sum of n_tok terms, at most 2 n_tok ulp(1) = n_tok * 2^-23
    off; the online softmax of the fp32 kernels builds l through rescales by exp2f factors (2 ulp each), for which 64 more ulp are
    allowed.  A kept query gets exactly 0.0 on a dropped key; a dropped query's row is uniform (all entries equal, = 1 / n_tok rounded
    once)."""
    p = probs.double().cpu()
    assert torch.isfinite(p).all()
    assert (p.sum(-1) - 1).abs().max().item() <= (n_tok + 64) * 2 ** -23
    if keep is None:
        return
    kept_q = keep[:, None, :, None].expand_as(p)
    drop_k = ~keep[:, None, None, :].expand_as(p)
    assert not bool(p[kept_q & drop_k].any()), "a kept query has a nonzero probability on a dropped key"
    rows = p.permute(0, 2, 1, 3)[~keep]                            # [n_dropped, heads, n_tok]
    assert bool((rows == rows[..., :1]).all()), "a dropped query's row is not uniform"
    assert (rows - 1.0 / n_tok).abs().max().item() <= 2 ** -24 / n_tok * 2


# ---------------------------------------------------------------------------------------------
# 1. one attention, every kernel family
# ---------------------------------------------------------------------------------------------
SHAPES = [(32, 12), (32, 17), (32, 49), (64, 17), (64, 64), (64, 65), (64, 129), (64, 256)]


@pytest.mark.parametrize("dh,n_tok", SHAPES)
@pytest.mark.parametrize("masked", [False, True])
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_attention_probs(dh, n_tok, masked, dtype):
    torch.manual_seed(dh * 1000 + n_tok)
    n_seq, heads = 5, 8
    qkv = torch.randn(n_seq * n_tok, 3 * heads * dh, device="cuda").to(dtype)
    keep = _keep(n_seq, n_tok, n_tok + dh) if masked else None
    kc = keep.cuda() if masked else None
    out, probs = AF.attention_fwd_probs(qkv, n_seq, n_tok, heads, dh, kc)
    assert probs.shape == (n_seq, heads, n_tok, n_tok) and probs.dtype == torch.float32 and probs.is_contiguous()
    assert torch.equal(out, AF.attention_fwd(qkv, n_seq, n_tok, heads, dh, kc)), "O of the map-writing launch differs"
    # The q / k values are exact in fp64, so the error is fp32 arithmetic only: the score's fp32 accumulation over dh products
    # (|s| <= ~40 here, relative error ~dh * 2^-24, i.e. <= 1e-5 in the exp2 argument), exp2f (2 ulp) and the fp32 row sum
    # (<= n_tok * 2^-24 relative).  The tensor-core accumulation of the bf16 kernels truncates instead of rounding: 4x the margin.
    # Both bounds sit far below the bf16 resolution of P (2^-8 relative), which a wrong key, row or head would exceed.
    err = (probs.double().cpu() - _probs_ref(qkv, n_seq, n_tok, heads, dh, keep)).abs().max().item()
    assert err <= (2.5e-5 if dtype == torch.float32 else 1e-4), f"max |p - p64| = {err:.3e}"
    _check_map_invariants(probs, keep, n_tok)
    if masked:
        everything = torch.ones(n_seq, n_tok, dtype=torch.bool, device="cuda")
        o_all, p_all = AF.attention_fwd_probs(qkv, n_seq, n_tok, heads, dh, everything)
        o_none, p_none = AF.attention_fwd_probs(qkv, n_seq, n_tok, heads, dh)
        assert torch.equal(p_all, p_none) and torch.equal(o_all, o_none)


# ---------------------------------------------------------------------------------------------
# 2. stacks
# ---------------------------------------------------------------------------------------------
STACKS = {"d128": (128, 2, 8, 32, 256, 12), "d256": (256, 1, 8, 32, 512, 49), "d512": (512, 3, 8, 64, 1024, 17)}


def _stack(name, precision, seed=3):
    dim, depth, heads, dh, mlp, n_tok = STACKS[name]
    p = O.params_from_spec(list(O._encoder_spec("", dim, depth, heads * dh, mlp)), seed)
    m = A.Transformer(dim, depth, heads, dh, mlp)
    m.load_state_dict(p, strict=True)
    m.precision = precision
    return m.cuda().eval(), {k: v.double() for k, v in p.items()}, n_tok


def _oracle_attn(fn, *args):
    """Run an oracle function and collect the ``attn`` of each of its softmax calls (models/heads.py:234); returns (result, maps)."""
    seen, real = [], torch.softmax

    def record(t, dim):
        out = real(t, dim=dim)
        seen.append(out)
        return out
    with mock.patch.object(torch, "softmax", record):
        res = fn(*args)
    return res, torch.stack(seen)


@pytest.mark.parametrize("name", list(STACKS))
@pytest.mark.parametrize("masked", [False, True])
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_stack_maps(name, masked, precision):
    m, p64, n_tok = _stack(name, precision)
    dim, depth, heads = m.dim, m.depth, m.heads
    n_seq = 7
    x = torch.randn(n_seq, n_tok, dim, generator=torch.Generator().manual_seed(n_tok)).cuda()
    keep = _module_keep(_keep(n_seq, n_tok, 11)) if masked else None
    mask = keep[:, 1:].cuda() if masked else None
    m.packed()                                                # the bf16 weight copies are made once, outside the counted calls
    with torch.no_grad(), _FusedOff():
        n0 = L().avf_launch_count()
        ref = m(x, mask)
        n1 = L().avf_launch_count()
        y, maps = m.attention_maps(x, mask)
        n2 = L().avf_launch_count()
    assert torch.equal(y, ref), f"max |diff| {(y - ref).abs().max().item():.3e}"
    assert n2 - n1 == n1 - n0, f"{n2 - n1} launches with maps, {n1 - n0} without"
    assert maps.shape == (depth, n_seq, heads, n_tok, n_tok) and maps.is_contiguous()
    for l in range(depth):
        _check_map_invariants(maps[l], keep, n_tok)
    x64 = x.double().cpu()
    if precision == "fp32":
        # the oracle's own attn: fp32 parity mode agrees with it to the project's 1e-4 parity tolerance
        if masked:
            _, ref_maps = _oracle_attn(MO.transformer, x64, p64, "", depth, heads, keep[:, 1:])
        else:
            _, ref_maps = _oracle_attn(O.transformer, x64, p64, "", depth, heads)
        assert ref_maps.shape == maps.shape
        err = (maps.double().cpu() - ref_maps).abs().max().item()
        assert err <= 1e-4, f"fp32 maps: max |p - attn| = {err:.3e}"
    elif not masked:
        # per softmax row: RMS error against fp64, worst and median row against the bf16 emulation's (tests/bf16_oracle.py's form)
        _, ref_maps = BM.stack_maps(x64, p64, "", depth, heads)
        _, emu_maps = BM.stack_maps(x64, p64, "", depth, heads, path="per_op")
        got, exp = B.row_rms(maps.double().cpu() - ref_maps), B.row_rms(emu_maps - ref_maps)
        worst, median = (got.max() / exp.max()).item(), (got.median() / exp.median()).item()
        print(f"\nmaps {name}: worst-row ratio {worst:.3f}, median-row ratio {median:.3f}")
        assert MEDIAN_RATIO[0] <= median <= MEDIAN_RATIO[1], f"median-row ratio {median:.3f}: the emulation does not model the kernel"
        assert worst <= B.K, f"worst row {worst:.3f} x the emulation's (budget {B.K})"


def test_stack_maps_refuse_training_calls():
    m, _, n_tok = _stack("d128", "bf16")
    x = torch.randn(2, n_tok, m.dim, device="cuda")
    with pytest.raises(RuntimeError, match="no_grad"):
        m.attention_maps(x)                                   # parameters require grad, grad mode on
    m.dropout = 0.1
    m.train()
    with torch.no_grad(), pytest.raises(RuntimeError, match=r"eval\(\)"):
        m.attention_maps(x)


# ---------------------------------------------------------------------------------------------
# 3. the TFormer
# ---------------------------------------------------------------------------------------------
def _tformer(T, precision, seed=9):
    p = O.params_from_spec([("cls_token", (1, 1, 512), "normal"), ("pos_embedding", (1, T + 1, 512), "normal")]
                           + list(O._encoder_spec("spatial_transformer.", 512, 3, 512, 1024)), seed)
    tf = A.TFormer(num_patches=T).cuda().eval()
    tf.load_state_dict(p, strict=True)
    tf.spatial_transformer.precision = precision
    return tf


@pytest.mark.parametrize("T", [16, 64, 128, 255])
@pytest.mark.parametrize("masked", [False, True])
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_tformer_maps(T, masked, precision):
    tf = _tformer(T, precision)
    n_clips = 6
    frames = torch.randn(n_clips * T, 512, generator=torch.Generator().manual_seed(T)).cuda()
    keep = _module_keep(_keep(n_clips, T + 1, T)) if masked else None
    mask = keep[:, 1:].cuda() if masked else None
    with torch.no_grad():
        ref = tf.cls_features(frames, mask)
        n0 = L().avf_launch_count()
        cls, maps = tf.attention_maps(frames, mask)
        n1 = L().avf_launch_count()
        tf.cls_features(frames, mask)
        n2 = L().avf_launch_count()
    assert torch.equal(cls, ref), f"max |diff| {(cls - ref).abs().max().item():.3e}"
    assert n1 - n0 == n2 - n1
    assert maps.shape == (3, n_clips, 8, T + 1, T + 1)
    for l in range(3):                                        # the last layer too: every query row is written
        _check_map_invariants(maps[l], keep, T + 1)

    # the indexed form, with -1 entries, against the explicit gather with mask = index >= 0
    n_bank = 3 * T // 2 + 1
    bank = torch.randn(n_bank, 512, generator=torch.Generator().manual_seed(T + 1)).cuda()
    g = torch.Generator().manual_seed(T + 2)
    index = torch.randint(0, n_bank, (n_clips, T), generator=g)
    index[torch.rand(n_clips, T, generator=g) < 0.3] = -1
    index[1, 1:] = -1
    with torch.no_grad():
        cls_i, maps_i = tf.attention_maps_indexed(bank, index)
        cls_e, maps_e = tf.attention_maps(bank[index.clamp(min=0).cuda()].reshape(-1, 512), mask=(index >= 0).cuda())
    assert torch.equal(cls_i, cls_e) and torch.equal(maps_i, maps_e)


def test_tformer_maps_errors():
    tf = _tformer(16, "bf16")
    bank = torch.randn(20, 512, device="cuda")
    good = torch.zeros(3, 16, dtype=torch.long)
    with pytest.raises(RuntimeError, match="no_grad"):
        tf.attention_maps(torch.randn(3 * 16, 512, device="cuda"))
    with torch.no_grad():
        for bad, err in ((torch.zeros(3, 15, dtype=torch.long), ValueError), (torch.zeros(3, 16), TypeError),
                         (torch.full((3, 16), 20), ValueError), (torch.full((3, 16), -2), ValueError), (good.tolist(), TypeError)):
            with pytest.raises(err) as e_maps:
                tf.attention_maps_indexed(bank, bad)
            with pytest.raises(err) as e_cls:
                tf.cls_features_indexed(bank, bad)
            assert str(e_maps.value).replace("attention_maps_indexed", "cls_features_indexed") == str(e_cls.value)
        with pytest.raises(ValueError, match="bank must be"):
            tf.attention_maps_indexed(torch.randn(20, 256, device="cuda"), good)
        tf.spatial_transformer.dropout = 0.1
        tf.train()
        with pytest.raises(RuntimeError, match=r"eval\(\)"):
            tf.attention_maps_indexed(bank, good)


# ---------------------------------------------------------------------------------------------
# 4. the model
# ---------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def model_and_input():
    T, bs = 16, 2
    m = A.TwoStreamAuralVisualFormer(video_pretrained=False, audio_pretrained=False, task="AU")
    m.load_state_dict(O.make_state_dict(4, T), strict=True)
    m = m.cuda().eval().set_precision("bf16")
    for p in m.parameters():
        p.requires_grad_(False)
    clip, audio, _ = O.synth_inputs(4, bs, T)
    return m, {"clip": clip.cuda(), "audio_features": audio.cuda()}, T, bs


def test_model_maps(model_and_input):
    m, x, T, bs = model_and_input
    with torch.no_grad():
        with _FusedOff():
            ref = m(x)
        out_all, maps_all = m.attention_maps(x)
        shapes = {"sformer": (1, bs * T, 8, 49, 49), "tformer": (3, bs, 8, T + 1, T + 1), "audio_au_former": (2, bs, 8, 12, 12),
                  "video_au_former": (2, bs, 8, 12, 12), "fusion_head": (3, bs, 8, 12, 12)}
        assert {k: tuple(v.shape) for k, v in maps_all.items()} == shapes
        assert torch.equal(out_all, ref)
        for stacks in (["tformer"], []):
            out, maps = m.attention_maps(x, stacks)
            assert torch.equal(out, ref) and set(maps) == set(stacks)
        for name in shapes:
            out, maps = m.attention_maps(x, [name])
            assert torch.equal(out, ref) and torch.equal(maps[name], maps_all[name]), name
            for l in range(maps[name].shape[0]):
                _check_map_invariants(maps[name][l], None, maps[name].shape[-1])
    assert AF.set_fused_enabled(True), "attention_maps left the fused kernel switched off"


def test_model_maps_errors(model_and_input):
    m, x, _, _ = model_and_input
    with torch.no_grad(), pytest.raises(ValueError, match="unknown stack"):
        m.attention_maps(x, ["tformer", "s_former"])
    p = m.au_head.pos_embedding
    p.requires_grad_(True)
    try:
        with pytest.raises(RuntimeError, match="no_grad"):
            m.attention_maps(x)
    finally:
        p.requires_grad_(False)
    m.train()
    try:
        with torch.no_grad(), pytest.raises(RuntimeError, match=r"eval\(\)"):
            m.attention_maps(x, ["tformer"])
    finally:
        m.eval()
