"""Attention relevance: gradient maps G = P o dP written by the attention backward kernels, their rollout, and the per-AU relevance
of the whole model (include/avformer_b200.h, "attention relevance"; INTEGRATION.md section 1).

1. one attention backward, every kernel family (dh 32 at 1-64 tokens, dh 64 at 17-256, fp32 and bf16, masked and not): dqkv bit-equal
   to avf_attention_bwd(_masked), G against the fp64 G of tests/relevance_oracle.py, exact zeros at (kept query, dropped key);
2. stacks at the SFormer, TFormer (T = 16, 128), AU_former and fusion-head geometries: dx bit-equal to the backward without maps and
   without weight gradients, every layer's G against fp64 (fp32) or within a per-row budget against the bf16 emulation (bf16);
3. the rollout kernel against fp64 within the fp32 summation bound of relevance_oracle.rollout_bound;
4. the model against the fp64 oracle model with retained attention gradients, for an AU index, a [12] and a [B, 12] weight;
5. no side effects; 6. errors."""
import os
import sys

import pytest
import torch

import avformer_b200 as A
from oracle import avformer_oracle as O

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import bf16_bwd_oracle as BB  # noqa: E402
import bf16_oracle as B  # noqa: E402
import relevance_oracle as RO  # noqa: E402

pytestmark = pytest.mark.gpu
AF = A.functional
N_FIELDS = len(AF.LayerWeights._fields_)

# bf16 stacks: worst_row(kernel) <= K_GMAP * worst_row(emulation), the median row within MEDIAN_RATIO of the emulation's.
# K_GMAP = 1.5 x the largest kernel / emulation ratio over the bf16 cases of test_stack_gradmaps, measured on one B200 (1000 W limit,
# 1965 MHz max SM clock) by tools/gradmap_budget_ratios.py: 1.371 (AU_former, masked); median-row ratios 0.99-1.02
# (profiles/r13_gradmap_budget_ratios.json).
K_GMAP = 2.06
MEDIAN_RATIO = (0.5, 2.0)


@pytest.fixture(autouse=True)
def _deterministic():
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    old = torch.backends.cudnn.deterministic, torch.backends.cudnn.benchmark
    torch.backends.cudnn.deterministic, torch.backends.cudnn.benchmark = True, False
    yield
    torch.backends.cudnn.deterministic, torch.backends.cudnn.benchmark = old


def _keep(n_seq, n_tok, seed):
    """Random keep rows (token 0 kept); sequence 1 keeps token 0 only, sequence 2 drops every token."""
    g = torch.Generator().manual_seed(seed)
    k = torch.rand(n_seq, n_tok, generator=g) < 0.6
    k[:, 0] = True
    k[1, 1:] = False
    k[2] = False
    return k


def _rel_err(got, ref):
    return ((got.double().cpu() - ref).abs().max() / ref.abs().max().clamp(min=1e-300)).item()


def _check_mask_zeros(g, keep):
    """A kept query gets exactly 0.0 on a dropped key (P is exactly 0 there)."""
    if keep is None:
        return
    gg = g.cpu()
    sel = keep[:, None, :, None].expand_as(gg) & ~keep[:, None, None, :].expand_as(gg)
    assert bool((gg[sel] == 0.0).all()), "a kept query has a nonzero G on a dropped key"


# ---------------------------------------------------------------------------------------------
# 1. one attention backward, every kernel family
# ---------------------------------------------------------------------------------------------
SHAPES = [(32, n) for n in (1, 12, 17, 33, 49, 64)] + [(64, n) for n in (17, 64, 65, 129, 256)]


@pytest.mark.parametrize("dh,n_tok", SHAPES)
@pytest.mark.parametrize("masked", [False, True])
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_attention_gradmaps(dh, n_tok, masked, dtype):
    torch.manual_seed(dh * 1000 + n_tok)
    n_seq, heads = 5, 8
    qkv = torch.randn(n_seq * n_tok, 3 * heads * dh, device="cuda").to(dtype)
    dout = torch.randn(n_seq * n_tok, heads * dh, device="cuda").to(dtype)
    keep = _keep(n_seq, n_tok, n_tok + dh) if masked else None
    kc = keep.cuda() if masked else None
    dqkv, g = AF.attention_bwd_gradmaps(qkv, dout, n_seq, n_tok, heads, dh, kc)
    assert g.shape == (n_seq, heads, n_tok, n_tok) and g.dtype == torch.float32 and g.is_contiguous()
    assert torch.equal(dqkv, AF.attention_bwd(qkv, dout, n_seq, n_tok, heads, dh, kc)), "dqkv of the map-writing launch differs"
    # The operands are exact in fp64 (bf16 ones too), and G is formed before anything is rounded, so both modes carry fp32 arithmetic
    # only: the fp32 scores and dP (dh-term sums) and the softmax, each a few 1e-6 relative.  The project's gradient tolerance, 1e-4 of
    # the tensor's max-abs, holds for both; a wrong key, row or head, or dS in place of P dP, moves G by its own size.
    ref = RO.gmap(qkv.double().cpu(), dout.double().cpu(), n_seq, n_tok, heads, dh, keep)
    err = _rel_err(g, ref)
    assert err <= 1e-4, f"max |G - G64| / max |G64| = {err:.3e}"
    _check_mask_zeros(g, keep)


# ---------------------------------------------------------------------------------------------
# 2. stacks
# ---------------------------------------------------------------------------------------------
GEOMS = {"sformer": (256, 1, 8, 32, 512, 49), "tformer16": (512, 3, 8, 64, 1024, 17), "tformer128": (512, 3, 8, 64, 1024, 129),
         "au_former": (128, 2, 8, 32, 256, 12), "fusion_head": (256, 3, 8, 32, 256, 12)}


def _stack(name, precision, seed=3):
    dim, depth, heads, dh, mlp, n_tok = GEOMS[name]
    p = O.params_from_spec(list(O._encoder_spec("", dim, depth, heads * dh, mlp)), seed)
    m = A.Transformer(dim, depth, heads, dh, mlp)
    m.load_state_dict(p, strict=True)
    m.precision = precision
    return m.cuda().eval(), {k: v.double() for k, v in p.items()}, n_tok


def stack_case(name, masked, precision):
    """Kernel and references of one stack case: (G kernel, G fp64, G emulated | None, keep)."""
    m, p64, n_tok = _stack(name, precision)
    n_seq = 4 if n_tok > 64 else 6
    g = torch.Generator().manual_seed(n_tok + 7 * masked)
    x = torch.randn(n_seq, n_tok, m.dim, generator=g)
    dy = BB.make_dy(n_seq * n_tok, m.dim, g).reshape(n_seq, n_tok, m.dim)
    keep = _keep(n_seq, n_tok, 11) if masked else None
    if masked:
        keep[:, 0] = True                                      # the module mask always keeps the first token (AF.keep_from_mask)
    mask = keep[:, 1:].cuda() if masked else None
    xc, dyc = x.cuda(), dy.cuda()
    y, gm, R = m.attention_relevance(xc, dyc, mask)
    kc = None if keep is None else keep.cuda()
    shape = m.shape(n_seq, n_tok)
    with torch.no_grad():
        y2, tape = AF.encoder_stack_fwd_train(xc.reshape(-1, m.dim), m.packed(), shape, keep=kc)
        assert torch.equal(y.reshape(-1, m.dim), y2), "y differs from the tape-keeping forward"
        d_ref = dyc.reshape(-1, m.dim).clone()
        AF.encoder_stack_bwd_(d_ref, m.packed(), shape, tape, [False] * (N_FIELDS * m.depth), keep=kc)
        d_new = dyc.reshape(-1, m.dim).clone()
        gm2 = AF.encoder_stack_bwd_gradmaps_(d_new, m.packed(), shape, tape, kc)
    assert torch.equal(d_new, d_ref), "dx of the map-writing backward differs"
    assert torch.equal(gm2, gm) and torch.equal(R, AF.attention_rollout(gm))
    assert gm.shape == (m.depth, n_seq, m.heads, n_tok, n_tok) and R.shape == (n_seq, n_tok, n_tok)
    _, g64 = RO.stack_gmaps(x.double(), p64, dy.double(), m.depth, m.heads, keep)
    emu = RO.stack_gmaps(x.double(), p64, dy.double(), m.depth, m.heads, keep, path="per_op")[1] if precision == "bf16" else None
    return gm, g64, emu, keep


def gmap_ratios(gm, g64, emu):
    """(worst-row ratio, median-row ratio) of the kernel's per-row RMS error against the emulation's (rows of G: one query of one
    head of one sequence of one layer), the emulation's error floored at 1e-6 of the reference's RMS (bf16_bwd_oracle.unit_floor)."""
    got, exp = B.row_rms(gm.double().cpu() - g64), B.row_rms(emu - g64).clamp(min=BB.unit_floor(g64))
    return (got.max() / exp.max()).item(), (got.median() / exp.median()).item()


@pytest.mark.parametrize("name", list(GEOMS))
@pytest.mark.parametrize("masked", [False, True])
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_stack_gradmaps(name, masked, precision):
    gm, g64, emu, keep = stack_case(name, masked, precision)
    for l in range(gm.shape[0]):
        _check_mask_zeros(gm[l], keep)
    if precision == "fp32":
        for l in range(gm.shape[0]):
            err = _rel_err(gm[l], g64[l])
            assert err <= 1e-4, f"layer {l}: max |G - G64| / max |G64| = {err:.3e}"
        return
    worst, median = gmap_ratios(gm, g64, emu)
    print(f"\ngradmaps {name} masked={masked}: worst-row ratio {worst:.3f}, median-row ratio {median:.3f}")
    assert MEDIAN_RATIO[0] <= median <= MEDIAN_RATIO[1], f"median-row ratio {median:.3f}: the emulation does not model the kernel"
    assert worst <= K_GMAP, f"worst row {worst:.3f} x the emulation's (budget {K_GMAP})"


# ---------------------------------------------------------------------------------------------
# 3. rollout
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n_tok", [12, 17, 49, 129, 256])
@pytest.mark.parametrize("depth", [1, 2, 3])
def test_rollout(n_tok, depth):
    g = torch.Generator().manual_seed(n_tok * 10 + depth)
    gm = (torch.randn(depth, 3, 8, n_tok, n_tok, generator=g) * 4.0 / n_tok).cuda()
    r = AF.attention_rollout(gm)
    assert r.shape == (3, n_tok, n_tok) and r.dtype == torch.float32
    g64 = gm.double().cpu()
    r64 = RO.rollout(g64)
    excess = ((r.double().cpu() - r64).abs() / RO.rollout_bound(g64, r64)).max().item()
    assert excess <= 1.0, f"rollout error {excess:.3f} x the fp32 summation bound"
    assert torch.equal(r, AF.attention_rollout(gm)), "the rollout is not deterministic"


# ---------------------------------------------------------------------------------------------
# 4. the model
# ---------------------------------------------------------------------------------------------
ORDER = (("sformer", 1), ("tformer", 3), ("video_au_former", 2), ("audio_au_former", 2), ("fusion_head", 3))   # softmax calls


def _model(seed, T, precision):
    m = A.TwoStreamAuralVisualFormer(video_pretrained=False, audio_pretrained=False, task="AU").set_clip_length(T)
    sd = O.make_state_dict(seed, T)
    m.load_state_dict(sd, strict=True)
    return m.cuda().eval().set_precision(precision), sd


def _oracle_relevance(sd, clip, audio, w):
    """{name: G [depth, n_seq, 8, n, n]} of the fp64 oracle model (on the GPU) seeded with d logits = w."""
    p = {k: v.double().cuda() for k, v in sd.items()}
    _, gs = RO.oracle_gmaps(O.avformer_forward, lambda out: (out["logits"] * w).sum(), clip.double(), audio.double(), p)
    res, i = {}, 0
    for name, depth in ORDER:
        res[name] = torch.stack(gs[i:i + depth])
        i += depth
    return res


MODEL_CASES = [(4, 8, "fp32"), (4, 16, "bf16"), (6, 16, "fp32"), (4, 32, "bf16")]
# max |G - G64| <= tol * max |G64| per stack.  fp32: the project's gradient tolerance (measured <= 3.2e-6 on one B200).  bf16: the
# stacks' bf16 operands compound over the fusion head, an AU_former and the TFormer (measured <= 8.3e-3).  The SFormer's gradient
# also passes through torch's fp32 convolution backward of stage 4 (cuDNN), which on one B200 was measured 1.5e-2 of max-abs off the
# fp64 d(sformer_out) at 32 frames (8e-6 at 96); its own kernels are held to 1e-4 in test_stack_gradmaps.
MODEL_TOL = {"fp32": 1e-4, "bf16": 3e-2}
SFORMER_TOL = {"fp32": 3e-2, "bf16": 1.5e-1}


@pytest.mark.parametrize("bs,T,precision", MODEL_CASES)
def test_model_relevance(bs, T, precision):
    seed = 5 + T
    m, sd = _model(seed, T, precision)
    clip, audio, _ = O.synth_inputs(seed, bs, T)
    x = {"clip": clip.cuda(), "audio_features": audio.cuda()}
    with torch.enable_grad():
        ref = m._forward_train(x["clip"], x["audio_features"]).detach()
    g = torch.Generator().manual_seed(seed)
    targets = {"au": 3, "vector": torch.randn(12, generator=g), "matrix": torch.randn(bs, 12, generator=g)}
    for kind, au in targets.items():
        out, rel = m.attention_relevance(x, au)
        assert torch.equal(out, ref), f"{kind}: out21 differs from _forward_train"
        w = torch.zeros(bs, 12) if kind == "au" else au.expand(bs, 12).double()
        if kind == "au":
            w[:, 3] = 1.0
            out1, rel1 = m.attention_relevance(x, w.cuda())
            assert all(torch.equal(rel[n][0], rel1[n][0]) and torch.equal(rel[n][1], rel1[n][1]) for n in rel), "au=j differs from one-hot"
        ref_g = _oracle_relevance(sd, x["clip"], x["audio_features"], w.double().cuda())
        errs = {}
        for name, (gm, R) in rel.items():
            assert gm.shape == ref_g[name].shape, name
            assert torch.equal(R, AF.attention_rollout(gm))
            errs[name] = _rel_err(gm, ref_g[name].cpu())
        print(f"\nmodel {precision} B={bs} T={T} {kind}: max |G - G64| / max |G64| " + ", ".join(f"{k} {v:.3e}" for k, v in errs.items()))
        for name, err in errs.items():
            assert err <= (SFORMER_TOL if name == "sformer" else MODEL_TOL)[precision], f"{kind} {name}: {err:.3e}"
    if precision == "fp32":
        # clip independence: the first two clips alone give their maps of the whole batch, within fp32 tolerance
        sub = {k: v[:2] for k, v in x.items()}
        w = targets["matrix"]
        _, rel_all = m.attention_relevance(x, w)
        _, rel_sub = m.attention_relevance(sub, w[:2])
        for name, (gm, _) in rel_sub.items():
            n = gm.shape[1]
            err = _rel_err(gm, rel_all[name][0][:, :n].double().cpu())
            assert err <= (SFORMER_TOL if name == "sformer" else MODEL_TOL)["fp32"], f"{name}: clip 0-1 maps depend on the other clips ({err:.3e})"


def test_model_relevance_stack_selection():
    m, _ = _model(2, 8, "bf16")
    clip, audio, _ = O.synth_inputs(2, 3, 8)
    x = {"clip": clip.cuda(), "audio_features": audio.cuda()}
    out_all, rel_all = m.attention_relevance(x, 0)
    shapes = {"sformer": (1, 24, 8, 49, 49), "tformer": (3, 3, 8, 9, 9), "audio_au_former": (2, 3, 8, 12, 12),
              "video_au_former": (2, 3, 8, 12, 12), "fusion_head": (3, 3, 8, 12, 12)}
    assert {k: tuple(v[0].shape) for k, v in rel_all.items()} == shapes
    assert {k: tuple(v[1].shape) for k, v in rel_all.items()} == {k: (s[1], s[3], s[4]) for k, s in shapes.items()}
    for stacks in (["tformer"], ["audio_au_former"], []):
        out, rel = m.attention_relevance(x, 0, stacks)
        assert torch.equal(out, out_all) and set(rel) == set(stacks)
        for n in stacks:
            assert torch.equal(rel[n][0], rel_all[n][0]) and torch.equal(rel[n][1], rel_all[n][1])


def test_tformer_relevance():
    m, _ = _model(4, 16, "bf16")
    tf = m.video_model.video_model.t_former
    frames = torch.randn(3 * 16, 512, device="cuda")
    d_cls = torch.randn(3, 512, device="cuda")
    mask = torch.rand(3, 16, device="cuda") < 0.7
    cls, gm, R = tf.attention_relevance(frames, d_cls, mask)
    with torch.enable_grad():
        ref = tf(frames.requires_grad_(True), mask)
    assert torch.equal(cls, ref.detach()), "cls differs from forward() with autograd"
    assert gm.shape == (3, 3, 8, 17, 17) and R.shape == (3, 17, 17)
    # the encoder stack on the embedded tokens, seeded with d_cls on the cls rows: the same maps and rollout, bit for bit
    tok = AF.tformer_embed(frames.detach(), tf.cls_token.detach().view(-1), tf.pos_embedding.detach()[0], 16).view(3, 17, 512)
    dy = torch.zeros_like(tok)
    dy[:, 0] = d_cls
    y, gm2, R2 = tf.spatial_transformer.attention_relevance(tok, dy, mask)
    assert torch.equal(y[:, 0], cls) and torch.equal(gm2, gm) and torch.equal(R2, R)
    # the last layer's rows 1..T reach nothing the cls row reads: their dO, and so their G, is exactly 0; the cls row is not
    assert not gm[-1, :, :, 1:].any() and gm[-1, :, :, 0].any()
    _check_mask_zeros(gm[-1], AF.keep_from_mask(mask, 3, 17).cpu())


# ---------------------------------------------------------------------------------------------
# 5. no side effects
# ---------------------------------------------------------------------------------------------
def test_model_relevance_no_side_effects():
    m, _ = _model(6, 8, "bf16")
    clip, audio, labels = O.synth_inputs(6, 3, 8)
    x = {"clip": clip.cuda(), "audio_features": audio.cuda()}
    opt = A.FusedAdam(m.parameters(), lr=1e-4)
    loss = m.get_au_loss(m(x), labels.cuda())             # one step: FusedAdam builds its bucket and the .grad views
    loss.backward()
    opt.step()
    m.eval()
    params = list(m.parameters())
    grads = [None if p.grad is None else p.grad.clone() for p in params]
    bucket = [t.clone() for b in opt._buckets if b for t in b.values() if torch.is_tensor(t)]
    bufs = {k: v.clone() for k, v in m.named_buffers()}
    versions = [p._version for p in params]
    for grad_mode in (True, False):
        with torch.set_grad_enabled(grad_mode):
            out, rel = m.attention_relevance(x, 1)
        assert out.grad_fn is None and all(g.grad_fn is None and r.grad_fn is None for g, r in rel.values())
    assert all((a is None and p.grad is None) or torch.equal(a, p.grad) for a, p in zip(grads, params)), ".grad changed"
    after = [t for b in opt._buckets if b for t in b.values() if torch.is_tensor(t)]
    assert len(after) == len(bucket) and all(torch.equal(a, b) for a, b in zip(bucket, after)), "the FusedAdam bucket changed"
    assert all(torch.equal(v, bufs[k]) for k, v in m.named_buffers()), "a buffer (BatchNorm statistics) changed"
    assert [p._version for p in params] == versions, "a parameter was modified"
    # the reference's frozen sub-models (models/avformer.py:78-85)
    for p in list(m.video_model.parameters()) + list(m.audio_model.parameters()):
        p.requires_grad_(False)
    out2, rel2 = m.attention_relevance(x, 1)
    assert torch.equal(out2, out) and all(torch.equal(rel2[n][0], rel[n][0]) for n in rel)


# ---------------------------------------------------------------------------------------------
# 6. errors
# ---------------------------------------------------------------------------------------------
def test_relevance_errors():
    m, _ = _model(7, 8, "bf16")
    clip, audio, _ = O.synth_inputs(7, 2, 8)
    x = {"clip": clip.cuda(), "audio_features": audio.cuda()}
    for bad in (12, -1, torch.randn(11), torch.randn(3, 12), torch.zeros(12, dtype=torch.long), "3", True):
        with pytest.raises(ValueError, match="au"):
            m.attention_relevance(x, bad)
    with pytest.raises(ValueError, match="unknown stack"):
        m.attention_relevance(x, 0, ["tformer", "s_former"])
    with pytest.raises(RuntimeError, match="CPU fallback"):
        m.attention_relevance({"clip": clip, "audio_features": audio}, 0)
    m.video_model.video_model.s_former.layer4.train()
    with pytest.raises(RuntimeError, match=r"eval\(\)"):
        m.attention_relevance(x, 0)
    m.eval()
    st = m.au_head.corr_transformer
    st.train()
    with pytest.raises(RuntimeError, match=r"eval\(\)"):
        st.attention_relevance(torch.randn(2, 12, 256, device="cuda"), torch.randn(2, 12, 256, device="cuda"))
    tf = m.video_model.video_model.t_former
    tf.train()
    with pytest.raises(RuntimeError, match=r"eval\(\)"):
        tf.attention_relevance(torch.randn(16, 512, device="cuda"), torch.randn(2, 512, device="cuda"))
