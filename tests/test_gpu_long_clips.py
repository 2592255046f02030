"""Long clips: TFormer attention of 65..256 tokens (T up to 255) with 64-wide heads, forward and backward, fp32 and bf16, masked and
gathered from a frame bank.

1. one attention against fp64 (tolerances of tests/test_gpu_masks.py), an all-kept mask bit for bit the unmasked call, and the dQ / dK
   of a dropped token exactly 0;
2. bf16 per-row budgets (tests/bf16_oracle.py, tests/bf16_bwd_oracle.py) for stacks of the TFormer's geometry at 65, 129, 256 tokens;
3. the TFormer at T in {64, 100, 128, 255} against the fp64 oracle, forward (cls_features: the last layer's attention computes the
   cls query only) and every gradient;
4. a T = 128 TFormer whose clips keep their first k frames against a T = k TFormer on those frames: the new kernels against the
   <= 64-token kernels the suite already trusts;
5. the frame-bank paths at T = 128 bit for bit against the explicit gather, and the engine / model entry points after
   set_clip_length(128);
6. the limits' errors."""
import ctypes
import os
import sys

import pytest
import torch

import avformer_b200 as A
from oracle import avformer_oracle as O

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import bf16_bwd_oracle as BB  # noqa: E402
import bf16_oracle as B  # noqa: E402

pytestmark = pytest.mark.gpu
AF = A.functional
DIM = 512
LONG_NTOK = [65, 80, 128, 129, 200, 256]
MEDIAN_RATIO = (0.5, 2.0)


@pytest.fixture(autouse=True)
def _no_tf32():
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False


def _rel(a, b):
    b = b.double().cpu()
    return (a.double().cpu() - b).abs().max().item() / max(b.abs().max().item(), 1e-30)


def _keep(n_seq, n_tok, seed):
    """Random keep rows (token 0 kept); sequence 1 keeps token 0 only, sequence 2 drops every token."""
    g = torch.Generator().manual_seed(seed)
    k = torch.rand(n_seq, n_tok, generator=g) < 0.6
    k[:, 0] = True
    k[1, 1:] = False
    k[2] = False
    return k


def _att_ref(qkv, n_seq, n_tok, heads, dh, keep):
    q, k, v = (t.reshape(n_seq, n_tok, heads, dh).permute(0, 2, 1, 3) for t in qkv.chunk(3, dim=-1))
    dots = q @ k.transpose(-1, -2) * dh ** -0.5
    if keep is not None:
        dots = dots.masked_fill(~(keep[:, None, :, None] & keep[:, None, None, :]), -torch.finfo(dots.dtype).max)
    return (torch.softmax(dots, dim=-1) @ v).permute(0, 2, 1, 3).reshape(n_seq * n_tok, heads * dh)


# ---------------------------------------------------------------------------------------------
# 1. one attention
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n_tok", LONG_NTOK)
@pytest.mark.parametrize("masked", [False, True])
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_long_attention_forward(n_tok, masked, dtype):
    torch.manual_seed(n_tok)
    n_seq, heads, dh = 5, 8, 64
    qkv = torch.randn(n_seq * n_tok, 3 * heads * dh, device="cuda").to(dtype)
    keep = _keep(n_seq, n_tok, n_tok) if masked else None
    got = AF.attention_fwd(qkv, n_seq, n_tok, heads, dh, keep.cuda() if masked else None)
    ref = _att_ref(qkv.double().cpu(), n_seq, n_tok, heads, dh, keep)
    assert torch.isfinite(got).all()
    assert _rel(got, ref) < (1e-5 if dtype == torch.float32 else 2 ** -7)
    if masked:
        everything = torch.ones(n_seq, n_tok, dtype=torch.bool, device="cuda")
        assert torch.equal(AF.attention_fwd(qkv, n_seq, n_tok, heads, dh, everything), AF.attention_fwd(qkv, n_seq, n_tok, heads, dh))


@pytest.mark.parametrize("n_tok", LONG_NTOK)
@pytest.mark.parametrize("masked", [False, True])
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_long_attention_backward(n_tok, masked, dtype):
    """dq, dk, dv against fp64 autograd; the loss covers every row, so the uniform rows of dropped queries feed dV."""
    torch.manual_seed(n_tok + 1)
    n_seq, heads, dh = 4, 8, 64
    inner = heads * dh
    qkv = torch.randn(n_seq * n_tok, 3 * inner, device="cuda").to(dtype)
    dout = torch.randn(n_seq * n_tok, inner, device="cuda").to(dtype)
    keep = _keep(n_seq, n_tok, n_tok * 7) if masked else None
    q = qkv.double().cpu().requires_grad_(True)
    _att_ref(q, n_seq, n_tok, heads, dh, keep).backward(dout.double().cpu())
    got = AF.attention_bwd(qkv, dout, n_seq, n_tok, heads, dh, keep.cuda() if masked else None)
    assert torch.isfinite(got).all()
    assert _rel(got.float(), q.grad) < (1e-5 if dtype == torch.float32 else 2 ** -7)
    if masked:
        dropped = ~keep.reshape(-1)
        assert not bool(got[dropped.cuda(), :2 * inner].any()), "dQ / dK of a dropped token is not 0"
        everything = torch.ones(n_seq, n_tok, dtype=torch.bool, device="cuda")
        assert torch.equal(AF.attention_bwd(qkv, dout, n_seq, n_tok, heads, dh, everything), AF.attention_bwd(qkv, dout, n_seq, n_tok, heads, dh))


# ---------------------------------------------------------------------------------------------
# 2. bf16 per-row budgets at the TFormer's geometry
# ---------------------------------------------------------------------------------------------
BUDGET_NTOK = [65, 129, 256]


def _fwd_case(n_tok):
    return dict(name=f"rows-d512-t{n_tok}", kind="rows", dim=512, dh=64, n_tok=n_tok, depth=3, mlp=1024, n_seq=6, sample=None)


@pytest.mark.parametrize("n_tok", BUDGET_NTOK)
def test_long_stack_forward_within_bf16_budget(n_tok):
    case = _fwd_case(n_tok)
    p, x, pos = B.make_inputs(case)
    m = A.Transformer(DIM, 3, 8, 64, 1024)
    m.load_state_dict(p, strict=True)
    m.precision = "bf16"
    m = m.cuda().eval()
    shape = m.shape(case["n_seq"], n_tok)
    assert not AF.encoder_fused_supported(shape)
    with torch.no_grad():
        y = AF.token_stack_fwd_(x.cuda(), m.packed(), shape, pos.cuda()).view(case["n_seq"], n_tok, DIM)
    ref, _, emu, _, _ = B.references(case)
    got, exp = B.row_rms(y.double().cpu() - ref), B.row_rms(emu - ref)
    worst, median = (got.max() / exp.max()).item(), (got.median() / exp.median()).item()
    print(f"\n{case['name']}: worst-row ratio {worst:.3f}, median-row ratio {median:.3f}")
    assert MEDIAN_RATIO[0] <= median <= MEDIAN_RATIO[1], f"median-row ratio {median:.3f}: the emulation does not model the kernel"
    assert worst <= B.K, f"worst row {worst:.3f} x the emulation's (budget {B.K})"


def _check_bwd(ratios, label):
    for k, (worst, median) in ratios.items():
        assert worst <= BB.K_BWD, f"{label} {k}: worst unit {worst:.3f} x the emulation's (budget {BB.K_BWD})"
        if median is not None:
            lo, hi = BB.MEDIAN_RATIO
            assert lo <= median <= hi, f"{label} {k}: median-unit ratio {median:.3f}: the emulation does not model the kernel"


@pytest.mark.parametrize("n_tok", BUDGET_NTOK)
@pytest.mark.parametrize("masked", [False, True])
def test_long_attention_bwd_within_bf16_budget(n_tok, masked):
    case = dict(name=f"att-{'m' if masked else 'u'}-dh64-t{n_tok}", kind="att", dh=64, heads=8, n_tok=n_tok, n_seq=12, masked=masked)
    qkv, dout, keep = BB.att_inputs(case)
    got = AF.attention_bwd(qkv.cuda(), dout.cuda(), case["n_seq"], n_tok, 8, 64, keep=keep.cuda() if keep is not None else None).double().cpu()
    ref, emu = BB.att_references(case)
    if keep is not None:
        assert not bool(got[~keep.reshape(-1), :2 * 512].any()), "dQ / dK of a dropped token is not 0"
    _check_bwd({"dqkv": BB.ratios("dqkv", got, emu, ref, 8)}, case["name"])


@pytest.mark.parametrize("n_tok,masked", [(65, False), (129, True), (256, False)])
def test_long_stack_bwd_within_bf16_budget(n_tok, masked):
    case = BB._stack(f"d512-t{n_tok}{'-masked' if masked else ''}", DIM, 64, 3, 1024, n_tok, 6, masked=masked)
    p, x, dy, keep = BB.stack_inputs(case)
    m = A.Transformer(DIM, 3, 8, 64, 1024)
    m.load_state_dict(p, strict=True)
    m.precision = "bf16"
    m = m.cuda()
    packed, shape = m.packed(), m.shape(case["n_seq"], n_tok)
    kc = keep.cuda() if keep is not None else None
    _, tape = AF.encoder_stack_fwd_train(x.cuda(), packed, shape, keep=kc)
    dx, grads = AF.encoder_stack_bwd_(dy.cuda().clone(), packed, shape, tape, [True] * 33, keep=kc)
    got = {"dx": dx}
    got.update(zip(BB.grad_names(3), grads))
    ref = BB.stack_reference(case, device="cuda")
    emu = BB.stack_reference(case, path="per_op", device="cuda")
    _check_bwd(BB.stack_ratios(got, emu, ref), case["name"])


# ---------------------------------------------------------------------------------------------
# 3. the TFormer against the fp64 oracle
# ---------------------------------------------------------------------------------------------
def _tformer(T, precision, seed):
    p = O.params_from_spec([("cls_token", (1, 1, DIM), "normal"), ("pos_embedding", (1, T + 1, DIM), "normal")]
                           + list(O._encoder_spec("spatial_transformer.", DIM, 3, 512, 1024)), seed)
    tf = A.TFormer(num_patches=T).cuda().eval()
    tf.load_state_dict(p, strict=True)
    tf.spatial_transformer.precision = precision
    return tf, {k: v.double() for k, v in p.items()}


def _cls_stack(frames, p, T, keep, path):
    """The TFormer's cls rows in fp64 (path None) or with the bf16 rounding of the per-op path ("per_op"); ``keep`` [n_clips, T] bool
    frames kept (None: all)."""
    x = frames.double().reshape(-1, T, DIM)
    n = x.shape[0]
    x = torch.cat([p["cls_token"].expand(n, -1, -1), x], dim=1) + p["pos_embedding"][:, :T + 1]
    k = None if keep is None else torch.nn.functional.pad(keep, (1, 0), value=True)
    sp = {key[len("spatial_transformer."):]: v for key, v in p.items() if key.startswith("spatial_transformer.")}
    for l in range(3):
        a, f = f"layers.{l}.0.", f"layers.{l}.1."
        x = x + B._attention(B._layer_norm(x, sp[a + "fn.norm.weight"], sp[a + "fn.norm.bias"], path), sp, a, 8, path, None, keep=k)
        x = x + B._feed_forward(B._layer_norm(x, sp[f + "fn.norm.weight"], sp[f + "fn.norm.bias"], path), sp, f, path)
    return x[:, 0]


def _frame_mask(n_clips, T, seed):
    g = torch.Generator().manual_seed(seed)
    m = torch.rand(n_clips, T, generator=g) < 0.7
    m[0] = True
    m[1] = False
    m[2, 1:] = False
    return m


def _cls_within_budget(got, frames, p, T, keep):
    ref = _cls_stack(frames, p, T, keep, None)
    emu = _cls_stack(frames, p, T, keep, "per_op")
    ratio = (B.row_rms(got.double().cpu() - ref).max() / B.row_rms(emu - ref).max()).item()
    return ratio


@pytest.mark.parametrize("T", [64, 100, 128, 255])
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_long_tformer_cls_features_against_oracle(T, precision):
    n_clips = 6
    tf, p = _tformer(T, precision, 500 + T)
    frames = torch.randn(n_clips * T, DIM, generator=torch.Generator().manual_seed(T))
    mask = _frame_mask(n_clips, T, T)
    with torch.no_grad():
        plain = tf.cls_features(frames.cuda())
        masked = tf.cls_features(frames.cuda(), mask.cuda())
        every = tf.cls_features(frames.cuda(), torch.ones(n_clips, T, dtype=torch.bool, device="cuda"))
    assert torch.isfinite(plain).all() and torch.isfinite(masked).all()
    if precision == "fp32":
        assert _rel(plain, _cls_stack(frames, p, T, None, None)) < 1e-4
        assert _rel(masked, _cls_stack(frames, p, T, mask, None)) < 1e-4
        assert torch.equal(every, plain)
    else:
        for got, keep in ((plain, None), (masked, mask)):
            ratio = _cls_within_budget(got, frames, p, T, keep)
            assert ratio <= B.K, f"cls worst row {ratio:.3f} x the emulation's (budget {B.K})"


@pytest.mark.parametrize("T", [64, 100, 128, 255])
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_long_tformer_gradients_against_oracle(T, precision):
    n_clips = 4
    tf, p = _tformer(T, precision, 600 + T)
    g = torch.Generator().manual_seed(T + 1)
    frames = torch.randn(n_clips * T, DIM, generator=g)
    mask = _frame_mask(n_clips, T, T + 1)
    dcls = torch.randn(n_clips, DIM, generator=g)
    fr = frames.cuda().requires_grad_(True)
    tf.train()
    tf(fr, mask.cuda()).backward(dcls.cuda())
    pr = {k: v.clone().requires_grad_(True) for k, v in p.items()}
    frr = frames.double().requires_grad_(True)
    _cls_stack(frr, pr, T, mask, None).backward(dcls.double())
    tol = 1e-4 if precision == "fp32" else 3e-2
    assert _rel(fr.grad, frr.grad) < tol
    for k, v in tf.named_parameters():
        assert _rel(v.grad, pr[k].grad) < tol, k


# ---------------------------------------------------------------------------------------------
# 4. across the boundary: a T = 128 clip keeping k frames is a T = k clip
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("k", [16, 63])
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_prefix_mask_at_t128_equals_short_tformer(k, precision):
    T, n_clips = 128, 6
    tf, p = _tformer(T, precision, 700 + k)
    tfk = A.TFormer(num_patches=k).cuda().train()
    with torch.no_grad():
        tfk.cls_token.copy_(tf.cls_token)
        tfk.pos_embedding.copy_(tf.pos_embedding[:, :k + 1])
        for a, b in zip(tfk.spatial_transformer.parameters(), tf.spatial_transformer.parameters()):
            a.copy_(b)
    tfk.spatial_transformer.precision = precision
    tf.train()
    g = torch.Generator().manual_seed(k)
    frames = torch.randn(n_clips, T, DIM, generator=g)
    dcls = torch.randn(n_clips, DIM, generator=g).cuda()
    prefix = (torch.arange(T)[None, :] < k).expand(n_clips, T).contiguous()
    short_frames = frames[:, :k].reshape(-1, DIM)
    with torch.no_grad():
        inf_long = tf.cls_features(frames.reshape(-1, DIM).cuda(), prefix.cuda())
        inf_short = tfk.cls_features(short_frames.cuda())
    y_long = tf(frames.reshape(-1, DIM).cuda(), prefix.cuda())
    y_long.backward(dcls)
    y_short = tfk(short_frames.cuda())
    y_short.backward(dcls)
    pk = {n: v for n, v in p.items()}
    pk["pos_embedding"] = p["pos_embedding"][:, :k + 1]
    assert float(tf.pos_embedding.grad[:, k + 1:].abs().max()) == 0.0
    grads_long = {n: v.grad for n, v in tf.named_parameters()}
    grads_long["pos_embedding"] = grads_long["pos_embedding"][:, :k + 1]
    grads_short = {n: v.grad for n, v in tfk.named_parameters()}
    if precision == "fp32":
        assert _rel(inf_long, inf_short) < 1e-5
        assert _rel(y_long.detach(), y_short.detach()) < 1e-5
        for n in grads_short:
            assert _rel(grads_long[n], grads_short[n]) < 1e-5, n
    else:
        for got in (inf_long, inf_short, y_long.detach(), y_short.detach()):
            ratio = _cls_within_budget(got, short_frames, pk, k, None)
            assert ratio <= B.K, f"cls worst row {ratio:.3f} x the k-frame emulation's (budget {B.K})"
        pr = {n: v.clone().requires_grad_(True) for n, v in pk.items()}
        _cls_stack(short_frames, pr, k, None, None).backward(dcls.double().cpu())
        for n in grads_short:
            assert _rel(grads_long[n], pr[n].grad) < 3e-2, n
            assert _rel(grads_short[n], pr[n].grad) < 3e-2, n


# ---------------------------------------------------------------------------------------------
# 5. frame bank at T = 128
# ---------------------------------------------------------------------------------------------
def _tables(T, n_clips, F, seed):
    g = torch.Generator().manual_seed(seed)
    start = torch.randint(-T // 2, F - T // 2, (n_clips, 1), generator=g)
    raw = start + torch.arange(T)[None, :]
    return {"clamp": raw.clamp(0, F - 1), "minus1": torch.where((raw >= 0) & (raw < F), raw, torch.full_like(raw, -1))}


def _cpu_scatter(rows, idx, n_bank):
    acc = torch.zeros(n_bank, rows.shape[1], dtype=torch.float32)
    for s, i in enumerate(idx.reshape(-1).tolist()):
        if 0 <= i < n_bank:
            acc[i] = acc[i] + rows[s]
    return acc


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_bank_paths_at_t128_equal_explicit_gather(precision):
    T, n_clips, F = 128, 6, 300
    tf, _ = _tformer(T, precision, 800)
    for k, (name, idx) in enumerate(_tables(T, n_clips, F, 801).items()):
        bank = torch.randn(F, DIM, generator=torch.Generator().manual_seed(k)).cuda()
        mask = (idx >= 0).cuda()
        tf.eval()
        with torch.no_grad():
            got = tf.cls_features_indexed(bank, idx)
            ref = tf.cls_features(bank[idx.clamp(min=0).cuda()].reshape(-1, DIM), mask=mask)
        assert torch.equal(got, ref), name
        tf.train()
        w = torch.randn(n_clips, DIM, generator=torch.Generator().manual_seed(50 + k)).cuda()
        frames = bank[idx.clamp(min=0).cuda()].reshape(-1, DIM).requires_grad_(True)
        tf.zero_grad(set_to_none=True)
        cls_g = tf(frames, mask=mask)
        (cls_g * w).sum().backward()
        g_g = {n: v.grad.clone() for n, v in tf.named_parameters()}
        leaf = bank.clone().requires_grad_(True)
        tf.zero_grad(set_to_none=True)
        cls_i = tf.forward_indexed(leaf, idx)
        (cls_i * w).sum().backward()
        assert torch.equal(cls_i.detach(), cls_g.detach()), name
        for n, v in tf.named_parameters():
            assert torch.equal(v.grad, g_g[n]), (name, n)
        assert torch.equal(leaf.grad.cpu(), _cpu_scatter(frames.grad.cpu(), idx, F)), name


def _model(seed, T, precision):
    m = A.TwoStreamAuralVisualFormer(video_pretrained=False, audio_pretrained=False, task="AU").set_clip_length(T)
    m.load_state_dict(O.make_state_dict(seed, T), strict=True)
    return m.cuda().set_precision(precision)


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_engine_clips_and_model_training_step_at_t128(precision):
    T, F, n, seed = 128, 40, 3, 901
    m = _model(seed, T, precision).eval()
    frames = O.synth_inputs(seed, 1, F)[0][0].permute(1, 0, 2, 3).contiguous().cuda()          # [F, 3, 112, 112]
    raw = torch.tensor([[-60], [-20], [0]]) + torch.arange(T)[None, :]
    idx = raw.clamp(0, F - 1)
    audio = O.synth_inputs(seed + 1, n, 8)[1].cuda()
    eng = A.InferenceEngine(m, backbone_dtype=torch.float32)
    bank = eng.frame_features(frames)
    out21, dec = eng.clips(bank, idx, audio)
    with torch.no_grad():
        ref = m({"clip": frames[idx.cuda()].permute(0, 2, 1, 3, 4), "audio_features": audio})
    assert out21.shape == (n, 21) and torch.isfinite(out21).all()
    assert torch.equal(dec, (out21[:, :12] > 0).to(torch.int32))
    assert (out21[:, :12] - ref[:, :12]).abs().max().item() < (5e-3 if precision == "fp32" else 0.25)
    m.train()
    opt = A.FusedAdam(m.parameters(), lr=1e-4)
    labels = O.synth_inputs(seed, n, 8, image=8)[2].cuda()
    loss = m.get_au_loss(m.forward_indexed(frames, torch.where(raw >= 0, raw, torch.full_like(raw, -1)).clamp(max=F - 1), audio), labels)
    loss.backward()
    tp = m.video_model.video_model.t_former
    assert torch.isfinite(loss) and all(torch.isfinite(q.grad).all() for q in tp.parameters())
    assert float(tp.pos_embedding.grad.abs().max()) > 0
    opt.step()
    assert all(torch.isfinite(q).all() for q in m.parameters())


# ---------------------------------------------------------------------------------------------
# 6. errors
# ---------------------------------------------------------------------------------------------
def test_long_clip_limits_are_loud():
    tf = A.TFormer(num_patches=256).cuda().eval()
    with pytest.raises(RuntimeError, match="256"), torch.no_grad():
        tf.cls_features(torch.zeros(256, DIM, device="cuda"))
    tf.train()
    with pytest.raises(RuntimeError, match="256"):
        tf(torch.zeros(256, DIM, device="cuda", requires_grad=True))
    narrow = A.Transformer(256, 1, 8, 32, 256).cuda().eval()
    with pytest.raises(RuntimeError, match="sequences longer than 64 tokens"), torch.no_grad():
        narrow(torch.zeros(1, 65, 256, device="cuda"))
    with pytest.raises(RuntimeError, match="256"):
        AF.attention_fwd(torch.zeros(257, 3 * 512, device="cuda", dtype=torch.bfloat16), 1, 257, 8, 64)
    with pytest.raises(RuntimeError):
        AF.attention_fwd(torch.zeros(65, 3 * 256, device="cuda", dtype=torch.bfloat16), 1, 65, 8, 32)
    # the workspace and tape contracts at a long shape: too small -> AVF_EWORKSPACE, nothing computed
    L = A._lib.lib()
    tr = A.Transformer(DIM, 1, 8, 64, 1024).cuda()
    shape, packed = tr.shape(2, 129), tr.packed()
    need = L.avf_encoder_workspace_bytes(ctypes.byref(shape), packed.mode)
    ws = torch.empty(need - 256, dtype=torch.uint8, device="cuda")
    x = torch.zeros(2 * 129, DIM, device="cuda")
    rc = L.avf_encoder_stack_fwd(packed.mode, ctypes.byref(shape), packed.array, AF._ptr(x), DIM, None, 0, AF._ptr(ws), ws.numel(), AF._stream())
    assert rc == -3 and b"too small" in L.avf_last_error()
    tape_need = L.avf_encoder_tape_bytes(ctypes.byref(shape), packed.mode)
    tape = torch.empty(tape_need - 256, dtype=torch.uint8, device="cuda")
    out = torch.zeros_like(x)
    rc = L.avf_encoder_stack_fwd_train(packed.mode, ctypes.byref(shape), packed.array, AF._ptr(x), DIM, AF._ptr(out), DIM, AF._ptr(tape), tape.numel(),
                                       0.0, 0, None, AF._stream())
    assert rc == -3 and b"too small" in L.avf_last_error()
