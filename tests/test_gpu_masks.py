"""Attention masks on the CUDA path (Transformer.forward(x, mask), TFormer clips with fewer real frames), forward and backward,
against the literal fp64 masked_fill(-finfo.max) form of tests/masked_oracle.py (built on the oracle's primitives).

Tolerances: fp32 mode 1e-4 of each tensor's max-abs for stacks (1e-5 for one attention), bf16 mode the budgets of the unmasked
tests (2e-2 forward, 3e-2 gradients, 2^-7 for one attention).  An all-True mask must reproduce the unmasked kernels bit for bit."""
import os
import sys

import pytest
import torch

import avformer_b200 as A
from oracle import avformer_oracle as O

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import masked_oracle as M  # noqa: E402

pytestmark = pytest.mark.gpu
AF = A.functional


@pytest.fixture(autouse=True)
def _no_tf32():
    torch.backends.cuda.matmul.allow_tf32 = False


def _rel(a, b):
    b = b.double().cpu()
    return (a.double().cpu() - b).abs().max().item() / max(b.abs().max().item(), 1e-30)


def _keep(n_seq, n_tok, seed):
    """Random non-prefix keep rows [n_seq, n_tok] (token 0 always kept), different per sequence; sequence 1 keeps the cls token only."""
    g = torch.Generator().manual_seed(seed)
    k = torch.rand(n_seq, n_tok, generator=g) < 0.6
    k[:, 0] = True
    k[1, 1:] = False
    return k


def _att_ref(qkv, n_seq, n_tok, heads, dh, keep):
    q, k, v = (t.reshape(n_seq, n_tok, heads, dh).permute(0, 2, 1, 3) for t in qkv.chunk(3, dim=-1))
    dots = q @ k.transpose(-1, -2) * dh ** -0.5
    dots = dots.masked_fill(~(keep[:, None, :, None] & keep[:, None, None, :]), -torch.finfo(dots.dtype).max)
    return (torch.softmax(dots, dim=-1) @ v).permute(0, 2, 1, 3).reshape(n_seq * n_tok, heads * dh)


# ---------------------------------------------------------------------------------------------
# one attention
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n_tok", [1, 2, 12, 17, 33, 49, 64])
@pytest.mark.parametrize("dh", [32, 64])
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_masked_attention_forward(n_tok, dh, dtype):
    torch.manual_seed(n_tok * dh)
    n_seq, heads = 6, 8
    qkv = torch.randn(n_seq * n_tok, 3 * heads * dh, device="cuda").to(dtype)
    keep = _keep(n_seq, n_tok, n_tok + dh)
    got = AF.attention_fwd(qkv, n_seq, n_tok, heads, dh, keep.cuda())
    ref = _att_ref(qkv.double().cpu(), n_seq, n_tok, heads, dh, keep)
    assert torch.isfinite(got).all()
    assert _rel(got, ref) < (1e-5 if dtype == torch.float32 else 2 ** -7)
    everything = torch.ones(n_seq, n_tok, dtype=torch.bool, device="cuda")
    assert torch.equal(AF.attention_fwd(qkv, n_seq, n_tok, heads, dh, everything), AF.attention_fwd(qkv, n_seq, n_tok, heads, dh))


@pytest.mark.parametrize("n_tok,dh", [(1, 32), (12, 32), (17, 64), (33, 64), (49, 32), (64, 32)])
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_masked_attention_backward(n_tok, dh, dtype):
    """dq, dk, dv against fp64 autograd; the loss covers every row, so the uniform rows of dropped queries feed dV."""
    torch.manual_seed(n_tok * dh + 1)
    n_seq, heads = 5, 8
    inner = heads * dh
    qkv = torch.randn(n_seq * n_tok, 3 * inner, device="cuda").to(dtype)
    dout = torch.randn(n_seq * n_tok, inner, device="cuda").to(dtype)
    keep = _keep(n_seq, n_tok, n_tok * 7 + dh)
    q = qkv.double().cpu().requires_grad_(True)
    _att_ref(q, n_seq, n_tok, heads, dh, keep).backward(dout.double().cpu())
    got = AF.attention_bwd(qkv, dout, n_seq, n_tok, heads, dh, keep.cuda())
    assert torch.isfinite(got).all()
    assert _rel(got.float(), q.grad) < (1e-5 if dtype == torch.float32 else 2 ** -7)


# ---------------------------------------------------------------------------------------------
# stacks
# ---------------------------------------------------------------------------------------------
STACKS = {512: dict(heads=8, dh=64, mlp=1024, depth=3, n_tok=17), 256: dict(heads=8, dh=32, mlp=256, depth=3, n_tok=12),
          128: dict(heads=8, dh=32, mlp=256, depth=2, n_tok=12)}


def _stack(dim, precision, seed, dropout=0.0):
    g = STACKS[dim]
    torch.manual_seed(seed)
    tr = A.Transformer(dim, g["depth"], g["heads"], g["dh"], g["mlp"], dropout=dropout).cuda().eval()
    tr.precision = precision
    with torch.no_grad():
        for q in tr.parameters():
            if q.dim() == 1:
                q.add_(torch.randn_like(q) * 0.1)
    return tr, {"t." + k: v.detach().double().cpu() for k, v in tr.named_parameters()}


def _mask(n_seq, n_tok, seed):
    m = _keep(n_seq, n_tok, seed)[:, 1:]          # the module's mask: [n_seq, n_tok - 1], the cls token is implied
    m[2] = False
    return m


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
@pytest.mark.parametrize("dim", [512, 256, 128])
def test_masked_transformer_against_oracle(dim, precision):
    tr, pr = _stack(dim, precision, dim)
    g = STACKS[dim]
    n_seq, n_tok = 40, g["n_tok"]
    x = torch.randn(n_seq, n_tok, dim, device="cuda")
    mask = _mask(n_seq, n_tok, dim)
    with torch.no_grad():
        y = tr(x, mask=mask.cuda())
    ref = M.transformer(x.double().cpu(), pr, "t.", g["depth"], g["heads"], mask)
    assert _rel(y, ref) < (1e-4 if precision == "fp32" else 2e-2)
    everything = torch.ones(n_seq, n_tok - 1, dtype=torch.bool, device="cuda")
    with torch.no_grad():
        y_all = tr(x, mask=everything)
        if dim in (256, 128):                       # the masked call never takes the fused kernel: compare with the kernel-per-op path
            prev = AF.set_fused_enabled(False)
            try:
                y_ref = tr(x)
            finally:
                AF.set_fused_enabled(prev)
        else:
            y_ref = tr(x)
    assert torch.equal(y_all, y_ref)


def test_masked_attention_module_against_oracle():
    torch.manual_seed(5)
    att = A.Attention(256, heads=8, dim_head=32).cuda()
    p = {"a.fn.fn." + k: v.detach().double().cpu() for k, v in att.named_parameters()}
    x = torch.randn(9, 12, 256, device="cuda")
    mask = _mask(9, 12, 5)
    with torch.no_grad():
        y = att(x, mask=mask.cuda())
    assert _rel(y, M.attention(x.double().cpu(), p, "a.", 8, mask)) < 2e-2


# ---------------------------------------------------------------------------------------------
# TFormer: clips with fewer real frames
# ---------------------------------------------------------------------------------------------
def _tformer(T, precision, seed):
    p = O.params_from_spec([("cls_token", (1, 1, 512), "normal"), ("pos_embedding", (1, T + 1, 512), "normal")]
                           + list(O._encoder_spec("spatial_transformer.", 512, 3, 512, 1024)), seed)
    tf = A.TFormer(num_patches=T).cuda().eval()
    tf.load_state_dict(p, strict=True)
    tf.spatial_transformer.precision = precision
    return tf, {"tf." + k: v.double() for k, v in p.items()}


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_masked_tformer_512_clips(precision):
    T, n_clips = 16, 512
    tf, p = _tformer(T, precision, 21)
    g = torch.Generator().manual_seed(22)
    frames = torch.randn(n_clips * T, 512, generator=g)
    lengths = torch.randint(1, T + 1, (n_clips,), generator=g)
    mask = torch.arange(T)[None, :] < lengths[:, None]
    with torch.no_grad():
        got = tf(frames.cuda(), mask.cuda())
    sub = torch.arange(0, n_clips, 8)                 # clips are independent: the fp64 oracle checks every 8th
    ref = M.tformer(frames.view(n_clips, T, 512)[sub].reshape(-1, 512).double(), p, "tf.", T, mask[sub])
    assert _rel(got[sub], ref) < (1e-4 if precision == "fp32" else 2e-2)
    # a clip of k real frames gives what TFormer(num_patches=k) gives on those frames (expected: bit-identical)
    for k in (1, 5, 12):
        tfk, _ = _tformer(k, precision, 21)
        with torch.no_grad():
            tfk.pos_embedding.copy_(tf.pos_embedding[:, : k + 1])
            prefix = torch.arange(T)[None, :].expand(n_clips, T) < k
            masked = tf(frames.cuda(), prefix.cuda())
            short = tfk(frames.view(n_clips, T, 512)[:, :k].reshape(-1, 512).cuda())
        diff = (masked - short).abs().max().item() / short.abs().max().item()
        print(f"TFormer[{precision}] prefix k={k}: max|masked - TFormer(num_patches=k)| / max|.| = {diff:.3e}")
        assert diff <= (1e-5 if precision == "fp32" else 1e-3)
    # cls_features stays one library call: the same launches as the unmasked call (the mask pad is a torch op)
    L = A._lib.lib()
    with torch.no_grad():
        n0 = L.avf_launch_count()
        tf.cls_features(frames.cuda())
        n1 = L.avf_launch_count()
        tf.cls_features(frames.cuda(), mask.cuda())
        n2 = L.avf_launch_count()
    assert n2 - n1 == n1 - n0


# ---------------------------------------------------------------------------------------------
# training
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
@pytest.mark.parametrize("dim", [512, 256])
def test_masked_transformer_gradients(dim, precision):
    tr, _ = _stack(dim, precision, dim + 1)
    g = STACKS[dim]
    n_seq, n_tok = 24, g["n_tok"]
    x = torch.randn(n_seq, n_tok, dim, device="cuda", requires_grad=True)
    dy = torch.randn(n_seq, n_tok, dim, device="cuda")
    mask = _mask(n_seq, n_tok, dim + 1)
    tr(x, mask=mask.cuda()).backward(dy)
    pr = {"t." + k: v.detach().double().cpu().requires_grad_(True) for k, v in tr.named_parameters()}
    xr = x.detach().double().cpu().requires_grad_(True)
    M.transformer(xr, pr, "t.", g["depth"], g["heads"], mask).backward(dy.double().cpu())
    tol = 1e-4 if precision == "fp32" else 3e-2
    assert _rel(x.grad, xr.grad) < tol
    for k, v in tr.named_parameters():              # all 11 weight kinds of every layer
        assert _rel(v.grad, pr["t." + k].grad) < tol, k


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_masked_tformer_gradients(precision):
    T, n_clips = 16, 32
    tf, p = _tformer(T, precision, 31)
    g = torch.Generator().manual_seed(32)
    frames = torch.randn(n_clips * T, 512, generator=g)
    lengths = torch.randint(1, T + 1, (n_clips,), generator=g)
    mask = torch.arange(T)[None, :] < lengths[:, None]
    dcls = torch.randn(n_clips, 512, generator=g)
    fr = frames.cuda().requires_grad_(True)
    tf(fr, mask.cuda()).backward(dcls.cuda())
    pr = {k: v.clone().requires_grad_(True) for k, v in p.items()}
    frr = frames.double().requires_grad_(True)
    M.tformer(frr, pr, "tf.", T, mask).backward(dcls.double())
    tol = 1e-4 if precision == "fp32" else 3e-2
    assert _rel(fr.grad, frr.grad) < tol
    for k, v in tf.named_parameters():
        assert _rel(v.grad, pr["tf." + k].grad) < tol, k


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_masked_transformer_with_dropout_against_oracle_with_the_same_masks(precision):
    dim, p_drop, seed = 256, 0.2, 123456789
    tr, _ = _stack(dim, precision, 77, dropout=p_drop)
    tr.train()
    tr.fixed_dropout_seed = seed
    g = STACKS[dim]
    n_seq, n_tok, depth = 9, g["n_tok"], g["depth"]
    x = torch.randn(n_seq, n_tok, dim, device="cuda", requires_grad=True)
    dy = torch.randn(n_seq, n_tok, dim, device="cuda")
    mask = _mask(n_seq, n_tok, 78)
    y = tr(x, mask=mask.cuda())
    y.backward(dy)
    R = n_seq * n_tok
    drops = {(l, s): AF.dropout_mask(p_drop, seed, l, s, R, g["mlp"] if s == 1 else dim, "cuda").double().cpu() for l in range(depth) for s in range(3)}
    pr = {"t." + k: v.detach().double().cpu().requires_grad_(True) for k, v in tr.named_parameters()}
    xr = x.detach().double().cpu().requires_grad_(True)
    yr = M.transformer(xr, pr, "t.", depth, g["heads"], mask, drops)
    yr.backward(dy.double().cpu())
    tol_y, tol_g = (1e-4, 1e-4) if precision == "fp32" else (2e-2, 3e-2)
    assert _rel(y, yr.detach()) < tol_y
    assert _rel(x.grad, xr.grad) < tol_g
    for k, v in tr.named_parameters():
        assert _rel(v.grad, pr["t." + k].grad) < tol_g, k


# ---------------------------------------------------------------------------------------------
# model level and errors
# ---------------------------------------------------------------------------------------------
def test_hot_path_with_frame_mask():
    T, B, seed = 16, 24, 41
    sd = O.make_state_dict(seed, T, hot_path_only=True)
    stage3, frame, audio = O.synth_hot_path_inputs(seed, B, T)
    m = A.TwoStreamAuralVisualFormer(video_pretrained=False, audio_pretrained=False, task="AU")
    m.load_state_dict(sd, strict=False)
    m = m.cuda().eval()
    lengths = torch.randint(1, T + 1, (B,), generator=torch.Generator().manual_seed(seed))
    mask = torch.arange(T)[None, :] < lengths[:, None]
    with torch.no_grad():
        _, out21, dec = m.hot_path(stage3.cuda(), frame.cuda(), audio.cuda(), want_decisions=True, frame_mask=mask.cuda())
        _, plain = m.hot_path(stage3.cuda(), frame.cuda(), audio.cuda())
        _, every = m.hot_path(stage3.cuda(), frame.cuda(), audio.cuda(), frame_mask=torch.ones(B, T, dtype=torch.bool, device="cuda"))
    assert torch.equal(every, plain)
    p = O.cast_params(sd, torch.float64)
    cls = M.tformer(frame.double(), p, "video_model.video_model.t_former.", T, mask)
    _, vt = O.au_former(cls, p, "video_model.au_head.")
    _, at = O.au_former(audio.double(), p, "audio_model.au_head.")
    ref = O.fusion_head(torch.cat([at, vt], dim=2), p, "au_head.")
    assert (out21[:, :12].double().cpu() - ref).abs().max().item() < 2e-2
    sure = ref.abs() > 2e-2
    assert bool((((dec.cpu() > 0) == (ref > 0)) | ~sure).all())
    assert not torch.equal(out21, plain)            # the mask reaches the logits


def test_mask_errors_are_loud():
    tr = A.Transformer(256, 1, 8, 32, 512).cuda().eval()
    x = torch.zeros(2, 12, 256, device="cuda")
    with pytest.raises(NotImplementedError, match="mask"), torch.no_grad():
        tr(x, mask=torch.ones(2, 12, dtype=torch.bool, device="cuda"))
    with pytest.raises(NotImplementedError, match="mask"), torch.no_grad():
        tr(x, mask=torch.ones(2, 1, 11, dtype=torch.bool, device="cuda"))
    with pytest.raises(TypeError), torch.no_grad():
        tr(x, mask=torch.ones(2, 11, device="cuda"))
    with pytest.raises(RuntimeError, match="no CPU fallback"), torch.no_grad():
        tr(x, mask=torch.ones(2, 11, dtype=torch.bool))
    tf = A.TFormer(num_patches=4).cuda().eval()
    with pytest.raises(NotImplementedError, match="mask"), torch.no_grad():
        tf.cls_features(torch.zeros(8, 512, device="cuda"), torch.ones(2, 5, dtype=torch.bool, device="cuda"))
