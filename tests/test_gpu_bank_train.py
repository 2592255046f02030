"""Training over a frame bank: TFormer.forward_indexed with autograd, the deterministic scatter-add backward into the bank
(avf_tformer_embed_indexed_bwd) and TwoStreamAuralVisualFormer.forward_indexed.

forward_indexed must equal the explicit gather + frames-kept mask through autograd bit for bit.  Only the values in the missing slots
differ between the two paths (bank row 0 against 0).  Those rows are dropped keys: no kept row reads them, and their token gradient is
exactly zero in every layer.  The bank's gradient must equal, bit for bit, a CPU fp32 loop over the slots in ascending order applied
to the gather path's per-slot frame gradients.

For a bf16 bank the gather path takes the bank's values widened to fp32 as its frames.  The embed widens bf16 exactly, so its tokens
are the same, and its per-slot frame gradients stay fp32 rather than being rounded to bf16 slot by slot before the sum."""
import os
import sys

import pytest
import torch

import avformer_b200 as A
from oracle import avformer_oracle as O

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import masked_oracle as M  # noqa: E402
from test_gpu_video_bank import _offsets, _tables  # noqa: E402

pytestmark = pytest.mark.gpu
AF = A.functional
DIM = 512


@pytest.fixture(autouse=True)
def _no_tf32():
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False


def _tformer(T, precision, seed, dropout=0.0):
    p = O.params_from_spec([("cls_token", (1, 1, DIM), "normal"), ("pos_embedding", (1, T + 1, DIM), "normal")]
                           + list(O._encoder_spec("spatial_transformer.", DIM, 3, 512, 1024)), seed)
    tf = A.TFormer(num_patches=T, dropout=dropout).cuda().train()
    tf.load_state_dict(p, strict=True)
    tf.spatial_transformer.precision = precision
    return tf, {"tf." + k: v.double() for k, v in p.items()}


def _all_tables(T, seed):
    out = dict(_tables(T, seed))
    out["one_row_4096"] = (10, torch.full((4096 // T, T), 3, dtype=torch.int64))          # 256 x 16 at T = 16: one serial chain
    return out


def _mixed_dtok(n_clips, T, seed):
    """Token gradients whose magnitudes span 12 decades, so that the order of a sum shows in its bits."""
    g = torch.Generator().manual_seed(seed)
    mag = 10.0 ** torch.randint(-6, 7, (n_clips * (T + 1), DIM), generator=g).float()
    return torch.randn(n_clips * (T + 1), DIM, generator=g) * mag


def _cpu_scatter(rows, idx, n_bank, reverse=False):
    """rows [n_clips*T, dim] fp32, one per slot -> acc [n_bank, dim]: acc = acc + row over the valid slots in ascending (or
    descending) slot order, from +0.0."""
    acc = torch.zeros(n_bank, rows.shape[1], dtype=torch.float32)
    flat = idx.reshape(-1).tolist()
    order = range(len(flat) - 1, -1, -1) if reverse else range(len(flat))
    for s in order:
        i = flat[s]
        if 0 <= i < n_bank:
            acc[i] = acc[i] + rows[s]
    return acc


def _slot_rows(dtok, n_clips, T):
    return dtok.view(n_clips, T + 1, DIM)[:, 1:].reshape(-1, DIM)


# ---------------------------------------------------------------------------------------------
# 1. the scatter kernel against a plain CPU loop
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("T", [8, 16, 32])
@pytest.mark.parametrize("out_dtype", [torch.float32, torch.bfloat16])
def test_scatter_equals_ascending_cpu_loop(T, out_dtype):
    order_matters = False
    for k, (name, (n_bank, idx)) in enumerate(_all_tables(T, T).items()):
        n_clips = idx.shape[0]
        dtok = _mixed_dtok(n_clips, T, 1000 + k)
        idx32 = idx.to(torch.int32).cuda()
        got = AF.tformer_embed_indexed_bwd(dtok.cuda(), idx32, n_bank, T, out_dtype)
        again = AF.tformer_embed_indexed_bwd(dtok.cuda(), idx32, n_bank, T, out_dtype)
        rows = _slot_rows(dtok, n_clips, T)
        ref32 = _cpu_scatter(rows, idx, n_bank)
        ref = ref32.to(out_dtype)
        assert got.shape == (n_bank, DIM) and got.dtype == out_dtype
        assert torch.equal(got.cpu(), ref), f"{name}: {(got.cpu().float() - ref.float()).abs().max().item():.3e}"
        assert torch.equal(got, again), name
        unused = torch.ones(n_bank, dtype=torch.bool)
        unused[idx[(idx >= 0) & (idx < n_bank)]] = False
        if unused.any():                                        # exactly +0.0, sign bit clear
            z = got[unused.cuda()].float()
            assert torch.equal(z, torch.zeros_like(z)) and not torch.signbit(z).any(), name
        order_matters |= not torch.equal(_cpu_scatter(rows, idx, n_bank, reverse=True), ref32)      # in fp32: bf16 rounding can hide it
    assert order_matters, "no table shows that the summation order changes the bits: the test could not see a reordered sum"


def test_scatter_ignores_entries_outside_the_bank_and_writes_only_the_bank():
    """Entries n_bank and -7 are missing frames like -1; dbank is a view inside a NaN-filled buffer whose other rows must stay NaN."""
    T, n_bank = 16, 24
    idx = torch.randint(0, n_bank, (6, T), generator=torch.Generator().manual_seed(4))
    bad, good = idx.clone(), idx.clone()
    bad[:, 0], bad[:, 5], bad[2, 9] = n_bank, -7, 1 << 30
    good[:, 0], good[:, 5], good[2, 9] = -1, -1, -1
    dtok = _mixed_dtok(6, T, 5).cuda()
    big = torch.full((n_bank + 16, DIM), float("nan"), device="cuda")
    view = big[8: 8 + n_bank]
    L = A._lib.lib()
    ws = AF.workspace(L.avf_tformer_embed_indexed_bwd_workspace_bytes(6, T, n_bank), view.device)
    idx_bad = bad.to(torch.int32).cuda()
    rc = L.avf_tformer_embed_indexed_bwd(A._lib.AVF_FP32, AF._ptr(dtok), AF._ptr(idx_bad), 6, T, DIM, n_bank, AF._ptr(view), AF._ptr(ws), ws.numel(),
                                         AF._stream())
    assert rc == 0
    ref = AF.tformer_embed_indexed_bwd(dtok, good.to(torch.int32).cuda(), n_bank, T)
    assert torch.equal(view, ref)
    assert torch.isnan(big[:8]).all() and torch.isnan(big[8 + n_bank:]).all()


# ---------------------------------------------------------------------------------------------
# 2. forward_indexed against the explicit gather through autograd, bit for bit
# ---------------------------------------------------------------------------------------------
def _gather_path(tf, bank, idx, w, seed):
    frames = bank.detach().float()[idx.clamp(min=0).cuda()].reshape(-1, DIM).requires_grad_(True)
    tf.zero_grad(set_to_none=True)
    torch.manual_seed(seed)
    cls = tf(frames, mask=(idx >= 0).cuda())
    (cls * w).sum().backward()
    return cls.detach(), {k: p.grad.clone() for k, p in tf.named_parameters()}, frames.grad


def _indexed_path(tf, bank, idx, w, seed):
    leaf = bank.detach().clone().requires_grad_(True)
    tf.zero_grad(set_to_none=True)
    torch.manual_seed(seed)
    cls = tf.forward_indexed(leaf, idx)
    (cls * w).sum().backward()
    return cls.detach(), {k: p.grad.clone() for k, p in tf.named_parameters()}, leaf.grad


@pytest.mark.parametrize("T", [8, 16, 32])
@pytest.mark.parametrize("dropout", [0.0, 0.2])
@pytest.mark.parametrize("bank_dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_forward_indexed_equals_explicit_gather_through_autograd(precision, bank_dtype, dropout, T):
    tf, _ = _tformer(T, precision, 200 + T, dropout)
    for k, (name, (n_bank, idx)) in enumerate(_tables(T, T).items()):
        bank = torch.randn(n_bank, DIM, generator=torch.Generator().manual_seed(k)).cuda().to(bank_dtype)
        w = torch.randn(idx.shape[0], DIM, generator=torch.Generator().manual_seed(50 + k)).cuda()
        cls_g, g_g, dframes = _gather_path(tf, bank, idx, w, 7 + k)
        cls_i, g_i, dbank = _indexed_path(tf, bank, idx.cuda() if k % 2 else idx, w, 7 + k)
        assert torch.isfinite(cls_i).all(), name
        assert torch.equal(cls_i, cls_g), f"{name}: cls max |diff| {(cls_i - cls_g).abs().max().item():.3e}"
        for pn in g_g:
            assert torch.equal(g_i[pn], g_g[pn]), f"{name}: {pn} max |diff| {(g_i[pn] - g_g[pn]).abs().max().item():.3e}"
        assert dbank.dtype == bank_dtype and dbank.shape == bank.shape
        ref = _cpu_scatter(dframes.cpu(), idx, n_bank).to(bank_dtype)
        assert torch.equal(dbank.cpu(), ref), f"{name}: d_bank max |diff| {(dbank.cpu().float() - ref.float()).abs().max().item():.3e}"
        cls_2, g_2, dbank_2 = _indexed_path(tf, bank, idx, w, 7 + k)        # a second backward replays the bits
        assert torch.equal(cls_2, cls_i) and torch.equal(dbank_2, dbank) and all(torch.equal(g_2[pn], g_i[pn]) for pn in g_i), name


# ---------------------------------------------------------------------------------------------
# 3. against the fp64 oracle
# ---------------------------------------------------------------------------------------------
def _rel(a, b):
    a, b = a.double().cpu(), b.double().cpu()
    return ((a - b).abs().max() / b.abs().max().clamp_min(1e-30)).item()


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_forward_indexed_gradients_against_fp64_oracle(precision):
    T = 16
    tf, p = _tformer(T, precision, 31)
    tol = 1e-4 if precision == "fp32" else 3e-2
    for name in ("minus1_edges", "clamp_edges", "clips_gt_bank"):
        n_bank, idx = _tables(T, 2)[name]
        bank = torch.randn(n_bank, DIM, generator=torch.Generator().manual_seed(3))
        w = torch.randn(idx.shape[0], DIM, generator=torch.Generator().manual_seed(4))
        _, g_i, dbank = _indexed_path(tf, bank.cuda(), idx, w.cuda(), 0)
        pr = {k: v.clone().requires_grad_(True) for k, v in p.items()}
        bank64 = bank.double().requires_grad_(True)
        ref = M.tformer(bank64[idx.clamp(min=0)].reshape(-1, DIM), pr, "tf.", T, idx >= 0)
        (ref * w.double()).sum().backward()
        assert _rel(dbank, bank64.grad) < tol, (name, _rel(dbank, bank64.grad))
        for k, g in g_i.items():
            assert _rel(g, pr["tf." + k].grad) < tol, (name, k, _rel(g, pr["tf." + k].grad))


# ---------------------------------------------------------------------------------------------
# 4. nothing to differentiate: the inference call; the backward's launch count
# ---------------------------------------------------------------------------------------------
def test_no_grad_and_frozen_take_the_inference_call():
    T = 16
    tf, _ = _tformer(T, "bf16", 12)
    tf.eval()
    n_bank, idx = _tables(T, 3)["minus1_edges"]
    bank = torch.randn(n_bank, DIM, device="cuda")
    L = A._lib.lib()

    def counted(fn):
        n0 = L.avf_launch_count()
        out = fn()
        return out, L.avf_launch_count() - n0

    with torch.no_grad():
        tf.cls_features_indexed(bank, idx)                   # the first call also packs the weights
        ref, n_ref = counted(lambda: tf.cls_features_indexed(bank, idx))
        got, n_got = counted(lambda: tf.forward_indexed(bank, idx))
    assert torch.equal(got, ref) and n_got == n_ref
    for prm in tf.parameters():
        prm.requires_grad_(False)
    got, n_got = counted(lambda: tf.forward_indexed(bank, idx))
    assert got.grad_fn is None and torch.equal(got, ref) and n_got == n_ref


@pytest.mark.parametrize("bank_grad", [True, False])
def test_backward_launch_count(bank_grad):
    """The indexed backward is the gather path's backward plus the three scatter launches when the bank needs a gradient, and exactly
    the gather path's backward when it does not (the gather path's frame gradient is a view of the token gradient: no launch)."""
    T = 16
    tf, _ = _tformer(T, "bf16", 13)
    n_bank, idx = _tables(T, 4)["clamp_edges"]
    bank = torch.randn(n_bank, DIM, device="cuda")
    w = torch.randn(idx.shape[0], DIM, device="cuda")
    L = A._lib.lib()
    frames = bank[idx.cuda()].reshape(-1, DIM).requires_grad_(bank_grad)
    loss = (tf(frames, mask=(idx >= 0).cuda()) * w).sum()
    n0 = L.avf_launch_count()
    loss.backward()
    n_gather = L.avf_launch_count() - n0
    leaf = bank.clone().requires_grad_(bank_grad)
    loss = (tf.forward_indexed(leaf, idx) * w).sum()
    n0 = L.avf_launch_count()
    loss.backward()
    n_indexed = L.avf_launch_count() - n0
    assert n_indexed == n_gather + (3 if bank_grad else 0), (n_indexed, n_gather)
    assert (leaf.grad is not None) == bank_grad


# ---------------------------------------------------------------------------------------------
# 5. FusedAdam: the gradients handed over straight into the optimiser's bucket
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_fused_adam_steps_equal_the_gather_path(precision):
    T = 16
    tf1, _ = _tformer(T, precision, 41, dropout=0.2)
    tf2, _ = _tformer(T, precision, 41, dropout=0.2)
    o1 = A.FusedAdam(tf1.parameters(), lr=1e-3, weight_decay=5e-5)
    o2 = A.FusedAdam(tf2.parameters(), lr=1e-3, weight_decay=5e-5)
    n_bank, idx = _tables(T, 6)["minus1_edges"]
    bank = torch.randn(n_bank, DIM, device="cuda")
    w = torch.randn(idx.shape[0], DIM, device="cuda")
    for step in range(3):                  # from the second step on, .grad is a view of the bucket: the direct hand-over
        o1.zero_grad()
        torch.manual_seed(step)
        (tf1(bank[idx.clamp(min=0).cuda()].reshape(-1, DIM), mask=(idx >= 0).cuda()) * w).sum().backward()
        o1.step()
        o2.zero_grad()
        torch.manual_seed(step)
        (tf2.forward_indexed(bank, idx) * w).sum().backward()
        o2.step()
        for (k, a), b in zip(tf1.named_parameters(), tf2.parameters()):
            assert torch.equal(a, b), (step, k)


# ---------------------------------------------------------------------------------------------
# 6. the whole model
# ---------------------------------------------------------------------------------------------
def _model(seed, T, precision):
    m = A.TwoStreamAuralVisualFormer(video_pretrained=False, audio_pretrained=False, task="AU").set_clip_length(T)
    m.load_state_dict(O.make_state_dict(seed, T), strict=True)
    return m.cuda().set_precision(precision)


def _grads(m):
    return {k: (None if p.grad is None else p.grad.clone()) for k, p in m.named_parameters()}


def _video_inputs(seed, F, n_clips, T):
    frames = O.synth_inputs(seed, 1, F)[0][0].permute(1, 0, 2, 3).contiguous().cuda()       # [F, 3, 112, 112]
    processed = torch.linspace(0, F - 1, n_clips).round().long()
    raw = processed[:, None] + _offsets(T)
    audio = O.synth_inputs(seed + 1, n_clips, T)[1].cuda()
    return frames, raw, audio


def test_model_forward_indexed_equals_model_on_gathered_clips():
    T, F, n, seed = 8, 30, 12, 71
    m = _model(seed, T, "fp32").eval()                       # BatchNorm on running statistics, gradients on
    frames, raw, audio = _video_inputs(seed, F, n, T)
    idx = raw.clamp(0, F - 1)
    w = torch.randn(n, 21, device="cuda")
    m.zero_grad(set_to_none=True)
    ref = m({"clip": frames[idx.cuda()].permute(0, 2, 1, 3, 4), "audio_features": audio})
    (ref * w).sum().backward()
    g_ref = _grads(m)
    m.zero_grad(set_to_none=True)
    got = m.forward_indexed(frames, idx, audio)
    (got * w).sum().backward()
    g_got = _grads(m)
    assert got.shape == (n, 21) and float(got[:, 12:].abs().max()) == 0.0
    assert _rel(got, ref) < 1e-4, _rel(got, ref)
    for k, g in g_ref.items():
        assert (g is None) == (g_got[k] is None), k
        if g is not None and float(g.abs().max()) > 0:
            # The conv trunks' weight gradients are cuDNN reductions over 96 gathered images in model(x) and over the 30 unique
            # frames here, with algorithms chosen per batch size: conv1.weight differed by 3.6e-4 of its max-abs on a B200 (fp32, TF32
            # off).  Everything this package computes -- the transformers, the heads, the bank's gradient -- holds 1e-4.
            tol = 2e-3 if O.is_backbone_key(k) else 1e-4
            assert _rel(g_got[k], g) < tol, (k, _rel(g_got[k], g), tol)


def test_model_forward_indexed_with_missing_frames_matches_hot_path_train(monkeypatch):
    T, F, n, seed = 8, 30, 12, 72
    m = _model(seed, T, "fp32").eval()
    frames, raw, audio = _video_inputs(seed, F, n, T)
    idx = torch.where(raw >= 0, raw, torch.full_like(raw, -1))
    assert (idx == -1).any()
    vm = m.video_model.video_model
    w = torch.randn(n, 21, device="cuda")
    m.zero_grad(set_to_none=True)
    got = m.forward_indexed(frames, idx, audio)
    (got * w).sum().backward()
    assert torch.isfinite(got).all() and all(torch.isfinite(p.grad).all() for p in m.parameters() if p.grad is not None)
    g_got = _grads(m)
    bank = vm.s_former(frames[None]).detach()                # the trunk's training path, as inside forward_indexed
    a_feat = m.audio_model.audio_model(audio).detach()
    m.zero_grad(set_to_none=True)
    stage3 = torch.zeros(1, 256, 7, 7, device="cuda")
    _, ref = m.hot_path_train(stage3, bank[idx.clamp(min=0).cuda()].reshape(-1, DIM), a_feat, frame_mask=(idx >= 0).cuda())
    (ref * w).sum().backward()
    g_ref = _grads(m)
    assert _rel(got, ref) < 1e-5, _rel(got, ref)
    heads = [k for k in g_ref if k.startswith(("au_head.", "video_model.au_head.", "audio_model.au_head.", "video_model.video_model.t_former."))]
    assert heads
    for k in heads:
        if g_ref[k] is not None and float(g_ref[k].abs().max()) > 0:
            assert _rel(g_got[k], g_ref[k]) < 1e-5, (k, _rel(g_got[k], g_ref[k]))
    # a frozen video branch: no bank gradient, so no scatter
    for p in m.video_model.parameters():
        p.requires_grad_(False)

    def no_scatter(*a, **k):
        raise AssertionError("the scatter ran for a frozen video branch")

    monkeypatch.setattr(AF, "tformer_embed_indexed_bwd", no_scatter)
    m.zero_grad(set_to_none=True)
    (m.forward_indexed(frames, idx, audio) * w).sum().backward()
    assert all(p.grad is None for p in m.video_model.parameters())
    assert m.au_head.pos_embedding.grad is not None


def test_model_forward_indexed_train_step_with_batch_statistics():
    T, F, n, seed = 8, 24, 10, 73
    m = _model(seed, T, "bf16").train()
    frames, raw, audio = _video_inputs(seed, F, n, T)
    idx = raw.clamp(0, F - 1)
    opt = A.FusedAdam(m.parameters(), lr=1e-4, weight_decay=5e-5)
    labels = O.synth_inputs(seed, n, T, image=8)[2].cuda()
    bn = m.video_model.video_model.s_former.bn1
    before = bn.num_batches_tracked.item()
    opt.zero_grad()
    loss = m.get_au_loss(m.forward_indexed(frames, idx, audio), labels)
    loss.backward()
    opt.step()
    assert torch.isfinite(loss) and bn.num_batches_tracked.item() == before + 1
    assert all(torch.isfinite(p).all() for p in m.parameters())
    assert m.video_model.video_model.s_former.conv1.weight.grad is not None


# ---------------------------------------------------------------------------------------------
# 7. errors
# ---------------------------------------------------------------------------------------------
def test_forward_indexed_errors_match_cls_features_indexed():
    T = 8
    tf, _ = _tformer(T, "bf16", 3)
    bank = torch.randn(10, DIM, device="cuda", requires_grad=True)
    idx = torch.zeros(4, T, dtype=torch.int64)
    cases = [(ValueError, bank, torch.zeros(4, T + 1, dtype=torch.int64)), (ValueError, bank, torch.zeros(0, T, dtype=torch.int64)),
             (ValueError, torch.randn(10, 256, device="cuda"), idx), (TypeError, bank, idx.float()), (TypeError, bank, idx.tolist()),
             (RuntimeError, bank.detach().cpu(), idx)]
    for v in (-2, 10):
        bad = idx.clone()
        bad[2, 3] = v
        cases += [(ValueError, bank, bad), (ValueError, bank, bad.cuda())]
    for cls_, b, i in cases:
        with pytest.raises(cls_) as e_ref:
            tf.eval()
            with torch.no_grad():
                tf.cls_features_indexed(b, i)
        tf.train()
        with pytest.raises(cls_) as e_got:
            tf.forward_indexed(b, i)
        assert str(e_got.value) == str(e_ref.value).replace("cls_features_indexed", "forward_indexed")
    with pytest.raises(TypeError):
        tf.forward_indexed(bank.detach().half(), idx)
    # a host index under capture
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    g = torch.cuda.CUDAGraph()
    with pytest.raises(RuntimeError, match="must already be on the"), torch.no_grad():
        with torch.cuda.graph(g, stream=side):
            tf.forward_indexed(bank.detach(), idx)


def test_model_forward_indexed_errors_launch_nothing():
    m = _model(5, 8, "bf16").eval()
    frames = torch.zeros(12, 3, 112, 112, device="cuda")
    audio = torch.zeros(2, 1, 64, 1001, device="cuda")
    L = A._lib.lib()
    n0 = L.avf_launch_count()
    with pytest.raises(ValueError, match="one audio window per clip"):
        m.forward_indexed(frames, torch.zeros(3, 8, dtype=torch.int64), audio)
    with pytest.raises(ValueError, match="frames must be"):
        m.forward_indexed(torch.zeros(2, 12, 3, 112, 112, device="cuda"), torch.zeros(2, 8, dtype=torch.int64), audio)
    with pytest.raises(ValueError, match=r"\[-1, 12\)"):
        m.forward_indexed(frames, torch.full((2, 8), 12), audio)
    assert L.avf_launch_count() == n0
    with torch.no_grad():
        out = m.forward_indexed(frames, torch.zeros(2, 8, dtype=torch.int64), audio)
    assert out.shape == (2, 21)
    m.task = "EX"
    with torch.no_grad():
        assert float(m.forward_indexed(frames, torch.zeros(2, 8, dtype=torch.int64), audio).abs().max()) == 0.0
