"""Whole-video inference: TFormer clips gathered on the device from a per-video frame bank (TFormer.cls_features_indexed,
avf_tformer_fwd_indexed) and the InferenceEngine's frame_features / clips pair built on it.

The indexed call must equal the explicit gather + frames-kept mask bit for bit: after the embed the kernels are the same, the embed
adds the same two fp32 values, and a missing slot never reaches the cls row (the masked kernels give its key probability exactly 0),
so its value (bank row 0 in the explicit gather, 0 in the indexed embed) cannot matter."""
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
DIM = 512


@pytest.fixture(autouse=True)
def _no_tf32():
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False


def _tformer(T, precision, seed):
    p = O.params_from_spec([("cls_token", (1, 1, DIM), "normal"), ("pos_embedding", (1, T + 1, DIM), "normal")]
                           + list(O._encoder_spec("spatial_transformer.", DIM, 3, 512, 1024)), seed)
    tf = A.TFormer(num_patches=T).cuda().eval()
    tf.load_state_dict(p, strict=True)
    tf.spatial_transformer.precision = precision
    return tf, {"tf." + k: v.double() for k, v in p.items()}


def _offsets(T):
    """The example offsets of the README: T frames three apart that end at the processed frame."""
    return 3 * (torch.arange(T) - (T - 1))


def _tables(T, seed):
    """name -> (n_bank, index [n_clips, T] int64, -1 = missing frame)."""
    g = torch.Generator().manual_seed(seed)
    out = {}
    rnd = torch.randint(0, 50, (37, T), generator=g)              # repeats, out of order
    rnd[3] = -1
    rnd[3, T // 2] = 5                                            # a clip with one real frame, in the middle
    out["random"] = (50, rnd)
    n = 40
    clamp = torch.arange(n)[:, None] + _offsets(T)
    out["clamp_edges"] = (n, clamp.clamp(0, n - 1))
    out["minus1_edges"] = (n, torch.where((clamp >= 0) & (clamp < n), clamp, torch.full_like(clamp, -1)))   # clip 0: one real frame
    many = torch.randint(0, 7, (64, T), generator=g)
    many[torch.rand(64, T, generator=g) < 0.3] = -1
    many[0] = -1                                                  # no real frame at all: the cls token alone
    out["clips_gt_bank"] = (7, many)
    out["clips_lt_bank"] = (300, torch.randint(0, 300, (5, T), generator=g))
    return out


def _explicit(tf, bank, idx):
    """The reference: gathered frames (bank row 0 in the missing slots) + the frames-kept mask."""
    idx = idx.to(bank.device)
    return tf.cls_features(bank[idx.clamp(min=0)].reshape(-1, DIM), mask=idx >= 0)


# ---------------------------------------------------------------------------------------------
# 1. indexed TFormer == explicit gather + mask, bit for bit, at the same launch count
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("T", [8, 16, 32])
@pytest.mark.parametrize("bank_dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_indexed_equals_explicit_gather_and_mask(precision, bank_dtype, T):
    tf, _ = _tformer(T, precision, 100 + T)
    L = A._lib.lib()
    for k, (name, (n_bank, idx)) in enumerate(_tables(T, T).items()):
        bank = torch.randn(n_bank, DIM, generator=torch.Generator().manual_seed(k)).cuda().to(bank_dtype)
        host_or_device = idx if k % 2 else idx.cuda().to(torch.int32)       # the index may live on the host or the device
        with torch.no_grad():
            ref = _explicit(tf, bank, idx)
            n0 = L.avf_launch_count()
            got = tf.cls_features_indexed(bank, host_or_device)
            n1 = L.avf_launch_count()
            _explicit(tf, bank, idx)
            n2 = L.avf_launch_count()
        assert got.shape == (idx.shape[0], DIM) and got.dtype == torch.float32 and not got.requires_grad
        assert torch.isfinite(got).all(), name
        assert torch.equal(got, ref), f"{name}: max |diff| {(got - ref).abs().max().item():.3e}"
        assert n1 - n0 == n2 - n1, f"{name}: {n1 - n0} launches indexed, {n2 - n1} gathered + masked"


def test_indexed_runs_the_inference_kernels_under_grad_mode():
    tf, _ = _tformer(16, "bf16", 7)
    n_bank, idx = _tables(16, 3)["minus1_edges"]
    bank = torch.randn(n_bank, DIM, device="cuda", requires_grad=True)
    got = tf.cls_features_indexed(bank, idx)
    assert not got.requires_grad and got.grad_fn is None
    with torch.no_grad():
        assert torch.equal(got, _explicit(tf, bank.detach(), idx))


# ---------------------------------------------------------------------------------------------
# 2. against the fp64 oracle
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_indexed_against_oracle_512_clips(precision):
    T, n_clips, n_bank = 16, 512, 600
    tf, p = _tformer(T, precision, 21)
    bank = torch.randn(n_bank, DIM, generator=torch.Generator().manual_seed(22))
    centre = torch.arange(n_clips) * n_bank // n_clips
    raw = centre[:, None] + 3 * (torch.arange(T) - T // 2)
    idx = torch.where((raw >= 0) & (raw < n_bank), raw, torch.full_like(raw, -1))      # -1 edges at both ends of the video
    assert (idx[0] == -1).any() and (idx[-1] == -1).any()
    with torch.no_grad():
        got = tf.cls_features_indexed(bank.cuda(), idx)
    sub = torch.arange(0, n_clips, 8)
    ref = M.tformer(bank[idx[sub].clamp(min=0)].reshape(-1, DIM).double(), p, "tf.", T, idx[sub] >= 0)
    ref = ref.double()
    err = (got[sub].double().cpu() - ref).abs().max().item() / ref.abs().max().item()
    assert err < (1e-4 if precision == "fp32" else 2e-2), err


# ---------------------------------------------------------------------------------------------
# 3. the kernel's bounds guard, without any read outside an allocation; the Python errors
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("bank_dtype", [torch.float32, torch.bfloat16])
def test_out_of_range_entries_are_missing_frames_and_never_read(bank_dtype):
    """The bank is a view big[8 : 8 + n_bank] of a tensor whose other rows are NaN: an entry n_bank reads the NaN row right after the
    bank and -7 the one 7 rows before it, if the guard is missing.  Nothing outside ``big`` is ever touched."""
    T, n_bank = 16, 24
    tf, _ = _tformer(T, "bf16", 9)
    big = torch.full((n_bank + 16, DIM), float("nan"), device="cuda", dtype=bank_dtype)
    big[8: 8 + n_bank] = torch.randn(n_bank, DIM, device="cuda").to(bank_dtype)
    bank = big[8: 8 + n_bank]
    idx = torch.randint(0, n_bank, (6, T), generator=torch.Generator().manual_seed(4)).to(torch.int32)
    bad, good = idx.clone(), idx.clone()
    bad[:, 0], bad[:, 5], bad[2, 9] = n_bank, -7, n_bank
    good[:, 0], good[:, 5], good[2, 9] = -1, -1, -1
    st = tf.spatial_transformer
    shape = st.shape(idx.shape[0], T + 1)

    def call(index):          # the C entry point itself, through its thin wrapper: no range check on the Python side
        return AF.tformer_fwd_indexed(bank, index.cuda().contiguous(), tf.cls_token.view(-1), tf.pos_embedding[0], st.packed(), shape)

    with torch.no_grad():
        got_bad, got_good = call(bad), call(good)
    assert torch.isfinite(got_good).all() and torch.isfinite(got_bad).all()
    assert torch.equal(got_bad, got_good)


def test_indexed_errors_are_loud():
    T = 8
    tf, _ = _tformer(T, "bf16", 3)
    bank = torch.randn(10, DIM, device="cuda")
    idx = torch.zeros(4, T, dtype=torch.int64)
    with torch.no_grad():
        with pytest.raises(ValueError, match="num_patches"):
            tf.cls_features_indexed(bank, torch.zeros(4, T + 1, dtype=torch.int64))
        with pytest.raises(ValueError, match="num_patches"):
            tf.cls_features_indexed(bank, torch.zeros(4 * T, dtype=torch.int64))
        with pytest.raises(ValueError, match="num_patches"):
            tf.cls_features_indexed(bank, torch.zeros(0, T, dtype=torch.int64))
        with pytest.raises(ValueError, match="bank"):
            tf.cls_features_indexed(torch.randn(10, 256, device="cuda"), idx)
        with pytest.raises(TypeError):
            tf.cls_features_indexed(bank, idx.float())
        with pytest.raises(TypeError):
            tf.cls_features_indexed(bank, idx.bool())
        with pytest.raises(TypeError):
            tf.cls_features_indexed(bank, idx.tolist())
        with pytest.raises(TypeError):
            tf.cls_features_indexed(bank.half(), idx)
        for v in (-2, 10, 1 << 40):
            bad = idx.clone()
            bad[2, 3] = v
            with pytest.raises(ValueError, match=r"\[-1, 10\)"):
                tf.cls_features_indexed(bank, bad)
            with pytest.raises(ValueError, match=r"\[-1, 10\)"):
                tf.cls_features_indexed(bank, bad.cuda())
        with pytest.raises(RuntimeError, match="no CPU fallback"):
            tf.cls_features_indexed(bank.cpu(), idx)
    dropout = A.TFormer(num_patches=T, dropout=0.1).cuda().train()
    with pytest.raises(RuntimeError, match="inference only"):
        dropout.cls_features_indexed(bank, idx)
    dropout.eval()
    with torch.no_grad():
        assert dropout.cls_features_indexed(bank, idx).shape == (4, DIM)


def test_indexed_call_can_be_captured_in_a_cuda_graph():
    """The range check reads the index on the host; while a graph is captured it is skipped (the kernel's guard still holds), and the
    replay gives the eager result."""
    T = 16
    tf, _ = _tformer(T, "bf16", 12)
    n_bank, idx = _tables(T, 5)["minus1_edges"]
    bank = torch.randn(n_bank, DIM, device="cuda")
    idx = idx.cuda()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.no_grad():
        with torch.cuda.stream(side):
            eager = tf.cls_features_indexed(bank, idx)
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=side):
            out = tf.cls_features_indexed(bank, idx)
    g.replay()
    torch.cuda.synchronize()
    assert torch.equal(out, eager)
    # a host index cannot be copied inside a capture: a clear error, raised before any work is captured
    host = idx.cpu()
    g2 = torch.cuda.CUDAGraph()
    with pytest.raises(RuntimeError, match="must already be on the"), torch.no_grad():
        with torch.cuda.graph(g2, stream=side):
            tf.cls_features_indexed(bank, host)


# ---------------------------------------------------------------------------------------------
# 4. InferenceEngine.frame_features / clips
# ---------------------------------------------------------------------------------------------
def _model(seed, T):
    m = A.TwoStreamAuralVisualFormer(video_pretrained=False, audio_pretrained=False, task="AU").set_clip_length(T)
    m.load_state_dict(O.make_state_dict(seed, T), strict=True)
    return m.cuda().eval().set_precision("bf16")


def _maxerr(a, b):
    return (a.double().cpu() - b.double().cpu()).abs().max().item()


def _module_path_masked(m, frames, idx, audio):
    """model(x)'s modules on a -1 table: module-path frame features -> masked cls_features -> AU_formers -> fusion head."""
    vm = m.video_model.video_model
    n = idx.shape[0]
    with torch.no_grad():
        feat = vm.s_former(frames[None])                                        # [F, 512]
        cls = vm.t_former.cls_features(feat[idx.clamp(min=0)].reshape(-1, DIM), mask=idx >= 0)
        fused = torch.empty((n * 12, 256), dtype=torch.float32, device="cuda")
        a_feat = m.audio_model.audio_model(audio).float().contiguous()
        m.audio_model.au_head.tokens_into(a_feat, a_feat.shape[1], n, out=fused, ld_out=256)
        m.video_model.au_head.tokens_into(cls, cls.shape[1], n, out=fused[:, 128:], ld_out=256)
        return m.au_head.logits21_(fused, n)


def _by_hand(eng, frames, idx, audio):
    """The engine's pieces composed by hand: folded trunks, the SFormer, cls_features_indexed, the heads."""
    m = eng.model
    vm = m.video_model.video_model
    n = idx.shape[0]
    with torch.no_grad():
        s3 = eng.video.to_stage(eng.video.stem_fwd(frames), 1, 3).to(torch.bfloat16)
        s3 = vm.s_former.sformer(s3.contiguous())
        bank = eng.video.to_stage(s3.to(eng.dtype).contiguous(memory_format=torch.channels_last), 4, 4).float().mean(dim=(2, 3))
        cls = vm.t_former.cls_features_indexed(bank, idx)
        fused = torch.empty((n * 12, 256), dtype=torch.float32, device="cuda")
        a_feat = eng.audio.to_stage(eng.audio.stem_fwd(audio), 1, 4).float().mean(dim=(2, 3))
        m.audio_model.au_head.tokens_into(a_feat, a_feat.shape[1], n, out=fused, ld_out=256)
        m.video_model.au_head.tokens_into(cls, cls.shape[1], n, out=fused[:, 128:], ld_out=256)
        return m.au_head.logits21_(fused, n, want_decisions=True)


@pytest.mark.parametrize("backbone", [torch.float32, torch.bfloat16])
def test_engine_clips_from_frame_bank(backbone):
    T, F, seed = 8, 40, 311
    m = _model(seed, T)
    eng = A.InferenceEngine(m, backbone_dtype=backbone)
    frames = O.synth_inputs(seed, 1, F)[0][0].permute(1, 0, 2, 3).contiguous().cuda()       # [F, 3, 112, 112]
    processed = torch.linspace(0, F - 1, 24).round().long()
    raw = processed[:, None] + _offsets(T)
    tables = {"clamp": raw.clamp(0, F - 1), "minus1": torch.where(raw >= 0, raw, torch.full_like(raw, -1))}
    audio = O.synth_inputs(seed + 1, 24, T)[1].cuda()
    tol = 5e-3 if backbone == torch.float32 else 0.25
    bank = torch.cat([eng.frame_features(frames[i: i + 16]) for i in range(0, F, 16)])    # frame chunks, as for a long video
    assert bank.shape == (F, DIM) and bank.dtype == torch.float32
    for name, idx in tables.items():
        out21, dec = eng.clips(bank, idx, audio)
        assert out21.shape == (24, 21) and dec.shape == (24, 12) and dec.dtype == torch.int32
        assert float(out21[:, 12:].abs().max()) == 0.0
        assert torch.equal(dec, (out21[:, :12] > 0).to(torch.int32))
        if name == "clamp":
            clips = frames[idx.cuda()].permute(0, 2, 1, 3, 4)                            # [n, C, T, H, W]: today's input
            with torch.no_grad():
                ref = m({"clip": clips, "audio_features": audio})
        else:
            ref = _module_path_masked(m, frames, idx.cuda(), audio)
        err = _maxerr(out21, ref)
        print(f"engine[{backbone}] {name}: max |logit - module path| = {err:.3e}")
        assert err < tol, (name, err)
        if backbone == torch.bfloat16:
            sure = ref[:, :12].abs() > 0.25
            assert bool((((out21[:, :12] > 0) == (ref[:, :12] > 0)) | ~sure).all()), name
        # the same engine's pieces composed by hand, on the whole video in one frame chunk
        whole = eng.frame_features(frames)
        o2, d2 = eng.clips(whole, idx, audio)
        h21, hdec = _by_hand(eng, frames, idx, audio)
        assert torch.equal(o2, h21) and torch.equal(d2, hdec), name


def test_engine_video_errors_are_loud():
    m = _model(5, 8)
    eng = A.InferenceEngine(m)
    with pytest.raises(ValueError, match="frame_features"):
        eng.frame_features(torch.zeros(4, 1, 112, 112, device="cuda"))
    with pytest.raises(ValueError, match="frame_features"):
        eng.frame_features(torch.zeros(2, 4, 3, 112, 112, device="cuda"))
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        eng.frame_features(torch.zeros(4, 3, 112, 112))
    bank = torch.randn(12, DIM, device="cuda")
    with pytest.raises(ValueError, match="one window per clip"):
        eng.clips(bank, torch.zeros(3, 8, dtype=torch.int64), torch.zeros(2, 1, 64, 1001, device="cuda"))
    with pytest.raises(ValueError, match=r"\[-1, 12\)"):
        eng.clips(bank, torch.full((2, 8), 12), torch.zeros(2, 1, 64, 1001, device="cuda"))
