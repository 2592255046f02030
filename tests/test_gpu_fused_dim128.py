"""The fused encoder kernel at model width 128 (AU_formers, VA_former) and the positional add / AU logits folded into its input and
output sweeps: against the fp64 oracle, and against the kernel-per-operation path (set_fused_enabled(False)), which runs the
positional add and the AU logits as kernels of their own."""
import pytest
import torch

import avformer_b200 as A
from oracle import avformer_oracle as O

pytestmark = pytest.mark.gpu
AF = A.functional
N_CLIPS, T = 512, 16


def _maxerr(a, b):
    return (a.double().cpu() - b.double().cpu()).abs().max().item()


def _stack(dim, depth, mlp, seed):
    torch.manual_seed(seed)
    tr = A.Transformer(dim, depth, 8, 32, mlp).cuda().eval()
    tr.precision = "bf16"
    pr = {"t." + k: v.detach().double().cpu() for k, v in tr.named_parameters()}
    return tr, pr


@pytest.mark.parametrize("depth,mlp", [(1, 128), (2, 256), (3, 256)])
@pytest.mark.parametrize("n_tok", [1, 2, 12, 16, 17, 33, 64])
def test_dim128_fused_stack_against_oracle(n_tok, depth, mlp):
    tr, pr = _stack(128, depth, mlp, 100 * n_tok + depth)
    n_seq = 7
    assert AF.encoder_fused_supported(tr.shape(n_seq, n_tok))
    x = torch.randn(n_seq, n_tok, 128, device="cuda")
    pos = torch.randn(n_tok, 128, device="cuda") * 0.5
    ref = O.transformer((x + pos).double().cpu(), pr, "t.", depth, 8)
    packed, xs = tr.packed(), x.reshape(-1, 128).clone()      # (the first packing casts the weights to bf16: launches of its own)
    n0 = A._lib.lib().avf_launch_count()
    with torch.no_grad():
        y = AF.token_stack_fwd_(xs, packed, tr.shape(n_seq, n_tok), pos)
    assert A._lib.lib().avf_launch_count() - n0 == 1          # positional add and the whole stack: one launch
    assert _maxerr(y.view(n_seq, n_tok, 128), ref) < 6e-2
    with torch.no_grad():
        assert _maxerr(tr(x + pos), ref) < 6e-2


def test_dim128_ragged_tiles_beyond_one_wave():
    """1500 sequences of 12 tokens: 188 tiles of 8 sequences on at most 148 CTAs, the last tile half full."""
    tr, pr = _stack(128, 2, 256, 77)
    x = torch.randn(1500, 12, 128, device="cuda")
    with torch.no_grad():
        y = tr(x)
    ref = O.transformer(x.double().cpu(), pr, "t.", 2, 8)
    assert _maxerr(y, ref) < 6e-2
    assert _maxerr(y[-4:], ref[-4:]) < 6e-2


def _model(seed):
    m = A.TwoStreamAuralVisualFormer(video_pretrained=False, audio_pretrained=False, task="AU").set_clip_length(T)
    m.load_state_dict(O.make_state_dict(seed, T), strict=True)
    return m.cuda().eval().set_precision("bf16")


def _chain(m, cls, audio, fused):
    """Both AU_formers into the [B*12, 256] fusion input, then the fusion head, with the fused path on or off."""
    prev = AF.set_fused_enabled(fused)
    try:
        n = cls.shape[0]
        tokens = torch.empty((n * 12, 256), dtype=torch.float32, device="cuda")
        with torch.no_grad():
            m.audio_model.au_head.tokens_into(audio, audio.shape[1], n, out=tokens, ld_out=256)
            m.video_model.au_head.tokens_into(cls, cls.shape[1], n, out=tokens[:, 128:], ld_out=256)
            out21, dec = m.au_head.logits21_(tokens.clone(), n, True)
        return tokens, out21, dec
    finally:
        AF.set_fused_enabled(prev)


def test_au_formers_and_head_fused_against_unfused_512_clips():
    seed = 4545
    m = _model(seed)
    g = torch.Generator(device="cpu").manual_seed(seed)
    cls = (torch.randn(N_CLIPS, 512, generator=g).abs() * 1.2).cuda()
    audio = torch.randn(N_CLIPS, 512, generator=g).abs().cuda()
    tok_on, out_on, dec_on = _chain(m, cls, audio, True)
    tok_off, out_off, dec_off = _chain(m, cls, audio, False)
    assert _maxerr(tok_on[:, :128], tok_off[:, :128]) < 6e-2          # audio AU_former
    assert _maxerr(tok_on[:, 128:], tok_off[:, 128:]) < 6e-2          # video AU_former
    assert _maxerr(out_on, out_off) < 2e-2
    sure = out_off[:, :12].abs() > 2e-2
    assert bool(((dec_on == dec_off) | ~sure).all())
    # the fp64 oracle on a few clips
    p = O.cast_params(O.make_state_dict(seed, T, hot_path_only=True), torch.float64)
    idx = torch.tensor([0, 1, 255, 256, 510, 511])
    _, vt = O.au_former(cls[idx].double().cpu(), p, "video_model.au_head.")
    _, at = O.au_former(audio[idx].double().cpu(), p, "audio_model.au_head.")
    ref = O.fusion_head(torch.cat([at, vt], 2), p, "au_head.")
    assert _maxerr(out_on[idx.cuda(), :12], ref) < 2e-2


def test_head_folded_logits():
    """The fusion head's AU logits from the fused output sweep: padding columns exactly 0, decisions exactly logit > 0, no token
    rows stored when no output is given."""
    m = _model(99)
    head = m.au_head
    tr = head.corr_transformer
    n = 300
    x = torch.randn(n * 12, 256, device="cuda")
    x0 = x.clone()
    with torch.no_grad():
        out21, dec = AF.token_stack_fwd_(x, tr.packed(), tr.shape(n, 12), head.pos_embedding[0], w_last=head._packed_last().w,
                                         want_decisions=True)
    assert out21.shape == (n, 21) and dec.shape == (n, 12) and dec.dtype == torch.int32
    assert float(out21[:, 12:].abs().max()) == 0.0
    assert torch.equal(dec, (out21[:, :12] > 0).int())
    assert torch.equal(x, x0)                                   # the input rows were read, nothing was stored
    with torch.no_grad():
        y = AF.token_stack_fwd_(x0.clone(), tr.packed(), tr.shape(n, 12), head.pos_embedding[0])
    ref, _ = AF.au_logits(y, head._packed_last().w, n, True)
    assert _maxerr(out21, ref) < 1e-4
    pr = {k: v.detach().double().cpu() for k, v in head.named_parameters()}
    ref64 = O.fusion_head(x0.view(n, 12, 256).double().cpu(), pr, "")
    assert _maxerr(out21[:, :12], ref64) < 5e-2

