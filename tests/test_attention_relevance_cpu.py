"""CPU checks of the attention-relevance references (tests/relevance_oracle.py): the oracle's G and rollout pinned to independent
torch autograd, and every injected definition bug missing the GPU tests' checks by at least 1.5x at the sizes those tests use."""
import os
import sys

import numpy as np
import pytest
import torch

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import relevance_oracle as RO  # noqa: E402

# the attention sizes and rollout sizes of tests/test_gpu_attention_relevance.py
ATT = [(32, n) for n in (1, 12, 17, 33, 49, 64)] + [(64, n) for n in (17, 64, 65, 129, 256)]
ROLL = [(n, d) for n in (12, 17, 49, 129, 256) for d in (1, 2, 3)]
G_TOL = 1e-4                  # test_attention_gradmaps / test_stack_gradmaps (fp32): max |G - G64| <= 1e-4 max |G64|


def _keep(n_seq, n_tok, seed):
    g = torch.Generator().manual_seed(seed)
    k = torch.rand(n_seq, n_tok, generator=g) < 0.6
    k[:, 0] = True
    k[1, 1:] = False
    k[2] = False
    return k


def _att(dh, n_tok, seed, n_seq=5, heads=8):
    g = torch.Generator().manual_seed(seed)
    qkv = torch.randn(n_seq * n_tok, 3 * heads * dh, generator=g, dtype=torch.float64)
    dout = torch.randn(n_seq * n_tok, heads * dh, generator=g, dtype=torch.float64)
    return qkv, dout, n_seq, heads


@pytest.mark.parametrize("masked", [False, True])
def test_gmap_against_autograd_of_torch_softmax(masked):
    """G = P * dL/dP with L = <softmax(S) V, dO>: torch.softmax and torch.autograd.grad, and the closed form dP = dO V^T."""
    dh, n_tok = 32, 17
    qkv, dout, n_seq, heads = _att(dh, n_tok, 1)
    keep = _keep(n_seq, n_tok, 2) if masked else None
    got = RO.gmap(qkv, dout, n_seq, n_tok, heads, dh, keep)
    q, k, v = (t.reshape(n_seq, n_tok, heads, dh).permute(0, 2, 1, 3) for t in qkv.split(heads * dh, dim=-1))
    do = dout.reshape(n_seq, n_tok, heads, dh).permute(0, 2, 1, 3)
    s = q @ k.transpose(-1, -2) * dh ** -0.5
    if masked:
        s = s.masked_fill(~keep[:, None, None, :], -float("inf")).masked_fill(~keep[:, None, :, None], 0.0)
    p = torch.softmax(s, dim=-1).requires_grad_(True)
    (dp,) = torch.autograd.grad((torch.matmul(p, v) * do).sum(), p)
    assert torch.allclose(got, p.detach() * dp, rtol=1e-12, atol=1e-14)
    assert torch.allclose(dp, do @ v.transpose(-1, -2), rtol=1e-12, atol=1e-14)
    if masked:                                            # dropped query: uniform P, so G = dP / n_tok; kept query x dropped key: 0
        rows = got.permute(0, 2, 1, 3)[~keep]
        assert torch.allclose(rows, (do @ v.transpose(-1, -2)).permute(0, 2, 1, 3)[~keep] / n_tok, rtol=1e-12, atol=1e-14)
        assert not got[keep[:, None, :, None].expand_as(got) & ~keep[:, None, None, :].expand_as(got)].any()


def test_rollout_against_explicit_products():
    g = torch.Generator().manual_seed(3)
    gm = torch.randn(3, 2, 4, 6, 6, generator=g, dtype=torch.float64)
    r = RO.rollout(gm).numpy()
    for b in range(2):
        ref = np.eye(6)
        for l in range(3):
            a = np.maximum(gm[l, b].numpy(), 0).mean(axis=0)
            ref = (np.eye(6) + a) @ ref
        assert np.allclose(r[b], ref, rtol=1e-13, atol=1e-15)


def test_stack_gmaps_follow_the_layers():
    """stack_gmaps (G from the hand-written backward's own qkv and dob, layer 0 first) equals P * dL/dP that autograd gives every
    softmax of the oracle's transformer, layer by layer."""
    import bf16_bwd_oracle as BB
    from oracle import avformer_oracle as O
    p = {k: v.double() for k, v in O.params_from_spec(list(O._encoder_spec("", 128, 2, 256, 256)), 1).items()}
    g = torch.Generator().manual_seed(4)
    x = torch.randn(3, 12, 128, generator=g, dtype=torch.float64)
    dy = BB.make_dy(36, 128, g).reshape(3, 12, 128).double()
    _, gm = RO.stack_gmaps(x, p, dy, 2, 8)
    assert gm.shape == (2, 3, 8, 12, 12)
    _, seen = RO.oracle_gmaps(O.transformer, lambda y: (y * dy).sum(), x, p, "", 2, 8)
    assert torch.allclose(gm, torch.stack(seen), rtol=1e-10, atol=1e-14)


@pytest.mark.parametrize("bug", RO.G_BUGS)
@pytest.mark.parametrize("masked", [False, True])
def test_gmap_bugs_miss_the_check(bug, masked):
    worst = float("inf")
    for dh, n_tok in ATT:
        if bug == "g_from_unnormalised_e" and n_tok == 1:
            continue                                      # one token: e = 1 = P, the bug is no bug
        qkv, dout, n_seq, heads = _att(dh, n_tok, dh * 1000 + n_tok)
        keep = _keep(n_seq, n_tok, n_tok + dh) if masked else None
        ref = RO.gmap(qkv, dout, n_seq, n_tok, heads, dh, keep)
        bad = RO.gmap(qkv, dout, n_seq, n_tok, heads, dh, keep, bug=bug)
        worst = min(worst, ((bad - ref).abs().max() / ref.abs().max()).item() / G_TOL)
    assert worst >= 1.5, f"{bug}: misses the G check by only {worst:.2f}x at some size"


@pytest.mark.parametrize("bug", RO.R_BUGS)
def test_rollout_bugs_miss_the_check(bug):
    worst = float("inf")
    for n, depth in ROLL:
        if bug == "r_times_a" and depth == 1:
            continue                                      # one layer: A R_0 = R_0 A = A
        g = torch.Generator().manual_seed(n * 10 + depth)
        gm = (torch.randn(depth, 3, 8, n, n, generator=g) * 4.0 / n).double()   # the inputs of test_rollout
        ref = RO.rollout(gm)
        bad = RO.rollout(gm, bug=bug)
        worst = min(worst, ((bad - ref).abs() / RO.rollout_bound(gm, ref)).max().item())
    assert worst >= 1.5, f"{bug}: misses the rollout check by only {worst:.2f}x at some size"


def test_cls_row_only_misses_the_check():
    """A last layer run on the cls rows alone (as the inference TFormer does) leaves rows 1.. of its G at 0: the stack check of that
    layer (1e-4 of its max-abs) and the rollout both see it, at T = 16 and 128."""
    for n in (17, 129):
        qkv, dout, n_seq, heads = _att(64, n, n)
        g = torch.stack([RO.gmap(qkv, dout, n_seq, n, heads, 64)] * 3)
        bad = RO.cls_row_only(g)
        assert ((bad[-1] - g[-1]).abs().max() / g[-1].abs().max()).item() >= 1.5 * G_TOL
        ref = RO.rollout(g)
        assert ((RO.rollout(bad) - ref).abs() / RO.rollout_bound(g, ref)).max().item() >= 1.5
