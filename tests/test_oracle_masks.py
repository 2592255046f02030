"""CPU checks of the masked fp64 restatement (tests/masked_oracle.py: the ``mask`` of Transformer.forward, models/heads.py:225-232, in
its ViT form): the contract the masked CUDA kernels are tested against.  The AVFormer path never passes a mask, so no golden vector of the reference
pins it; these tests pin its consequences instead."""
import os
import sys

import torch

from oracle import avformer_oracle as O

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import masked_oracle as M  # noqa: E402

HEADS, DH, DIM, MLP, DEPTH = 2, 8, 16, 32, 2


def _stack_params(seed):
    return O.params_from_spec(O._encoder_spec("t.", DIM, DEPTH, HEADS * DH, MLP), seed, torch.float64)


def test_all_true_mask_is_exactly_the_unmasked_oracle():
    p = _stack_params(1)
    x = torch.randn(3, 7, DIM, dtype=torch.float64, generator=torch.Generator().manual_seed(1))
    keep = torch.ones(3, 6, dtype=torch.bool)
    assert torch.equal(M.transformer(x, p, "t.", DEPTH, HEADS, keep), O.transformer(x, p, "t.", DEPTH, HEADS))


def test_prefix_mask_equals_the_shorter_clip():
    """Keeping the first k frames gives the cls output of a TFormer run on those k frames with pos[:k+1]."""
    T, B, D = 6, 4, 512                                  # the oracle TFormer has the reference geometry (O.STACKS["tformer"])
    p = O.params_from_spec([("tf.cls_token", (1, 1, D), "normal"), ("tf.pos_embedding", (1, T + 1, D), "normal")]
                           + list(O._encoder_spec("tf.spatial_transformer.", D, 3, 512, 1024)), 2, torch.float64)
    frames = torch.randn(B * T, D, dtype=torch.float64, generator=torch.Generator().manual_seed(2))
    for k in (1, 3, T):
        keep = torch.zeros(B, T, dtype=torch.bool)
        keep[:, :k] = True
        got = M.tformer(frames, p, "tf.", T, keep)
        ref = O.tformer(frames.view(B, T, D)[:, :k].reshape(B * k, D), p, "tf.", k)
        assert torch.allclose(got, ref, rtol=0, atol=1e-12 * ref.abs().max().item()), k


def test_dropped_row_attends_uniformly_to_all_tokens():
    """A dropped query's scores are all filled alike: its output is the mean of V over all N tokens, dropped ones included."""
    B, N = 3, 9
    inner = HEADS * DH
    p = {"a.fn.fn.to_qkv.weight": torch.randn(3 * inner, inner, dtype=torch.float64, generator=torch.Generator().manual_seed(3)),
         "a.fn.fn.to_out.0.weight": torch.eye(inner, dtype=torch.float64), "a.fn.fn.to_out.0.bias": torch.zeros(inner, dtype=torch.float64)}
    x = torch.randn(B, N, inner, dtype=torch.float64, generator=torch.Generator().manual_seed(4))
    keep = torch.rand(B, N - 1, generator=torch.Generator().manual_seed(5)) < 0.5
    keep[0, 2] = False
    y = M.attention(x, p, "a.", HEADS, keep)
    v = (x @ p["a.fn.fn.to_qkv.weight"].t())[..., 2 * inner:]
    full = torch.nn.functional.pad(keep, (1, 0), value=True)
    for b in range(B):
        for i in range(N):
            if not full[b, i]:
                assert torch.allclose(y[b, i], v[b].mean(0), rtol=1e-12, atol=1e-12)
    assert torch.isfinite(y).all()
    # a kept query gives probability 0 to the dropped keys: changing the dropped tokens' values leaves its output unchanged
    x2 = x.clone()
    x2[~full] += 5.0
    y2 = M.attention(x2, p, "a.", HEADS, keep)
    assert torch.allclose(y2[full], y[full], rtol=0, atol=1e-12)
