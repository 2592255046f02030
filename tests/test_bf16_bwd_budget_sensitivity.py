"""The bf16 backward budgets of tests/test_gpu_bf16_bwd_budget.py catch the bugs they are meant to catch (CPU only).

First, the hand-written backward of tests/bf16_bwd_oracle.py is pinned to torch autograd: stack_bwd over O.transformer (and, masked,
over tests/masked_oracle.py) in dx and all 11 gradients per layer, attention_bwd over a plain softmax attention, both to 1e-10
relative.  Then, for every case the GPU tests run and on the same inputs, each applicable bug of bf16_bwd_oracle.MUTANTS (computed
in fp64) must miss the case's budget by a margin: for some tensor, its worst unit >= 1.5 * K_BWD * the emulation's worst unit.  Run
with -s for every mutant's margin and whether the bounds the older tests use (3e-2 of each gradient's max-abs, 2^-7 of dqkv's
max-abs) would have caught it.  The list of bugs that sit below bf16 rounding by nature is in the oracle's docstring."""
import functools
import os
import sys

import pytest
import torch

from oracle import avformer_oracle as O

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import bf16_bwd_oracle as BB  # noqa: E402
import masked_oracle as MO  # noqa: E402

MARGIN = 1.5
OLD_STACK_RTOL = 3e-2
OLD_DQKV_RTOL = 2 ** -7


def _rel(a, b):
    return ((a - b).abs().max() / b.abs().max().clamp_min(1e-300)).item()


@pytest.mark.parametrize("masked", [False, True])
def test_stack_bwd_is_autograd_of_the_oracle(masked):
    case = next(c for c in BB.STACK_CASES if c["name"] == ("tformer-masked" if masked else "au-former"))
    p, x, dy, keep = BB.stack_inputs(case)
    if masked:        # masked_oracle's mask always keeps token 0 (the cls slot); the kernel-level pin below covers the rest
        keep[:, 0] = True
    n_seq, n_tok, dim, depth = case["n_seq"], case["n_tok"], case["dim"], case["depth"]
    p64 = {k: v.double().requires_grad_(True) for k, v in p.items()}
    x64 = x.double().view(n_seq, n_tok, dim).requires_grad_(True)
    dy64 = dy.double().view(n_seq, n_tok, dim)
    y = MO.transformer(x64, p64, "", depth, 8, keep[:, 1:]) if masked else O.transformer(x64, p64, "", depth, 8)
    y.backward(dy64)
    dx, grads = BB.stack_bwd(x64.detach(), {k: v.detach() for k, v in p64.items()}, dy64, depth, 8, keep)
    assert _rel(dx, x64.grad) < 1e-10
    for l in range(depth):
        for j, key in enumerate(BB.KEYS):
            ref = p64[f"layers.{l}.{key}"].grad
            assert _rel(grads[11 * l + j], ref) < 1e-10, f"layer {l} {BB.NAMES[j]}"


@pytest.mark.parametrize("masked", [False, True])
def test_attention_bwd_is_autograd(masked):
    case = next(c for c in BB.ATT_CASES if c["name"] == f"att-{'m' if masked else 'u'}-dh32-t33-h3")
    qkv, dout, keep = BB.att_inputs(case)
    n_seq, n_tok, heads, dh = case["n_seq"], case["n_tok"], case["heads"], case["dh"]
    q64 = qkv.double().requires_grad_(True)
    q, k, v = (t.reshape(n_seq, n_tok, heads, dh).permute(0, 2, 1, 3) for t in q64.chunk(3, dim=-1))
    s = q @ k.transpose(-1, -2) * dh ** -0.5
    if masked:                                   # masked_oracle.attention: fill (i, j) unless both tokens are kept
        s = s.masked_fill(~(keep[:, None, :, None] & keep[:, None, None, :]), -torch.finfo(s.dtype).max)
    o = torch.softmax(s, dim=-1) @ v
    o.permute(0, 2, 1, 3).reshape(n_seq * n_tok, heads * dh).backward(dout.double())
    got = BB.attention_bwd(qkv.double(), dout.double(), n_seq, n_tok, heads, dh, keep)
    assert _rel(got, q64.grad) < 1e-10


def test_mask_edges_are_in_every_masked_case():
    """Each masked case has a sequence with every token dropped and one with only its first token kept."""
    for case in [c for c in BB.ATT_CASES + BB.STACK_CASES if c["masked"]]:
        keep = BB.att_inputs(case)[2] if case["kind"] == "att" else BB.stack_inputs(case)[3]
        assert not bool(keep[0].any()) and bool(keep[1, 0]) and not bool(keep[1, 1:].any())


@functools.lru_cache(maxsize=None)
def _stack_refs(name):
    case = next(c for c in BB.STACK_CASES if c["name"] == name)
    return BB.stack_reference(case), BB.stack_reference(case, path="per_op")


def _old_caught(got, ref):
    return any(_rel(got[k], ref[k]) > OLD_STACK_RTOL for k in ref if float(ref[k].abs().max()) > 0)


@pytest.mark.parametrize("case", BB.ATT_CASES, ids=[c["name"] for c in BB.ATT_CASES])
def test_every_attention_mutant_exceeds_the_budget(case):
    ref, emu = BB.att_references(case)
    margins, old = {}, {}
    for kind in BB.ATTENTION_MUTANTS:
        if not BB.mutant_applies(kind, case):
            continue
        bad, _ = BB.att_references(case, bug=kind)
        worst, _ = BB.ratios("dqkv", bad, emu, ref, case["heads"])
        margins[kind] = worst / BB.K_BWD
        old[kind] = _rel(bad, ref) > OLD_DQKV_RTOL
    print(f"\n{case['name']}: mutant worst unit / (K_BWD * budget) [old 2^-7 bound catches]: "
          + ", ".join(f"{k} {v:.1f} [{'y' if old[k] else 'n'}]" for k, v in margins.items()))
    missed = {k: round(v, 2) for k, v in margins.items() if not v >= MARGIN}
    assert not missed, f"mutants within {MARGIN} x K_BWD x budget: {missed}"


@pytest.mark.parametrize("case", BB.STACK_CASES, ids=[c["name"] for c in BB.STACK_CASES])
def test_every_stack_mutant_exceeds_the_budget(case):
    ref, emu = _stack_refs(case["name"])
    margins, old = {}, {}
    for kind in BB.MUTANTS:
        if not BB.mutant_applies(kind, case):
            continue
        bad = BB.stack_reference(case, bug=kind)
        r = BB.stack_ratios(bad, emu, ref)
        margins[kind] = max(w for w, _ in r.values()) / BB.K_BWD
        old[kind] = _old_caught(bad, ref)
    print(f"\n{case['name']}: mutant worst unit / (K_BWD * budget) [old 3e-2 bound catches]: "
          + ", ".join(f"{k} {v:.1f} [{'y' if old[k] else 'n'}]" for k, v in margins.items()))
    missed = {k: round(v, 2) for k, v in margins.items() if not v >= MARGIN}
    assert not missed, f"mutants within {MARGIN} x K_BWD x budget: {missed}"
