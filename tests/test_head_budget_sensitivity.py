"""The checks of tests/test_gpu_head_train.py catch the head bugs they are meant to catch (CPU only).

First, the hand-written backward of tests/head_oracle.py (front_emulate without rounding) is pinned to torch autograd over the restated
front (front_reference), and the loss and logit references to the oracle's closed forms.  Then every bug of head_oracle.MUTANTS,
computed in fp64 at every clip count the GPU tests run, must miss its check: a budgeted tensor's worst unit >= 1.5 x K_HEAD x the bf16
emulation's worst unit, a bounded quantity's error >= 1.5 x its fp32 bound, or an exact check failed.

Run with -s for the margins.  Three of the bugs cannot show at all at the 6 clips of the older whole-model tests
(test_bugs_invisible_at_six_clips): the loss loop that stops after 256 entries (72 entries at B = 6), dw_last summed over the first
8 clips only, and a dropped last split-K partial of dw_cat (one split up to 64 clips)."""
import functools
import math
import os
import sys

import pytest
import torch

from oracle import avformer_oracle as O

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import head_oracle as H  # noqa: E402

MARGIN = 1.5
SMS = 148                     # the B200's SM count: the split-K plan of the GPU run


def _rel(a, b):
    return ((a - b).abs().max() / b.abs().max().clamp_min(1e-300)).item()


@pytest.mark.parametrize("n", [2, 9, 65])
@pytest.mark.parametrize("batch_stats", [True, False])
def test_front_backward_is_autograd_of_the_restated_front(batch_stats, n):
    p = H.front_params(H.seed_of("pin", n))
    store, dx = H.front_inputs(n, H.seed_of("pin", n), p)
    emb = store[:, :H.IN_DIM].double()
    ref = H.front_reference(emb, p, batch_stats, dx)
    got = H.front_emulate(emb, p, batch_stats, dx)
    for k in ("tokens", "mean", "rstd", "run_mean", "run_var", "dgamma", "dbeta", "dw_cat", "db_cat", "dpos"):
        assert _rel(got[k], ref[k]) < 1e-10, k
    floor = (p["gamma"].double().abs() * got["rstd"] * got["dy"].abs().max(0).values).max()     # demb nearly cancels for a 2-row batch
    assert ((got["demb"] - ref["demb"]).abs().max() / floor).item() < 1e-10


def test_loss_and_logit_references_match_the_oracle():
    y_pred, labels = H.bce_inputs(9, "one", 3)
    x = y_pred[:, :12].double().requires_grad_(True)
    loss = O.au_loss(x, labels.double())
    loss.backward()
    l2, nv, g = H.bce(y_pred, labels)
    assert abs(l2 - loss.item()) < 1e-14 and nv == 8 and _rel(g, x.grad) < 1e-12
    xs = torch.randn(5 * 12, 128, dtype=torch.float64, requires_grad=True)
    w = torch.randn(12, 128, dtype=torch.float64, requires_grad=True)
    dl = torch.randn(5, 21, dtype=torch.float64)
    (xs.view(5, 12, 128) * w).sum(-1).backward(dl[:, :12])
    dx, dw = H.logits_bwd(dl, xs.detach(), w.detach(), 5)
    assert _rel(dx, xs.grad) < 1e-14 and _rel(dw, w.grad) < 1e-14


@functools.lru_cache(maxsize=None)
def _front_refs(n):
    p = H.front_params(H.seed_of("front-bf16-1", n))
    store, dx = H.front_inputs(n, H.seed_of("front-bf16-1", n), p)
    emb = store[:, :H.IN_DIM].double()
    return p, emb, dx, H.front_reference(emb, p, True, dx), H.front_emulate(emb, p, True, dx, path="per_op")


def margin(kind, n):
    """How far the mutant misses its check at n clips (>= 1: caught; inf: an exact check fails)."""
    if kind in ("running_var_biased", "bn_bwd_no_mean_dy", "bn_bwd_no_xhat_term", "dgamma_unnormalised_x", "splitk_drop_last_partial"):
        p, emb, dx, ref, emu = _front_refs(n)
        bad = H.front_emulate(emb, p, True, dx, bug=kind, sms=SMS)
        if kind == "running_var_biased":
            return float(((bad["run_var"] - ref["run_var"]).abs() / H.stat_bounds(emb, p, True)["run_var"]).max())
        if n > 2:
            return max(H.ratios(k, bad[k], emu[k], ref[k])[0] for k in H.BUDGET_TENSORS) / H.K_HEAD
        # demb of a 2-row batch is held to its fp32 cancellation bound, the rest to the budget
        two = ((bad["demb"] - ref["demb"]).abs() / H.two_row_demb_bound(emb, p, emu)).max().item()
        return max(two, max(H.ratios(k, bad[k], emu[k], ref[k])[0] for k in ("tokens", "dw_cat", "dgamma", "dbeta")) / H.K_HEAD)
    if kind in ("loss_nvalid_every_column", "bce_first_256_entries"):
        worst = 0.0
        for case in H.BCE_CASES:
            y_pred, labels = H.bce_inputs(n, case, H.seed_of(case, n))
            l0, nv0, g0 = H.bce(y_pred, labels)
            l1, nv1, g1 = H.bce(y_pred, labels, bug=kind)
            if nv1 != nv0:
                return math.inf
            lb, gb = H.bce_bounds(y_pred, labels)
            if nv0:
                worst = max(worst, abs(l1 - l0) / lb, float(((g1 - g0).abs() / gb.clamp_min(1e-300)).max()))
        return worst
    if kind == "dw_last_first_8_clips":
        g = torch.Generator().manual_seed(n)
        xs, w = torch.randn(n * 12, 256, generator=g), torch.randn(12, 256, generator=g) / 16
        dl = torch.randn(n, 21, generator=g) / (12.0 * n)
        _, dw0 = H.logits_bwd(dl, xs, w, n)
        _, dw1 = H.logits_bwd(dl, xs, w, n, bug=kind)
        bound = n * H.EPS32 * (dl[:, :12].double()[:, :, None].abs() * xs.double().view(n, 12, -1).abs()).sum(0)
        return float(((dw1 - dw0).abs() / bound).max())
    raise ValueError(kind)


@pytest.mark.parametrize("kind", H.MUTANTS)
def test_every_mutant_misses_its_check(kind):
    margins = {n: margin(kind, n) for n in H.CLIPS if H.mutant_applies(kind, n, sms=SMS)}
    print(f"\n{kind}: margin by clip count " + ", ".join(f"{n}: {m:.1f}" for n, m in margins.items()))
    assert margins, kind
    missed = {n: round(m, 2) for n, m in margins.items() if not m >= MARGIN}
    assert not missed, f"{kind} within {MARGIN} x its check at {missed}"


def test_bugs_invisible_at_six_clips():
    """The bugs no check can see at the 6 clips of the older whole-model tests: they only exist at larger batches."""
    invisible = {k for k in H.MUTANTS if not H.mutant_applies(k, 6, sms=SMS)}
    assert invisible == {"bce_first_256_entries", "dw_last_first_8_clips", "splitk_drop_last_partial"}
    for k in set(H.MUTANTS) - invisible:
        assert margin(k, 6) >= MARGIN, k
