"""The bf16 budgets of tests/test_gpu_bf16_budget.py catch the bugs they are meant to catch (CPU only).

For every case the GPU tests run, on the same inputs, each bug of bf16_oracle.mutant (computed in fp64, no rounding at all) must
miss the case's budget by a margin: max_row row_rms(mutant - fp64) >= 1.5 * K * budget, where the budget is the larger of the
two emulations' worst rows (fused and kernel-per-operation), so the margin holds for whichever path the case runs.  A bug that
is no bug at a shape (bf16_oracle.mutant_applies) is skipped there.  Run with -s for the margins of every case.

Out of reach of any bf16 test, by nature, because they sit below bf16 rounding (fp64, module-like weights): GELU with erf instead of
tanh (row RMS about 3e-4) and LayerNorm eps 1e-6 instead of 1e-5 (about 1e-5).  The fp32-mode tests cover both, on the
kernel-per-operation path, at 1e-4."""
import os
import sys

import pytest
import torch

from oracle import avformer_oracle as O

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import bf16_oracle as B  # noqa: E402

MARGIN = 1.5


def test_restatement_is_the_oracle():
    """The stack bf16_oracle rounds and mutates is O.transformer, operation for operation."""
    case = next(c for c in B.ALL_CASES if c["name"] == "rows-d256-t49")
    ref, _, _, t, p = B.references(case)
    assert (ref - O.transformer(t, p, "", case["depth"], 8)).abs().max().item() < 1e-12


def test_emulation_rounds_where_the_paths_differ():
    """The two emulations are not the same computation (and neither is fp64): a fused-path bug in rounding would otherwise
    hide behind the per-op model."""
    case = next(c for c in B.ALL_CASES if c["name"] == "rows-d128-t12")
    ref, emu_fused, emu_per_op, _, _ = B.references(case)
    assert B.budget(emu_fused, ref) > 0 and B.budget(emu_per_op, ref) > 0
    assert not torch.equal(emu_fused, emu_per_op)


@pytest.mark.parametrize("case", B.ALL_CASES, ids=[c["name"] for c in B.ALL_CASES])
def test_every_mutant_exceeds_the_budget(case):
    ref, emu_fused, emu_per_op, t, p = B.references(case, case["sample"])
    budget = max(B.budget(emu_fused, ref), B.budget(emu_per_op, ref))
    margins = {}
    for kind in B.MUTANTS:
        if not B.mutant_applies(kind, case["n_tok"], case["depth"], case["mlp"]):
            continue
        bad = B.mutant(kind, t, p, "", case["depth"], 8)
        margins[kind] = B.row_rms(bad - ref).max().item() / (B.K * budget)
    print(f"\n{case['name']}: budget {budget:.2e}, mutant worst row / (K * budget): " + ", ".join(f"{k} {v:.1f}" for k, v in margins.items()))
    missed = {k: round(v, 2) for k, v in margins.items() if not v >= MARGIN}
    assert not missed, f"mutants within {MARGIN} x K x budget: {missed}"
