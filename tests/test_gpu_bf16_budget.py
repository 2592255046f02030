"""bf16 encoder stacks against per-case error budgets (tests/bf16_oracle.py): the fused kernel on fp32 token rows at dim 256 and 128
and on NCHW maps of every size up to 64 positions, the kernel-per-operation bf16 path on the same inputs plus the TFormer geometry,
and the row strides of the C ABI.

Every case draws random LayerNorm vectors, biases and positional tables, so a swapped or stale per-layer vector shows.  A case
passes when its worst token row is within K times the bf16 emulation's worst token row (per-row RMS error against fp64), and the
median row within [0.5, 2] times the emulation's median row: the emulation has to model the kernel, not just bound it.  Cases
with more tiles than SMs compare the sequences of the first tile, the tiles at the wave boundary and the last tile."""
import ctypes
import functools
import os
import sys

import pytest
import torch

import avformer_b200 as A

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import bf16_oracle as B  # noqa: E402

pytestmark = pytest.mark.gpu
AF = A.functional
MEDIAN_RATIO = (0.5, 2.0)


@functools.lru_cache(maxsize=None)
def _references(name):
    case = next(c for c in B.ALL_CASES if c["name"] == name)
    ref, emu_fused, emu_per_op, _, _ = B.references(case, case["sample"])
    return ref, {"fused": emu_fused, "per_op": emu_per_op}


def _module(case, p, pos):
    """A.Transformer (rows) / A.ResFormer or A.SFormerBlock (nchw) holding the case's parameters, in bf16."""
    if case["kind"] == "rows":
        m = A.Transformer(case["dim"], case["depth"], 8, case["dh"], case["mlp"])
        m.load_state_dict(p, strict=True)
        m.precision = "bf16"
        return m.cuda().eval()
    if case["name"] == "nchw-resformer-7x7":
        m = A.ResFormer(A.BasicBlock, [2, 2, 2, 2])
    else:
        m = A.SFormerBlock(num_patches=case["num_patches"], dim=256, depth=case["depth"], heads=8, mlp_dim=case["mlp"], dim_head=32)
    m.spatial_transformer.load_state_dict(p, strict=True)
    with torch.no_grad():
        m.pos_embedding[0, :case["n_tok"]] = pos
    m.spatial_transformer.precision = "bf16"
    return m.cuda().eval()


def _launches():
    return A._lib.lib().avf_launch_count()


def run_case(case, path):
    """Run one case on the GPU through ``path`` ("fused" or "per_op"); returns (worst-row ratio, median-row ratio) of the kernel's
    per-row RMS error to the emulation's, and checks that the launch sequence is the one the path names."""
    p, x, pos = B.make_inputs(case)
    m = _module(case, p, pos)
    n_seq, n_tok, dim, depth = case["n_seq"], case["n_tok"], case["dim"], case["depth"]
    prev = AF.set_fused_enabled(path == "fused")
    try:
        with torch.no_grad():
            if case["kind"] == "rows":
                packed, shape = m.packed(), m.shape(n_seq, n_tok)
                assert AF.encoder_fused_supported(shape) == (dim in (128, 256))
                xs, posc = x.cuda(), pos.cuda()
                n0 = _launches()
                y = AF.token_stack_fwd_(xs, packed, shape, posc)
                n = _launches() - n0
                y = y.view(n_seq, n_tok, dim)
            else:
                fwd = m.sformer if isinstance(m, A.ResFormer) else m
                xc = x.cuda()
                fwd(xc)                                          # packs the weights (launches of their own)
                n0 = _launches()
                y = fwd(xc)
                n = _launches() - n0
                again = fwd(xc)
                assert torch.equal(y, again), "a second identical launch differs"     # the tile counter is re-armed per launch
                y = y.reshape(n_seq, dim, n_tok).transpose(1, 2)
            torch.cuda.synchronize()
    finally:
        AF.set_fused_enabled(prev)
    if path == "fused":
        # rows: positional add + stack in one launch; NCHW: pos_transpose_kernel + encoder_fused_kernel
        assert n == (1 if case["kind"] == "rows" else 2), f"{n} launches"
    else:
        assert n >= 7 * depth, f"{n} launches: not the kernel-per-operation path"
    if case["sample"] is not None:
        y = y[torch.tensor(case["sample"], device=y.device)]
    ref, emu = _references(case["name"])
    got = B.row_rms(y.double().cpu() - ref)
    exp = B.row_rms(emu[path] - ref)
    return (got.max() / exp.max()).item(), (got.median() / exp.median()).item()


def _check(case, path):
    worst, median = run_case(case, path)
    assert MEDIAN_RATIO[0] <= median <= MEDIAN_RATIO[1], f"median-row ratio {median:.3f}: the emulation does not model the kernel"
    assert worst <= B.K, f"worst row {worst:.3f} x the emulation's (budget {B.K})"


@pytest.mark.parametrize("case", B.FUSED_CASES, ids=[c["name"] for c in B.FUSED_CASES])
def test_fused_kernel_within_bf16_budget(case):
    _check(case, "fused")


@pytest.mark.parametrize("case", B.PER_OP_CASES, ids=[c["name"] for c in B.PER_OP_CASES])
def test_per_op_bf16_within_budget(case):
    _check(case, "per_op")


@pytest.mark.parametrize("name", ["rows-d256-t17", "rows-d128-t33"])
def test_fused_row_strides_through_c_abi(name):
    """avf_encoder_stack_fwd with ld_x > dim and out at ld_out > dim: one launch, the columns beyond dim untouched in both buffers,
    x unchanged (the fused kernel reads x and writes out), out within the budget."""
    case = next(c for c in B.FUSED_CASES if c["name"] == name)
    p, x, pos = B.make_inputs(case)
    m = _module(case, p, pos)
    n_seq, n_tok, dim = case["n_seq"], case["n_tok"], case["dim"]
    ld_x, ld_out = dim + 36, dim + 20
    xb = torch.full((n_seq * n_tok, ld_x), 7.25, device="cuda")
    xb[:, :dim] = (x + pos.repeat(n_seq, 1)).cuda()
    ob = torch.full((n_seq * n_tok, ld_out), -3.5, device="cuda")
    x0, o0 = xb.clone(), ob.clone()
    L = A._lib.lib()
    shape, packed = m.shape(n_seq, n_tok), m.packed()
    ws = AF.workspace(L.avf_encoder_workspace_bytes(ctypes.byref(shape), packed.mode), xb.device)
    n0 = _launches()
    rc = L.avf_encoder_stack_fwd(AF.AVF_BF16, ctypes.byref(shape), packed.array, AF._ptr(xb), ld_x, AF._ptr(ob), ld_out, AF._ptr(ws), ws.numel(),
                                 AF._stream())
    assert rc == 0, L.avf_last_error()
    torch.cuda.synchronize()
    assert _launches() - n0 == 1
    assert torch.equal(xb, x0)
    assert torch.equal(ob[:, dim:], o0[:, dim:])
    ref, emu = _references(name)
    got = B.row_rms(ob[:, :dim].double().cpu().view(n_seq, n_tok, dim) - ref)
    assert got.max().item() <= B.K * B.budget(emu["fused"], ref)
