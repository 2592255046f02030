"""The bf16 training backward against per-case error budgets (tests/bf16_bwd_oracle.py): the attention backward kernel at every
instantiation, masked and unmasked, the encoder-stack backward at the geometry of every module the training step runs, at split-K
edges and at the benchmarked training size, and gradient accumulation into FusedAdam's flat gradient bucket.

A case passes when, for every tensor, the kernel's worst unit (token row of dx, row of a weight gradient, (row, Q/K/V, head) slice of
dqkv, whole vector) is within K_BWD times the bf16 emulation's worst unit, both as RMS error against fp64, and the median unit within
[0.5, 2] times the emulation's median: the emulation has to model the kernel, not just bound it.  The stack references (fp64 and
emulated) are plain torch in float64; they run on the GPU, where the benchmark-size case takes seconds instead of minutes."""
import functools
import os
import sys

import pytest
import torch

import avformer_b200 as A
from oracle import avformer_oracle as O

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import bf16_bwd_oracle as BB  # noqa: E402

pytestmark = pytest.mark.gpu
AF = A.functional


def _check(ratios, label):
    for k, (worst, median) in ratios.items():
        assert worst <= BB.K_BWD, f"{label} {k}: worst unit {worst:.3f} x the emulation's (budget {BB.K_BWD})"
        if median is not None:
            lo, hi = BB.MEDIAN_RATIO
            assert lo <= median <= hi, f"{label} {k}: median-unit ratio {median:.3f}: the emulation does not model the kernel"


# ---------------------------------------------------------------------------------------------------------------------------------
# attention backward kernel
# ---------------------------------------------------------------------------------------------------------------------------------
@functools.lru_cache(maxsize=None)
def _att_refs(name):
    case = next(c for c in BB.ATT_CASES if c["name"] == name)
    return BB.att_references(case)


def run_att_case(case):
    """-> {"dqkv": (worst ratio, median ratio)} of attention_bwd_mma_kernel on the case."""
    qkv, dout, keep = BB.att_inputs(case)
    got = AF.attention_bwd(qkv.cuda(), dout.cuda(), case["n_seq"], case["n_tok"], case["heads"], case["dh"],
                           keep=keep.cuda() if keep is not None else None)
    torch.cuda.synchronize()
    ref, emu = _att_refs(case["name"])
    got = got.double().cpu()
    if keep is not None:          # a dropped token's dQ (its dS row is 0) and dK (no kept query sees it) are exactly 0
        dropped = ~keep.reshape(-1)
        assert not bool(got[dropped, :2 * case["heads"] * case["dh"]].any()), "dQ / dK of a dropped token is not 0"
    return {"dqkv": BB.ratios("dqkv", got, emu, ref, case["heads"])}


@pytest.mark.parametrize("case", BB.ATT_CASES, ids=[c["name"] for c in BB.ATT_CASES])
def test_attention_bwd_kernel_within_bf16_budget(case):
    _check(run_att_case(case), case["name"])


# ---------------------------------------------------------------------------------------------------------------------------------
# encoder-stack backward
# ---------------------------------------------------------------------------------------------------------------------------------
@functools.lru_cache(maxsize=None)
def _stack_refs(name):
    case = next(c for c in BB.STACK_CASES if c["name"] == name)
    return BB.stack_reference(case, device="cuda"), BB.stack_reference(case, path="per_op", device="cuda")


def run_stack_case(case):
    """encoder_stack_fwd_train + encoder_stack_bwd_ on a bf16 A.Transformer (dropout 0) -> {tensor: (worst ratio, median ratio)}."""
    p, x, dy, keep = BB.stack_inputs(case)
    n_seq, n_tok, depth = case["n_seq"], case["n_tok"], case["depth"]
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    plans = [BB.splitk_plan(m, n, n_seq * n_tok, sms) for m, n in BB.wgrad_shapes(case)]
    if case["splitk"] == "one":
        assert all(s == 1 for s, _, _ in plans), plans
    elif case["splitk"] == "short":
        assert all(s > 1 and last < per for s, last, per in plans), plans
    m = A.Transformer(case["dim"], depth, 8, case["dh"], case["mlp"])
    m.load_state_dict(p, strict=True)
    m.precision = "bf16"
    m = m.cuda()
    packed, shape = m.packed(), m.shape(n_seq, n_tok)
    kc = keep.cuda() if keep is not None else None
    _, tape = AF.encoder_stack_fwd_train(x.cuda(), packed, shape, keep=kc)
    dx, grads = AF.encoder_stack_bwd_(dy.cuda().clone(), packed, shape, tape, [True] * (11 * depth), keep=kc)
    torch.cuda.synchronize()
    got = {"dx": dx}
    got.update(zip(BB.grad_names(depth), grads))
    ref, emu = _stack_refs(case["name"])
    return BB.stack_ratios(got, emu, ref)


@pytest.mark.parametrize("case", BB.STACK_CASES, ids=[c["name"] for c in BB.STACK_CASES])
def test_encoder_stack_bwd_within_bf16_budget(case):
    _check(run_stack_case(case), case["name"])


# ---------------------------------------------------------------------------------------------------------------------------------
# gradient accumulation into FusedAdam's bucket
# ---------------------------------------------------------------------------------------------------------------------------------
ACCUM_RTOL = 1e-5        # fp32 reassociation: (0 + g1) + g2 in the kernels against g1 + g2 in autograd, per tensor's max-abs


@pytest.mark.parametrize("precision", ["bf16", "fp32"])
def test_bf16_and_fp32_gradient_accumulation_into_fused_adam_buckets(precision):
    """Two backward passes per optimiser step.  Under FusedAdam every hot-path gradient kernel adds into the flat bucket (split-K
    reduce with accumulate, colsum and the LayerNorm column sums with beta = 1, the multi-tensor hand-over); without it torch adds
    the gradients the kernels return.  Both must agree to fp32 reassociation.  5 clips give the AU_formers and the fusion head 60
    token rows: their wgrads run with one split, the `splits == 1 && accumulate` path."""
    T, n_clips, seed, w_sf = 16, 5, 61, 3.0
    sd = O.make_state_dict(seed, T)
    batches = [(O.synth_hot_path_inputs(seed + i, n_clips, T), O.synth_inputs(seed + i, n_clips, T, image=8)[2]) for i in range(2)]
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    au = dict(dim=128, dh=32, mlp=256)
    assert all(BB.splitk_plan(m, n, n_clips * 12, sms)[0] == 1 for m, n in BB.wgrad_shapes(au))

    def model():
        m = A.TwoStreamAuralVisualFormer(video_pretrained=False, audio_pretrained=False, task="AU").set_clip_length(T)
        m.load_state_dict(sd, strict=True)
        return m.cuda().set_precision(precision).set_dropout(0.0).eval()

    def hot(m):
        return {k: p_ for k, p_ in m.named_parameters() if not O.is_backbone_key(k)}

    def two_backwards(m):
        for (stage3, frame, audio), labels in batches:
            s_out, out21 = m.hot_path_train(stage3.cuda(), frame.cuda(), audio.cuda())
            loss = m.get_au_loss(out21, labels.cuda()) + w_sf * (s_out * O.sformer_probe(s_out.shape).cuda()).mean()
            loss.backward()
        torch.cuda.synchronize()

    fused, plain = model(), model()
    # FusedAdam builds its flat bucket at the first step() from the parameters that have a gradient: one backward and a step at
    # lr = 0 (parameters unchanged) make every gradient-receiving hot-path parameter's .grad a view of the bucket
    opt = A.FusedAdam(list(hot(fused).values()), lr=0.0)
    s_out, out21 = fused.hot_path_train(*(t.cuda() for t in batches[0][0]))
    (fused.get_au_loss(out21, batches[0][1].cuda()) + w_sf * (s_out * O.sformer_probe(s_out.shape).cuda()).mean()).backward()
    opt.step()
    opt.zero_grad()
    bucketed = [k for k, p_ in hot(fused).items() if p_.grad is not None]
    assert len(bucketed) >= 150 and all(getattr(hot(fused)[k], "_avf_direct_grad", False) for k in bucketed)
    assert all(torch.equal(hot(fused)[k], hot(plain)[k]) for k in bucketed)
    assert all(float(hot(fused)[k].grad.abs().max()) == 0.0 for k in bucketed)
    for p_ in plain.parameters():
        p_.grad = None
    two_backwards(fused)
    two_backwards(plain)
    got, ref = hot(fused), hot(plain)
    worst, checked = 0.0, 0
    for k, rp in ref.items():
        if rp.grad is None:
            assert got[k].grad is None or float(got[k].grad.abs().max()) == 0.0, k
            continue
        r = rp.grad.double()
        scale = float(r.abs().max())
        if scale == 0.0:
            continue
        err = float((got[k].grad.double() - r).abs().max()) / scale
        worst = max(worst, err)
        assert err <= ACCUM_RTOL, f"{k}: {err:.3e} of max-abs"
        checked += 1
    print(f"\n{precision}: {checked} hot-path gradients, worst difference {worst:.3e} of max-abs (tolerance {ACCUM_RTOL:.0e})")
    assert checked >= 150
