"""The training heads at training batch sizes against fp64: the AU_former front forward and backward (batch and running statistics),
the eval fronts, the AU logits and their backward, the AU loss, the confusion counters of metrics.py, and the whole hot-path
backward at 64 clips.

Clip counts (head_oracle.CLIPS, 2 to 2305) reach every batch-sized loop and dispatch of the head kernels: the 8 row lanes of the
BatchNorm kernels empty, full and taking a second row; the 256 threads of au_bce_kernel taking one step or more; the dw_cat wgrad in
1, 2 and 3 split-K partials; the forward GEMM (N = 1536) and the dgrad GEMM (N = 512) at tile widths 64 and 128.  Every dispatch
threshold is derived from the device's SM count (test_clip_counts_reach_every_dispatch).

fp32 mode is held to 1e-4 of each tensor's max-abs, like tests/test_gpu_train.py.  bf16 mode is held to per-case budgets
(tests/head_oracle.py): the kernel's worst unit within K_HEAD times the bf16 emulation's worst unit, the median unit within [0.5, 2]
times the emulation's median.  K_HEAD = 1.5 x the largest worst-unit ratio that tools/head_budget_ratios.py measured over the 155
(case, tensor) pairs of the bf16 cases here on one B200 (1000 W limit, 1965 MHz max SM clock, profiles/r12_head_budget_ratios.json):
1.5 x 1.0018 (training front, running statistics, 2305 clips, dw_cat) = 1.503, rounded up to 1.51.  The median-unit ratios lie in
0.9996-1.0005: the emulation rounds where the kernels round, and the fp32 accumulation it leaves out is invisible next to bf16.  Statistics, running statistics, db_cat, the loss and dw_last, which are
fp32 sums in either mode, are held to fp32 summation bounds; integer results and single fp32 products are compared exactly.  Every
output the kernels write is surrounded by sentinel values that must survive the call."""
import ctypes
import functools
import os
import sys

import numpy as np
import pytest
import torch

import avformer_b200 as A
from oracle import avformer_oracle as O

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import head_oracle as H  # noqa: E402

pytestmark = pytest.mark.gpu
AF = A.functional
FP32_RTOL = 1e-4
SENT = -1.2345678e37          # sentinel around every output
GUARD = 64                    # sentinel elements before and after each output


@pytest.fixture(autouse=True)
def _no_tf32():
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False


@functools.lru_cache(maxsize=None)
def sms():
    return AF.device_info()["sm_count"]


def _L():
    return A._lib.lib()


def _rel(a, b, floor=0.0):
    b = b.double()
    return ((a.double().to(b.device) - b).abs().max() / max(b.abs().max().item(), floor, 1e-300)).item()


class Guarded:
    """An fp32 output of `rows` x `cols` (row stride ld >= cols) inside a buffer of sentinels."""

    def __init__(self, rows, cols, ld=None, init=None):
        self.rows, self.cols, self.ld = rows, cols, ld or cols
        self.buf = torch.full((2 * GUARD + rows * self.ld,), SENT, dtype=torch.float32, device="cuda")
        if init is not None:
            self.view.copy_(init.reshape(rows, cols))

    @property
    def view(self):
        return self.buf[GUARD:GUARD + self.rows * self.ld].view(self.rows, self.ld)[:, :self.cols]

    def ptr(self):
        return ctypes.c_void_p(self.buf.data_ptr() + 4 * GUARD)

    def untouched(self):
        b = self.buf.cpu()
        ok = bool((b[:GUARD] == SENT).all()) and bool((b[-GUARD:] == SENT).all())
        if self.ld > self.cols:
            ok = ok and bool((b[GUARD:GUARD + self.rows * self.ld].view(self.rows, self.ld)[:, self.cols:] == SENT).all())
        return ok


def _dirty(nbytes):
    return torch.full((nbytes + 4 * GUARD,), 0xFF, dtype=torch.uint8, device="cuda")     # NaN bytes: nothing may rely on zeroed memory


# ---------------------------------------------------------------------------------------------------------------------------------
# dispatch coverage
# ---------------------------------------------------------------------------------------------------------------------------------
def test_clip_counts_reach_every_dispatch():
    s = sms()
    n_out = H.N_AU * H.EMB_DIM
    splits = {H.wgrad_plan(n, s)[0] for n in H.CLIPS}
    max_splits = H.wgrad_plan(max(H.CLIPS), s)[0]
    assert {1, 2, max_splits} <= splits and max_splits >= 2, (s, sorted(splits))
    assert {H.gemm_tile_n(n, n_out, s) for n in H.CLIPS} >= {64, 128}, "forward GEMM (N = 1536) tile widths"
    assert {H.gemm_tile_n(n, H.IN_DIM, s) for n in H.CLIPS} >= {64, 128}, "dgrad GEMM (N = 512) tile widths"
    lanes = {(n < H.BN_LANES, n == H.BN_LANES, n > H.BN_LANES) for n in H.CLIPS}
    assert len(lanes) == 3, "BatchNorm row lanes: some empty, all full, a second row"
    assert {n * H.N_AU > H.BCE_THREADS for n in H.CLIPS} == {False, True}
    # the first clip count past each threshold is in the list
    for thr_hit in (lambda n: H.wgrad_plan(n, s)[0] > 1, lambda n: H.gemm_tile_n(n, n_out, s) > 64, lambda n: H.gemm_tile_n(n, H.IN_DIM, s) > 64,
                    lambda n: n * H.N_AU > H.BCE_THREADS):
        first = next(n for n in range(2, 100000) if thr_hit(n))
        assert first in H.CLIPS, f"the first clip count past a threshold ({first}) is not among {H.CLIPS}"


# ---------------------------------------------------------------------------------------------------------------------------------
# AU_former front, training forward + backward
# ---------------------------------------------------------------------------------------------------------------------------------
def _front_tensors(n, precision, batch_stats):
    seed = H.seed_of(f"front-{precision}-{int(batch_stats)}", n)
    p = H.front_params(seed)
    store, dx = H.front_inputs(n, seed, p)
    return p, store, dx


def front_train_call(n, mode, store, p, batch_stats, dx, momentum=0.1):
    """au_former_front_fwd_train + au_former_front_bwd through the C ABI with guarded outputs and dirty tape / workspace."""
    L = _L()
    in_dim, emb_dim = H.IN_DIM, H.EMB_DIM
    n_out = 12 * emb_dim
    emb = store.cuda()
    g, b, pos, bc = (p[k].cuda().contiguous() for k in ("gamma", "beta", "pos", "b"))
    w = AF.to_bf16(p["w"].cuda()) if mode == AF.AVF_BF16 else p["w"].cuda().contiguous()
    rm, rv = Guarded(1, in_dim, init=p["run_mean"].cuda()), Guarded(1, in_dim, init=p["run_var"].cuda())
    x = Guarded(n * 12, emb_dim)
    tb = L.avf_au_former_front_tape_bytes(mode, n, in_dim)
    tape = _dirty(tb)
    AF.check(L.avf_au_former_front_fwd_train(mode, AF._ptr(emb), emb.stride(0), AF._ptr(g), AF._ptr(b), rm.ptr(), rv.ptr(), int(batch_stats),
                                             float(momentum), AF._ptr(w), AF._ptr(bc), AF._ptr(pos), x.ptr(), n, in_dim, emb_dim,
                                             AF._ptr(tape), tb, AF._stream()), "au_former_front_fwd_train")
    ld_demb = in_dim + 24
    demb, dg, db = Guarded(n, in_dim, ld=ld_demb), Guarded(1, in_dim), Guarded(1, in_dim)
    dw, dbc = Guarded(n_out, in_dim), Guarded(1, n_out)
    wb = L.avf_au_former_front_bwd_workspace_bytes(mode, n, in_dim, emb_dim)
    ws = _dirty(wb)
    dxd = dx.cuda().contiguous()
    AF.check(L.avf_au_former_front_bwd(mode, AF._ptr(emb), emb.stride(0), AF._ptr(g), rm.ptr(), rv.ptr(), int(batch_stats), AF._ptr(w),
                                       AF._ptr(tape), tb, AF._ptr(dxd), demb.ptr(), ld_demb, dg.ptr(), db.ptr(), dw.ptr(), dbc.ptr(), n, in_dim,
                                       emb_dim, AF._ptr(ws), wb, AF._stream()), "au_former_front_bwd")
    torch.cuda.synchronize()
    off = -(-n * in_dim * (2 if mode == AF.AVF_BF16 else 4) // 256) * 256
    stats = tape[off:off + 2 * 2048].view(torch.float32)
    out = {"tokens": x.view.clone(), "mean": stats[:in_dim].clone(), "rstd": stats[512:512 + in_dim].clone(),
           "run_mean": rm.view[0].clone(), "run_var": rv.view[0].clone(), "demb": demb.view.clone(), "dgamma": dg.view[0].clone(),
           "dbeta": db.view[0].clone(), "dw_cat": dw.view.clone(), "db_cat": dbc.view[0].clone()}
    guards = {"tokens": x, "run_mean": rm, "run_var": rv, "demb": demb, "dgamma": dg, "dbeta": db, "dw_cat": dw, "db_cat": dbc}
    return out, guards, (emb, g, b, pos, bc, w, dxd)


def _check_stats(got, emb, p, batch_stats, ref, label):
    bnd = H.stat_bounds(emb, p, batch_stats)
    cpu = {k: v.double().cpu() for k, v in got.items()}
    if batch_stats:
        assert bool(((cpu["mean"] - ref["mean"].cpu()).abs() <= bnd["mean"]).all()), f"{label}: saved mean"
        assert bool(((cpu["rstd"] / ref["rstd"].cpu() - 1).abs() <= bnd["rstd_rel"]).all()), f"{label}: saved rstd"
        for k in ("run_mean", "run_var"):
            err = (cpu[k] - ref[k].cpu()).abs()
            assert bool((err <= bnd[k]).all()), f"{label}: {k} {float((err / bnd[k]).max()):.2f} x its fp32 bound"
    else:         # running statistics are read, not written
        assert torch.equal(got["run_mean"].cpu(), p["run_mean"]) and torch.equal(got["run_var"].cpu(), p["run_var"]), label


def run_front_case(n, precision, batch_stats):
    """-> {tensor: (worst ratio, median ratio | None)} for a bf16 case; asserts every fp32 / bound / sentinel check on the way."""
    mode = AF.AVF_BF16 if precision == "bf16" else AF.AVF_FP32
    p, store, dx = _front_tensors(n, precision, batch_stats)
    got, guards, (emb_d, g, b, pos, bc, w, dxd) = front_train_call(n, mode, store, p, batch_stats, dx)
    label = f"{precision} bs={int(batch_stats)} n={n}"
    for k, gd in guards.items():
        assert gd.untouched(), f"{label}: a sentinel around {k} was overwritten"
    emb = store[:, :H.IN_DIM].double().cuda()
    pd = {k: v.cuda() for k, v in p.items()}
    ref = H.front_reference(emb, pd, batch_stats, dx.cuda())
    _check_stats(got, store[:, :H.IN_DIM], p, batch_stats, ref, label)
    # db_cat (== dpos): an fp32 column sum of the fp32 dx in either mode
    dsum = dx.double().cuda().reshape(n, -1).abs().sum(0)
    assert bool(((got["db_cat"].double() - ref["db_cat"]).abs() <= H.gamma_sum(n) * dsum).all()), f"{label}: db_cat"
    assert torch.allclose(ref["dpos"].reshape(-1), ref["db_cat"], rtol=1e-12, atol=1e-12)
    # with 2 rows BatchNorm leaves only ~eps / var of demb's terms: it is held to fp32 cancellation (head_oracle.two_row_demb_bound)
    two_rows = batch_stats and n == 2
    if two_rows:
        emu = H.front_emulate(emb, pd, batch_stats, dx.cuda(), path="per_op" if mode == AF.AVF_BF16 else None)
        ratio = ((got["demb"].double() - ref["demb"]).abs() / H.two_row_demb_bound(emb, pd, emu)).max().item()
        assert ratio <= 1.0, f"{label}: demb of a 2-row batch at {ratio:.2f} x its fp32 cancellation bound"
    # the AF wrappers give the same bits
    run = (p["run_mean"].cuda().clone(), p["run_var"].cuda().clone())
    x2, tape2 = AF.au_former_front_train(emb_d[:, :H.IN_DIM], n, g, b, run[0], run[1], batch_stats, 0.1, w, bc, pos, mode)
    demb2, dg2, db2, dw2, dbc2 = AF.au_former_front_bwd(emb_d[:, :H.IN_DIM], n, g, run[0], run[1], batch_stats, w, tape2, dxd, mode)
    for k, v in (("tokens", x2), ("demb", demb2), ("dgamma", dg2), ("dbeta", db2), ("dw_cat", dw2), ("db_cat", dbc2)):
        assert torch.equal(v, got[k]), f"{label}: AF wrapper differs in {k}"
    names = ("tokens", "dgamma", "dbeta", "dw_cat") + (() if two_rows else ("demb",))
    if mode == AF.AVF_FP32:
        for k in names:
            r = _rel(got[k], ref[k])
            assert r < FP32_RTOL, f"{label}: {k} rel err {r:.3e}"
        return {}
    emu = H.front_emulate(emb, pd, batch_stats, dx.cuda(), path="per_op")
    return {k: H.ratios(k, got[k], emu[k], ref[k]) for k in names}


def _check_budget(r, label):
    for k, (worst, median) in r.items():
        assert worst <= H.K_HEAD, f"{label} {k}: worst unit {worst:.3f} x the emulation's (budget {H.K_HEAD})"
        if median is not None:
            lo, hi = H.MEDIAN_RATIO
            assert lo <= median <= hi, f"{label} {k}: median-unit ratio {median:.3f}: the emulation does not model the kernel"


@pytest.mark.parametrize("n", H.CLIPS)
@pytest.mark.parametrize("batch_stats", [True, False], ids=["batch", "running"])
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_au_former_front_train_against_fp64(precision, batch_stats, n):
    _check_budget(run_front_case(n, precision, batch_stats), f"{precision} bs={int(batch_stats)} n={n}")


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_au_former_front_one_clip_with_batch_statistics_launches_nothing(precision):
    mode = AF.AVF_BF16 if precision == "bf16" else AF.AVF_FP32
    p, store, dx = _front_tensors(2, precision, True)
    L = _L()
    emb = store[:1].cuda()
    g, b, pos, bc = (p[k].cuda().contiguous() for k in ("gamma", "beta", "pos", "b"))
    w = AF.to_bf16(p["w"].cuda()) if mode == AF.AVF_BF16 else p["w"].cuda().contiguous()
    rm, rv = Guarded(1, H.IN_DIM, init=p["run_mean"].cuda()), Guarded(1, H.IN_DIM, init=p["run_var"].cuda())
    x = Guarded(12, H.EMB_DIM)
    tb = L.avf_au_former_front_tape_bytes(mode, 1, H.IN_DIM)
    tape = _dirty(tb)
    tape0 = tape.clone()
    torch.cuda.synchronize()
    n0 = L.avf_launch_count()
    with pytest.raises(RuntimeError, match="more than one row"):
        AF.check(L.avf_au_former_front_fwd_train(mode, AF._ptr(emb), emb.stride(0), AF._ptr(g), AF._ptr(b), rm.ptr(), rv.ptr(), 1, 0.1, AF._ptr(w),
                                                 AF._ptr(bc), AF._ptr(pos), x.ptr(), 1, H.IN_DIM, H.EMB_DIM, AF._ptr(tape), tb, AF._stream()),
                 "au_former_front_fwd_train")
    torch.cuda.synchronize()
    assert L.avf_launch_count() == n0
    assert torch.equal(rm.view[0].cpu(), p["run_mean"]) and torch.equal(rv.view[0].cpu(), p["run_var"])
    assert bool((x.buf == SENT).all()) and torch.equal(tape, tape0)
    with pytest.raises(RuntimeError, match="more than one row"):
        AF.au_former_front_train(emb, 1, g, b, p["run_mean"].cuda(), p["run_var"].cuda(), True, 0.1, w, bc, pos, mode)


# ---------------------------------------------------------------------------------------------------------------------------------
# eval fronts: AU_former (12 tokens) and VA_former (2 tokens)
# ---------------------------------------------------------------------------------------------------------------------------------
def run_eval_front_case(n, precision, n_tok):
    mode = AF.AVF_BF16 if precision == "bf16" else AF.AVF_FP32
    seed = H.seed_of(f"eval-{precision}-{n_tok}", n)
    p = H.front_params(seed, n_tok=n_tok)
    store, _ = H.front_inputs(n, seed, H.front_params(seed))
    emb = store.cuda()
    bn = tuple(p[k].cuda() for k in ("gamma", "beta", "run_mean", "run_var"))
    w = AF.to_bf16(p["w"].cuda()) if mode == AF.AVF_BF16 else p["w"].cuda().contiguous()
    if n_tok == 12:
        got = AF.au_former_front(emb, emb.stride(0), n, bn, w, p["b"].cuda(), p["pos"].cuda(), mode)
    else:
        got = AF.token_front(emb, emb.stride(0), n, n_tok, bn, w, p["b"].cuda(), p["pos"].cuda(), mode)
    torch.cuda.synchronize()
    pd = {k: v.cuda() for k, v in p.items()}
    e64 = store[:, :H.IN_DIM].double().cuda()
    ref = H.front_reference(e64, pd, False)["tokens"]
    if mode == AF.AVF_FP32:
        r = _rel(got, ref)
        assert r < FP32_RTOL, f"eval front n_tok={n_tok} n={n}: rel err {r:.3e}"
        return {}
    return {"tokens": H.ratios("tokens", got, H.front_emulate(e64, pd, False, path="per_op")["tokens"], ref)}


@pytest.mark.parametrize("n", H.CLIPS)
@pytest.mark.parametrize("n_tok", [12, 2], ids=["au_former", "va_former"])
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_eval_fronts_against_fp64(precision, n_tok, n):
    _check_budget(run_eval_front_case(n, precision, n_tok), f"eval {precision} n_tok={n_tok} n={n}")


# ---------------------------------------------------------------------------------------------------------------------------------
# AU logits, forward and backward
# ---------------------------------------------------------------------------------------------------------------------------------
def _logit_inputs(n, dim):
    g = torch.Generator().manual_seed(H.seed_of(f"logits-{dim}", n))
    ld_x = dim + 12
    xs = torch.randn(n * 12, ld_x, generator=g)
    w_last = (2 * torch.rand(12, dim, generator=g) - 1) * dim ** -0.5
    dl = torch.randn(n, 21, generator=g) / (12.0 * n)
    return xs, w_last, dl


@pytest.mark.parametrize("n", H.CLIPS)
@pytest.mark.parametrize("dim", [128, 256])
def test_au_logits_forward_and_backward(dim, n):
    xs, w_last, dl = _logit_inputs(n, dim)
    xsd, wd, dld = xs.cuda(), w_last.cuda(), dl.cuda()
    x = xsd[:, :dim]                                   # ld_x = dim + 12 > dim
    assert x.stride(0) > dim and dld.stride(0) == 21
    out, dec = AF.au_logits(x, wd, n, want_decisions=True)
    torch.cuda.synchronize()
    x64, w64 = xs[:, :dim].double().reshape(n, 12, dim), w_last.double()
    ref = (x64 * w64).sum(-1)
    bound = (dim + 24) * H.EPS32 * (x64 * w64).abs().sum(-1)
    assert bool(((out[:, :12].double().cpu() - ref).abs() <= bound).all()), "au_logits outside its fp32 dot-product bound"
    assert float(out[:, 12:].abs().max()) == 0.0
    assert torch.equal(dec.cpu(), (out[:, :12] > 0).int().cpu())
    # backward through the C ABI: dx with a row stride and sentinels
    L = _L()
    ld_dx = dim + 8
    dxg, dwg = Guarded(n * 12, dim, ld=ld_dx), Guarded(12, dim)
    AF.check(L.avf_au_logits_bwd(AF._ptr(dld), 21, AF._ptr(x), x.stride(0), AF._ptr(wd), dxg.ptr(), ld_dx, dwg.ptr(), n, dim, AF._stream()),
             "au_logits_bwd")
    torch.cuda.synchronize()
    assert dxg.untouched() and dwg.untouched()
    want = (dld[:, :12].reshape(-1, 1) * wd.repeat(n, 1))          # one fp32 product per element
    assert torch.equal(dxg.view, want), "dx is not the fp32 product dl * w"
    dx64, dw64 = H.logits_bwd(dl, xs[:, :dim], w_last, n)
    bound = n * H.EPS32 * (dl[:, :12].double()[:, :, None].abs() * x64.abs()).sum(0)
    assert bool(((dwg.view.double().cpu() - dw64).abs() <= bound).all()), "dw_last outside n_clips * 2^-24 * sum|dl x|"
    # want_dx / want_dw subsets and the AF wrapper: the same bits
    dx_a, dw_a = AF.au_logits_bwd(dld, x, wd, n)
    dx_b, none_w = AF.au_logits_bwd(dld, x, wd, n, want_dw=False)
    none_x, dw_c = AF.au_logits_bwd(dld, x, wd, n, want_dx=False)
    assert none_w is None and none_x is None
    for t in (dx_a, dx_b):
        assert torch.equal(t, dxg.view)
    for t in (dw_a, dw_c):
        assert torch.equal(t, dwg.view)


# ---------------------------------------------------------------------------------------------------------------------------------
# AU loss
# ---------------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n", H.CLIPS)
@pytest.mark.parametrize("case", H.BCE_CASES)
def test_au_bce_loss_against_fp64(case, n):
    y_pred, labels = H.bce_inputs(n, case, H.seed_of(case, n))
    pw = torch.tensor(O.AU_POS_WEIGHT, dtype=torch.float32).cuda()
    yp = y_pred.cuda()
    loss, nv, grad = AF.au_bce_loss(yp, labels.cuda(), pw, want_grad=True)
    loss2, nv2, none = AF.au_bce_loss(yp, labels.cuda(), pw)
    torch.cuda.synchronize()
    ref_loss, ref_nv, ref_g = H.bce(y_pred, labels)
    loss_b, grad_b = H.bce_bounds(y_pred, labels)
    assert none is None and torch.equal(torch.stack([loss, nv]).view(torch.int32), torch.stack([loss2, nv2]).view(torch.int32))
    assert int(nv.item()) == ref_nv and float(nv.item()) == ref_nv
    keep = labels[:, 0] != -1.0
    g = grad.double().cpu()
    assert bool((g[~keep] == 0).all()), "an ignored row has a gradient"
    if ref_nv == 0:
        assert torch.isnan(loss).item() and bool((g == 0).all())
        return
    assert abs(loss.item() - ref_loss) <= loss_b, f"loss {loss.item()} vs {ref_loss} (bound {loss_b:.3e})"
    assert bool(((g - ref_g).abs() <= grad_b).all()), f"gradient: worst {float(((g - ref_g).abs() / grad_b.clamp_min(1e-300)).max()):.2f} x bound"


# ---------------------------------------------------------------------------------------------------------------------------------
# confusion counters (metrics.py, avf_au_confusion_update): past the 296-CTA grid's first stride
# ---------------------------------------------------------------------------------------------------------------------------------
def _confusion_cpu(pred, labels, thresh, ignore):
    c = np.zeros((12, 4), dtype=np.int64)
    for au in range(12):
        y, p = labels[:, au], pred[:, au] > thresh
        lab = y != ignore
        t = y == 1.0
        c[au] += [(lab & p & t).sum(), (lab & p & ~t).sum(), (lab & ~p & t).sum(), (lab & ~p & ~t).sum()]
    return c


@pytest.mark.parametrize("n_rows", [6314, 6400, 20011])
def test_confusion_counters_exact_past_the_grid_stride(n_rows):
    from avformer_b200.metrics import MultiLabelAccF1
    g = torch.Generator().manual_seed(n_rows)
    logits = torch.randn(n_rows, 21, generator=g)
    labels = (torch.rand(n_rows, 12, generator=g) < 0.3).float()
    labels[torch.rand(n_rows, 12, generator=g) < 0.1] = -1.0
    m = MultiLabelAccF1(ignore_index=-1)
    m.update_from_logits(logits.cuda(), labels.cuda())
    want = _confusion_cpu(logits.numpy(), labels.numpy(), 0.0, -1.0)
    assert np.array_equal(m.confusion(), want)
    dec = (logits[:, :12] > 0).float()
    m.update(dec.numpy(), labels.numpy())                          # accumulates, threshold 0.5 on 0/1 predictions
    assert np.array_equal(m.confusion(), 2 * want)
    assert int(m.confusion().sum()) == 2 * int((labels != -1).sum())


# ---------------------------------------------------------------------------------------------------------------------------------
# whole hot path at the training batch size
# ---------------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("precision,batch_stats", [("fp32", False), ("fp32", True), ("bf16", False), ("bf16", True)])
def test_hot_path_gradients_against_oracle_at_64_clips(precision, batch_stats):
    """tests/test_gpu_train.py::test_hot_path_gradients_against_oracle at B = 64 (bench.py --mode train), with its tolerances."""
    T, B, seed, w_sf = 16, 64, 78, 3.0
    sd = O.make_state_dict(seed, T, hot_path_only=True)
    stage3, frame, audio = O.synth_hot_path_inputs(seed, B, T)
    labels = O.synth_inputs(seed, B, T, image=8)[2]
    labels[1, 0] = -1.0
    labels[40:43, 0] = -1.0
    ref_loss, ref_g, ref_in, ref_out = O.hot_path_grads(stage3.double(), frame.double(), audio.double(), labels.double(),
                                                        O.cast_params(sd, torch.float64), T, batch_stats, w_sf)
    m = A.TwoStreamAuralVisualFormer(video_pretrained=False, audio_pretrained=False, task="AU").set_clip_length(T)
    m.load_state_dict(O.make_state_dict(seed, T), strict=True)
    m = m.cuda().set_precision(precision).set_dropout(0.0)
    m.train(batch_stats)
    for p_ in m.parameters():
        p_.grad = None
    ins = [t.cuda().requires_grad_(True) for t in (stage3, frame, audio)]
    s_out, out21 = m.hot_path_train(*ins)
    loss = m.get_au_loss(out21, labels.cuda()) + w_sf * (s_out * O.sformer_probe(s_out.shape).cuda()).mean()
    loss.backward()
    torch.cuda.synchronize()
    tol = FP32_RTOL if precision == "fp32" else 3e-2
    assert abs(loss.item() - ref_loss.item()) < (1e-4 if precision == "fp32" else 2e-2) * max(1.0, abs(ref_loss.item()))
    for t, k in zip(ins, ("stage3", "frame_feat", "audio_feat")):
        assert _rel(t.grad, ref_in[k]) < tol, f"d{k}: {_rel(t.grad, ref_in[k]):.3e}"
    named = dict(m.named_parameters())
    summand = ref_in["tformer_cls"].abs().max().item()
    checked, num, den, worst = 0, 0.0, 0.0, {}
    for k, rg in ref_g.items():
        if O.is_backbone_key(k) or rg.abs().max() == 0:
            continue
        diff = named[k].grad.double().cpu() - rg
        num += float((diff * diff).sum())
        den += float((rg * rg).sum())
        in_t = batch_stats and ".t_former." in k
        floor = summand if (in_t and (rg.dim() == 1 or "cls_token" in k or "pos_embedding" in k)) else 0.0
        r = diff.abs().max().item() / max(rg.abs().max().item(), floor)
        lim = 5 * tol if in_t else (2 * tol if batch_stats else tol)
        worst[k] = r / lim
        assert r < lim, f"{k}: rel err {r:.3e} (|ref|max {rg.abs().max().item():.3e}, floor {floor:.3e})"
        checked += 1
    top = sorted(worst.items(), key=lambda kv: -kv[1])[:3]
    print(f"\nB=64 {precision} batch_stats={batch_stats}: largest error / tolerance " + ", ".join(f"{k} {v:.2f}" for k, v in top))
    assert (num / den) ** 0.5 < (tol if precision == "fp32" else 2e-2)
    assert checked >= 150
    if batch_stats:
        rm, rv = O.bn_running_update(ref_out["tformer_cls"], sd["video_model.au_head.AU_BN1.running_mean"].double(),
                                     sd["video_model.au_head.AU_BN1.running_var"].double())
        bn = m.video_model.au_head.AU_BN1
        st = 1e-4 if precision == "fp32" else 2e-2
        assert _rel(bn.running_mean, rm) < st and _rel(bn.running_var, rv) < st
