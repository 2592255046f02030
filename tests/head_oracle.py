"""fp64 references, bf16 emulation and inputs for the training heads at training batch sizes.  TEST INFRASTRUCTURE ONLY, shared by
tests/test_gpu_head_train.py (GPU) and tests/test_head_budget_sensitivity.py (CPU).

Covered: the AU_former front (BatchNorm1d with batch or running statistics -> 12 stacked Linear(512,128) -> + pos), forward and
backward; the AU logits and their backward; the AU loss (AULoss, models/loss.py:75-103) and its gradient.

bf16 rounding points of the head path, modelled by ``path="per_op"``:
  * the BatchNorm output stored on the tape, ``xb = bf(BN(emb))``: bn_train_fwd_kernel (avf_train.cu:569) with batch statistics,
    bn_rows_kernel (avf_rowops.cu:69-70) with running ones;
  * ``w_cat``, the bf16 image of the 12 stacked projections (heads.py:23);
  * the incoming token gradient ``dx``, cast to bf16 (avf_train_api.cu:407) before the dw_cat wgrad (:416) and the dgrad (:420).
Not rounded: the column sum db_cat (fp32 over fp32 dx, :415), the dgrad output and the BatchNorm backward (fp32, avf_train.cu:573-613,
which recomputes x-hat from the fp32 emb).  fp32 accumulation inside the GEMMs is not modelled: it sits far below bf16 rounding.

Budgets: a bf16 case passes when the kernel's worst unit (token row of the forward, clip row of demb, output row of dw_cat, the whole
vector of dgamma / dbeta) is within K_HEAD times the emulation's worst unit, both as RMS error against fp64, and the median unit is
within [0.5, 2] times the emulation's median.  Sums the kernels take in fp32 whatever the mode (batch statistics, running
statistics, db_cat, the loss, dw_last) are held to an fp32 summation bound instead (``gamma_sum``).

``bug`` names one deliberate error, computed in fp64; tests/test_head_budget_sensitivity.py shows that each misses its check."""
import math

import numpy as np
import torch

from oracle import avformer_oracle as O

# A bf16 case passes when worst_unit(kernel) <= K_HEAD * worst_unit(emulation).  K_HEAD = 1.5 x the largest kernel / emulation ratio
# over every bf16 case and tensor of tests/test_gpu_head_train.py, rounded up, measured on one B200 (1000 W limit, 1965 MHz max SM
# clock): 1.0018 (training front, running statistics, 2305 clips, dw_cat); median-unit ratios 0.9996-1.0005
# (profiles/r12_head_budget_ratios.json).
K_HEAD = 1.51
MEDIAN_RATIO = (0.5, 2.0)

CLIPS = (2, 3, 7, 8, 9, 21, 22, 64, 65, 129, 512, 769, 2305)
IN_DIM, EMB_DIM, N_AU = 512, 128, 12
LD_EMB = 531                 # emb is a strided view with an odd row stride (the model reads the TFormer's cls rows in place)
BM, BK = 128, 64             # avf_gemm_umma.cu: tile M and K block of the tcgen05 GEMM
BN_LANES = 8                 # bn_train_fwd_kernel / bn_bwd_kernel: 8 row lanes per 32-column block (avf_train.cu:523-613)
BCE_THREADS = 256            # au_bce_kernel: one CTA of 256 threads (avf_rowops.cu:677)
EPS32 = 2.0 ** -24

MUTANTS = ("running_var_biased", "bn_bwd_no_mean_dy", "bn_bwd_no_xhat_term", "dgamma_unnormalised_x", "loss_nvalid_every_column",
           "bce_first_256_entries", "dw_last_first_8_clips", "splitk_drop_last_partial")


def bf(t):
    """Round to bf16 (nearest even) and return in t's dtype."""
    return t.to(torch.float32).to(torch.bfloat16).to(t.dtype)


# ---------------------------------------------------------------------------------------------------------------------------------
# dispatch of the head's GEMMs (avf_gemm_umma.cu:537-574), from the device's SM count
# ---------------------------------------------------------------------------------------------------------------------------------
def wgrad_plan(n_clips, sms, m=N_AU * EMB_DIM, n=IN_DIM):
    """(splits, K blocks per split) of the dw_cat wgrad C[m, n] = dx^T xb over K = n_clips rows (avf_gemm_umma.cu:542-546)."""
    bn = 128 if n % 128 == 0 else 64
    mn_tiles = -(-m // BM) * (n // bn)
    kblocks = -(-n_clips // BK)
    splits = max(1, min(kblocks, sms // max(1, mn_tiles)))
    per = -(-kblocks // splits)
    return -(-kblocks // per), per


def gemm_tile_n(m, n, sms, bf16_out=False):
    """Tile width BN of the non-transposed GEMM C[m, n] (avf_gemm_umma.cu:569-574): the forward (n = 1536) and the dgrad (n = 512)."""
    m_tiles = -(-m // BM)
    if n % 256 == 0 and m_tiles * (n // 256) * 5 >= (4 if bf16_out else 10) * sms:
        return 256
    if n % 128 == 0 and m_tiles * (n // 128) >= sms:
        return 128
    if n % 128 == 0 and n // 128 * m_tiles >= sms // 2 and n >= 512:
        return 128
    return 64


def gamma_sum(n_terms):
    """fp32 summation bound factor: a sequential sum of n_terms, the tree of the partial sums and a few roundings of the operands."""
    return (n_terms + 24) * EPS32


# ---------------------------------------------------------------------------------------------------------------------------------
# inputs
# ---------------------------------------------------------------------------------------------------------------------------------
def _gen(seed):
    return torch.Generator().manual_seed(int(seed))


def front_params(seed, n_tok=N_AU, emb_dim=EMB_DIM, in_dim=IN_DIM):
    """fp32 parameters of one front: BatchNorm gamma 1 + 0.3 randn, beta 0.5 randn, running mean 0.5 randn, running var in [0.2, 1];
    Linear weights and biases uniform in +-1/sqrt(in_dim) (nn.Linear's initialisation); pos randn."""
    g = _gen(seed)
    s = in_dim ** -0.5
    return {"gamma": 1.0 + 0.3 * torch.randn(in_dim, generator=g), "beta": 0.5 * torch.randn(in_dim, generator=g),
            "run_mean": 0.5 * torch.randn(in_dim, generator=g), "run_var": 0.2 + 0.8 * torch.rand(in_dim, generator=g),
            "w": (2 * torch.rand(n_tok * emb_dim, in_dim, generator=g) - 1) * s, "b": (2 * torch.rand(n_tok * emb_dim, generator=g) - 1) * s,
            "pos": torch.randn(n_tok, emb_dim, generator=g)}


def front_inputs(n_clips, seed, p, in_dim=IN_DIM):
    """(emb_store [n_clips, LD_EMB] fp32 whose first in_dim columns are emb, dx [n_clips * 12, 128] fp32).

    emb columns have their own offset (0.5 randn) and scale (1-2), so batch and running statistics differ.  dx = 0.5 randn + a
    per-column offset common to every clip + 0.5 x-hat w^T: the offset makes mean(dy) of the BatchNorm backward matter, the last
    term (x-hat of the batch) makes mean(dy x-hat) matter, as in a trained model whose gradient follows its input."""
    g = _gen(seed * 7919 + n_clips)
    store = torch.randn(n_clips, LD_EMB, generator=g)
    col_off, col_scale = 0.5 * torch.randn(in_dim, generator=g), 1.0 + torch.rand(in_dim, generator=g)
    store[:, :in_dim] = store[:, :in_dim] * col_scale + col_off
    emb = store[:, :in_dim].double()
    xhat = (emb - emb.mean(0)) / emb.std(0, unbiased=False).clamp_min(1e-3)
    n_out = p["w"].shape[0]
    dx = 0.5 * torch.randn(n_clips, n_out, generator=g) + torch.randn(1, n_out, generator=g) + (0.5 * xhat @ p["w"].double().t()).float()
    return store, dx.reshape(-1, EMB_DIM)


def bce_inputs(n_clips, case, seed):
    """(y_pred [n, 21] fp32, labels [n, 12] fp32) for one label case: "none" (no ignored row), "one" (row 0 ignored), "all_but_one"
    (every row but the last ignored), "all" (every row ignored), "minus1_other_col" (-1 in columns 1-11 of valid rows).  Logits are
    randn scaled up to +-30, so softplus and sigmoid are used far from 0 too."""
    g = _gen(seed * 31 + n_clips)
    y_pred = torch.randn(n_clips, 21, generator=g) * (1.0 + 9.0 * torch.rand(n_clips, 1, generator=g))
    y_pred[:, :12] = y_pred[:, :12].clamp(-30.0, 30.0)
    y_pred[0, :3] = torch.tensor([30.0, -30.0, 0.0])
    labels = (torch.rand(n_clips, 12, generator=g) < 0.4).float()
    if case == "one":
        labels[0, 0] = -1.0
    elif case == "all_but_one":
        labels[:-1, 0] = -1.0
    elif case == "all":
        labels[:, 0] = -1.0
    elif case == "minus1_other_col":
        labels[:, 1:][torch.rand(n_clips, 11, generator=g) < 0.2] = -1.0
    return y_pred, labels


BCE_CASES = ("none", "one", "all_but_one", "all", "minus1_other_col")


# ---------------------------------------------------------------------------------------------------------------------------------
# AU_former front: fp64 autograd reference, hand-written backward with the kernels' rounding points
# ---------------------------------------------------------------------------------------------------------------------------------
def front_forward(emb, gamma, beta, w, b, pos, batch_stats, run_mean=None, run_var=None):
    """models/heads.py:293-323 restated: BatchNorm1d (biased batch variance with batch statistics) -> 12 stacked Linear -> + pos.
    Returns tokens [n * n_tok, emb_dim]."""
    if batch_stats:
        mu, var = emb.mean(0), emb.var(0, unbiased=False)
    else:
        mu, var = run_mean, run_var
    e = (emb - mu) / torch.sqrt(var + 1e-5) * gamma + beta
    n, n_tok = emb.shape[0], pos.shape[0]
    return ((e @ w.t() + b).reshape(n, n_tok, -1) + pos).reshape(n * n_tok, -1)


def front_reference(emb, p, batch_stats, dx=None, momentum=0.1):
    """fp64 autograd over front_forward: {tokens, mean, rstd, run_mean, run_var} and, with dx, {demb, dgamma, dbeta, dw_cat, db_cat}."""
    q = {k: v.double().detach().clone() for k, v in p.items()}
    emb = emb.double().detach().clone().requires_grad_(dx is not None)
    for k in ("gamma", "beta", "w", "b", "pos"):
        q[k].requires_grad_(dx is not None)
    tok = front_forward(emb, q["gamma"], q["beta"], q["w"], q["b"], q["pos"], batch_stats, q["run_mean"], q["run_var"])
    e = emb.detach()
    if batch_stats:
        mu, var = e.mean(0), e.var(0, unbiased=False)
        rm, rv = O.bn_running_update(e, q["run_mean"], q["run_var"], momentum)
    else:
        mu, var, rm, rv = q["run_mean"], q["run_var"], q["run_mean"], q["run_var"]
    out = {"tokens": tok.detach(), "mean": mu, "rstd": 1.0 / torch.sqrt(var + 1e-5), "run_mean": rm, "run_var": rv}
    if dx is not None:
        tok.backward(dx.double())
        out.update(demb=emb.grad, dgamma=q["gamma"].grad, dbeta=q["beta"].grad, dw_cat=q["w"].grad, db_cat=q["b"].grad,
                   dpos=q["pos"].grad)
    return out


def front_emulate(emb, p, batch_stats, dx=None, path=None, bug=None, momentum=0.1, sms=148):
    """The same quantities as front_reference from a hand-written backward in fp64.  path="per_op" rounds where the bf16 path rounds
    (module docstring); ``bug`` is one of MUTANTS (the front ones)."""
    r = bf if path else (lambda t: t)
    emb = emb.double()
    q = {k: v.double() for k, v in p.items()}
    n = emb.shape[0]
    if batch_stats:
        mu, var_b = emb.mean(0), emb.var(0, unbiased=False)
        var_run = var_b if bug == "running_var_biased" else emb.var(0, unbiased=True)
        rm = (1 - momentum) * q["run_mean"] + momentum * mu
        rv = (1 - momentum) * q["run_var"] + momentum * var_run
    else:
        mu, var_b, rm, rv = q["run_mean"], q["run_var"], q["run_mean"], q["run_var"]
    rstd = 1.0 / torch.sqrt(var_b + 1e-5)
    xhat = (emb - mu) * rstd
    xb = r(xhat * q["gamma"] + q["beta"])                                  # the tape (avf_train.cu:569, avf_rowops.cu:69-70)
    w = r(q["w"])                                                          # bf16 image of w_cat (heads.py:23)
    n_tok = q["pos"].shape[0]
    tok = ((xb @ w.t() + q["b"]).reshape(n, n_tok, -1) + q["pos"]).reshape(n * n_tok, -1)
    out = {"tokens": tok, "mean": mu, "rstd": rstd, "run_mean": rm, "run_var": rv}
    if dx is None:
        return out
    d = dx.double().reshape(n, -1)
    out["db_cat"] = d.sum(0)                                               # fp32 column sum of fp32 dx (avf_train_api.cu:415)
    dxo = r(d)                                                             # bf16 GEMM operand (avf_train_api.cu:407)
    if bug == "splitk_drop_last_partial":                                  # the reduction leaves the last split's partial tile out
        splits, per = wgrad_plan(n, sms, m=d.shape[1], n=xb.shape[1])
        if splits > 1:
            dxo = dxo.clone()
            dxo[(splits - 1) * per * BK:] = 0.0
    out["dw_cat"] = dxo.t() @ xb                                           # wgrad (:416)
    dy = r(d) @ w                                                          # dgrad, fp32 output (:420)
    xh = (emb - mu) * rstd                                                 # bn_bwd_kernel recomputes x-hat from the fp32 emb (avf_train.cu:590)
    out["dbeta"] = dy.sum(0)
    out["dgamma"] = (dy * ((emb - mu) if bug == "dgamma_unnormalised_x" else xh)).sum(0)
    if batch_stats:
        m1 = 0.0 if bug == "bn_bwd_no_mean_dy" else dy.mean(0)
        m2 = 0.0 if bug == "bn_bwd_no_xhat_term" else (dy * xh).mean(0)
        out["demb"] = q["gamma"] * rstd * (dy - m1 - xh * m2)
    else:
        out["demb"] = q["gamma"] * rstd * dy
    out["dpos"] = out["db_cat"].reshape(n_tok, -1)
    out["dy"] = dy
    return out


# ---------------------------------------------------------------------------------------------------------------------------------
# AU logits and the loss
# ---------------------------------------------------------------------------------------------------------------------------------
def logits_bwd(dl, x, w_last, n_clips, bug=None):
    """(dx [n*12, dim], dw_last [12, dim]) in fp64: dx[c*12+i] = dl[c,i] w[i];  dw[i] = sum_c dl[c,i] x[c*12+i]  (avf_train.cu:498-520)."""
    dl = dl[:, :N_AU].double()
    x = x.double().reshape(n_clips, N_AU, -1)
    w = w_last.double()
    dx = (dl[:, :, None] * w[None]).reshape(n_clips * N_AU, -1)
    use = slice(0, 8) if bug == "dw_last_first_8_clips" else slice(None)
    dw = (dl[use, :, None] * x[use]).sum(0)
    return dx, dw


def bce(y_pred, labels, bug=None):
    """(loss, n_valid, dlogits [n, 12]) of AULoss in fp64 (O.au_loss / O.au_loss_grad), with the loss mutants of au_bce_kernel."""
    x = y_pred[:, :N_AU].double()
    y = labels.double()
    n = x.shape[0]
    keep = y[:, 0] != -1.0
    w = torch.tensor(O.AU_POS_WEIGHT, dtype=torch.float64)
    n_valid = int(keep.sum())
    if n_valid:
        loss = O.au_loss(x, y).item()
        grad = O.au_loss_grad(x, y)
    else:                                  # .mean() of an empty tensor; every gradient entry is exactly 0
        loss, grad = math.nan, torch.zeros_like(x)
    if bug == "loss_nvalid_every_column":  # the count is taken in every column instead of once per row
        return loss, 12 * n_valid, grad
    if bug == "bce_first_256_entries":     # the strided loops stop after the first 256 entries (one step of one CTA)
        flat = torch.arange(n * N_AU).reshape(n, N_AU) < BCE_THREADS
        k = keep[:, None] & flat
        nv = int((k[:, 0]).sum())
        term = -(w * y * torch.nn.functional.logsigmoid(x) + (1.0 - y) * torch.nn.functional.logsigmoid(-x))
        loss = float((term * k).sum() / (12.0 * nv)) if nv else math.nan
        s = torch.sigmoid(x)
        g = (s * (1.0 + (w - 1.0) * y) - w * y) / (12.0 * max(nv, 1))
        return loss, nv, g * k
    return loss, n_valid, grad


def bce_bounds(y_pred, labels):
    """(loss bound, per-element gradient bound [n, 12]) for au_bce_kernel's fp32 evaluation: each term of the loss and of the gradient
    carries a few ulps of expf / log1pf (8 ulps allowed per term), the loss sum a 256-way strided sequential sum, a warp tree and an
    8-way final sum."""
    x = y_pred[:, :N_AU].double()
    y = labels.double()
    keep = (y[:, 0] != -1.0)[:, None]
    nv = int(keep.sum())
    w = torch.tensor(O.AU_POS_WEIGHT, dtype=torch.float64)
    sp = torch.nn.functional.softplus(-x)
    term = ((1.0 - y) * x).abs() + ((1.0 + (w - 1.0) * y) * sp).abs()
    n_terms = -(-x.numel() // BCE_THREADS)
    loss_b = (gamma_sum(n_terms) + 8 * EPS32) * float((term * keep).sum()) / (12.0 * max(nv, 1))
    s = torch.sigmoid(x)
    grad_b = 8 * EPS32 * ((s * (1.0 + (w - 1.0) * y)).abs() + (w * y).abs()) / (12.0 * max(nv, 1)) * keep
    return loss_b, grad_b


# ---------------------------------------------------------------------------------------------------------------------------------
# error units and budgets
# ---------------------------------------------------------------------------------------------------------------------------------
ROW_UNITS = ("tokens", "demb", "dw_cat")      # per token row / clip row / output row
VEC_UNITS = ("dgamma", "dbeta")               # the whole vector is one unit
BUDGET_TENSORS = ROW_UNITS + VEC_UNITS


def units(name, t):
    t = t.double()
    if name in ROW_UNITS:
        return t.reshape(t.shape[0], -1).pow(2).mean(-1).sqrt()
    return t.pow(2).mean().sqrt().reshape(1)


def ratios(name, got, emu, ref):
    """(worst-unit ratio, median-unit ratio | None) of got's error against the emulation's, per unit RMS against fp64.  The floor 1e-6
    of the reference's RMS keeps a unit the emulation rounds exactly from dividing by 0."""
    got, emu, ref = got.double().to(ref.device), emu.double().to(ref.device), ref.double()
    eg, ee = units(name, got - ref), units(name, emu - ref)
    floor = 1e-6 * ref.pow(2).mean().sqrt().item()
    worst = eg.max().item() / max(ee.max().item(), floor)
    if eg.numel() == 1:
        return worst, None
    nz = ee > 0
    if not bool(nz.any()):
        return worst, None
    return worst, (eg[nz].median() / ee[nz].median().clamp_min(floor)).item()


def stat_bounds(emb, p, batch_stats, momentum=0.1):
    """Per-column fp32 bounds of the saved mean, the saved rstd (relative) and the running mean / var after one step: bn_train_fwd_kernel
    sums ceil(n / 8) rows per lane, then the 8 lanes (avf_train.cu:537-556)."""
    emb = emb.double()
    n = emb.shape[0]
    gm = gamma_sum(-(-n // BN_LANES) + BN_LANES)
    rm, rv = p["run_mean"].double().abs(), p["run_var"].double().abs()
    mean_abs = emb.abs().mean(0)
    var_u = emb.var(0, unbiased=True) if n > 1 else torch.zeros_like(rm)
    b = {"mean": gm * mean_abs, "rstd_rel": gm + 8 * EPS32}
    if batch_stats:
        b["run_mean"] = gm * ((1 - momentum) * rm + momentum * mean_abs) + 4 * EPS32 * rm
        b["run_var"] = gm * ((1 - momentum) * rv + momentum * var_u) + 4 * EPS32 * rv
    return b


def two_row_demb_bound(emb, p, emu):
    """Per-column bound of demb for a 2-row batch with batch statistics.  BatchNorm then maps each column to +-d / sqrt(d^2 + eps)
    (d = x - mean), so demb = g rstd (dy - mean(dy) - x-hat mean(dy x-hat)) keeps only ~eps / var of its terms, and what fp32 computes
    of that rests on x - mean, which loses |x| / |d| of its relative precision: 64 ulps of the largest term, times that condition."""
    emb = emb.double()
    d = (emb - emb.mean(0)).abs().min(0).values
    kappa = 1.0 + emb.abs().max(0).values / d.clamp_min(1e-30)
    return 64 * EPS32 * p["gamma"].double().abs() * emu["rstd"] * emu["dy"].abs().max(0).values * kappa


def mutant_applies(kind, n_clips, batch_stats=True, sms=148):
    """Bugs that are no bugs at a size: the BatchNorm backward's batch terms need batch statistics, the 256-entry loop needs more than
    256 entries, the 8-clip sum more than 8 clips, a dropped split-K partial more than one split."""
    if kind in ("running_var_biased", "bn_bwd_no_mean_dy", "bn_bwd_no_xhat_term"):
        return batch_stats
    if kind == "bce_first_256_entries":
        return n_clips * N_AU > BCE_THREADS
    if kind == "dw_last_first_8_clips":
        return n_clips > 8
    if kind == "splitk_drop_last_partial":
        return wgrad_plan(n_clips, sms)[0] > 1
    return True


def seed_of(tag, n_clips):
    return int(np.frombuffer(tag.encode(), dtype=np.uint8).astype(np.int64).sum()) * 101 + n_clips
