"""Tensor-level wrappers over the C ABI (include/avformer_b200.h).

torch is used for device memory, streams and parameter storage only; every arithmetic step of the
hot path happens inside libavformer_b200.so.  All wrappers raise on CPU tensors — there is no fallback.
"""
from __future__ import annotations

import ctypes
from typing import Dict, List, Optional, Sequence, Tuple

import torch

from . import _lib
from ._lib import AVF_BF16, AVF_FP32, LayerWeights, StackShape, check

PRECISIONS = {"fp32": AVF_FP32, "bf16": AVF_BF16}


def _mode(precision) -> int:
    if isinstance(precision, int):
        return precision
    try:
        return PRECISIONS[precision]
    except KeyError:
        raise ValueError(f"precision must be 'bf16' or 'fp32', got {precision!r}") from None


def _io_mode(t: torch.Tensor) -> int:
    if t.dtype == torch.float32:
        return AVF_FP32
    if t.dtype == torch.bfloat16:
        return AVF_BF16
    raise TypeError(f"avformer_b200: unsupported activation dtype {t.dtype} (float32 or bfloat16)")


def _cuda(t: torch.Tensor, name: str) -> torch.Tensor:
    if not t.is_cuda:
        raise RuntimeError(f"avformer_b200: '{name}' is on {t.device}; the B200 path has no CPU fallback")
    # The library launches on the CURRENT device's current stream and never switches devices itself: a tensor that lives on another
    # GPU would be dereferenced by kernels running on the wrong device.  Fail loudly instead (use torch.cuda.device(...) / set_device).
    if t.device.index != torch.cuda.current_device():
        raise RuntimeError(f"avformer_b200: '{name}' is on {t.device} but the current CUDA device is cuda:{torch.cuda.current_device()}; "
                           f"select the tensor's device first (torch.cuda.set_device / with torch.cuda.device(...))")
    return t


def _ptr(t: Optional[torch.Tensor]):
    return None if t is None else ctypes.c_void_p(t.data_ptr())


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def keep_from_mask(mask, n_seq: int, n_tok: int) -> torch.Tensor:
    """The attention ``mask`` of Transformer.forward (models/heads.py:225-232): bool [n_seq, n_tok - 1], True = keep, on the input's
    CUDA device.  Returns the keep rows of the C ABI, bool [n_seq, n_tok] with the first (cls) token always kept; a bool tensor is one
    byte per element, so it is passed to the library as is."""
    shape = tuple(mask.shape) if torch.is_tensor(mask) else type(mask).__name__
    if shape != (n_seq, n_tok - 1):
        raise NotImplementedError(f"attention mask of shape {shape} for {n_seq} sequences of {n_tok} tokens: only the per-sequence keep mask "
                                  f"[{n_seq}, {n_tok - 1}] (bool, True = keep; the first token is always kept) is implemented")
    if mask.dtype != torch.bool:
        raise TypeError(f"avformer_b200: the attention mask must be a bool tensor (True = keep), got {mask.dtype}")
    _cuda(mask, "mask")
    return torch.nn.functional.pad(mask, (1, 0), value=True)


def _keep_ptr(keep: Optional[torch.Tensor], n_seq: int, n_tok: int):
    """Pointer of a keep array [n_seq, n_tok] (bool or uint8, 1 = keep) for the *_masked entry points."""
    if keep.dtype not in (torch.bool, torch.uint8) or tuple(keep.shape) != (n_seq, n_tok) or not keep.is_contiguous():
        raise ValueError(f"avformer_b200: keep must be a contiguous bool / uint8 tensor [{n_seq}, {n_tok}], got {keep.dtype} {tuple(keep.shape)}")
    return _ptr(_cuda(keep, "keep"))


def _f32c(t: torch.Tensor) -> torch.Tensor:
    t = t.detach()
    return t if (t.dtype == torch.float32 and t.is_contiguous()) else t.float().contiguous()


# ------------------------------------------------------------------------------------------------
# workspace: one growable byte buffer per (device, stream)
# ------------------------------------------------------------------------------------------------
_workspaces: Dict[Tuple[int, int], torch.Tensor] = {}


def workspace(nbytes: int, device: torch.device) -> torch.Tensor:
    key = (device.index if device.index is not None else torch.cuda.current_device(), torch.cuda.current_stream().cuda_stream)
    buf = _workspaces.get(key)
    if buf is None or buf.numel() < nbytes:
        buf = torch.empty(max(nbytes, 1 << 20), dtype=torch.uint8, device=device)
        _workspaces[key] = buf
    return buf


# ------------------------------------------------------------------------------------------------
# parameter preparation
# ------------------------------------------------------------------------------------------------
def to_bf16(src: torch.Tensor) -> torch.Tensor:
    """fp32 -> bf16 copy made by the library's own cast kernel."""
    src = _f32c(_cuda(src, "src"))
    dst = torch.empty(src.shape, dtype=torch.bfloat16, device=src.device)
    check(_lib.lib().avf_cast_f32_to_bf16(_ptr(src), _ptr(dst), src.numel(), _stream()), "cast_f32_to_bf16")
    return dst


def to_f32(src: torch.Tensor) -> torch.Tensor:
    src = _cuda(src, "src").contiguous()
    dst = torch.empty(src.shape, dtype=torch.float32, device=src.device)
    check(_lib.lib().avf_cast_bf16_to_f32(_ptr(src), _ptr(dst), src.numel(), _stream()), "cast_bf16_to_f32")
    return dst


def fresh_bf16_image(param: torch.Tensor) -> Optional[torch.Tensor]:
    """The bf16 copy of ``param`` that optim.FusedAdam's update kernel wrote next to the fp32 master (no cast kernel needed), or
    None when there is none or the parameter changed since (version counter)."""
    img = getattr(param, "_avf_bf16", None)
    if img is not None and img[1] == param._version and img[0].device == param.device:
        return img[0]
    return None


def _src_version(t: torch.Tensor) -> tuple:
    """What identifies the VALUE of a parameter for the packed (bf16 / stacked) copies made from it: address, torch's version counter
    (in-place edits, load_state_dict, .to()) and ``_avf_wver``, which optim.FusedAdam bumps on the parameters it updates through raw
    pointers.  Per parameter, so a frozen sub-model's copies stay valid while an optimiser steps the rest of the model."""
    return (t.data_ptr(), t._version, getattr(t, "_avf_wver", 0))


class PackedStack:
    """Device-side weight table of one encoder stack: an array of avf_layer_weights plus the tensors
    that keep the pointers alive.  ``sources`` are the live nn.Parameters; ``stale()`` compares their
    versions so an optimizer step or load_state_dict triggers a re-pack."""

    def __init__(self, layers: Sequence[Dict[str, torch.Tensor]], mode: int):
        self.mode = mode
        self.depth = len(layers)
        self.keep: List[torch.Tensor] = []
        self.sources: List[torch.Tensor] = []
        self.array = (LayerWeights * self.depth)()
        mats = ("w_qkv", "w_out", "w_ff1", "w_ff2")
        for i, lw in enumerate(layers):
            for name, _ in LayerWeights._fields_:
                src = lw[name]
                self.sources.append(src)
                t = _f32c(_cuda(src, name))
                if name in mats and mode == AVF_BF16:
                    t = fresh_bf16_image(src)
                    if t is None:
                        t = to_bf16(_f32c(src))
                self.keep.append(t)
                setattr(self.array[i], name, t.data_ptr())
        self.versions = [_src_version(s) for s in self.sources]
        self.epoch = WEIGHTS_EPOCH

    def stale(self) -> bool:
        return self.epoch != WEIGHTS_EPOCH or any(_src_version(s) != v for s, v in zip(self.sources, self.versions))


# ------------------------------------------------------------------------------------------------
# a1..a5
# ------------------------------------------------------------------------------------------------
def make_shape(n_seq, n_tok, dim, heads, dim_head, mlp_dim, depth) -> StackShape:
    return StackShape(n_seq, n_tok, dim, heads, dim_head, mlp_dim, depth)


def encoder_stack_fwd_(x: torch.Tensor, packed: PackedStack, shape: StackShape, out: Optional[torch.Tensor] = None,
                       ld_out: int = 0, keep: Optional[torch.Tensor] = None) -> torch.Tensor:
    """In-place encoder stack on the fp32 residual stream x [n_seq*n_tok, dim] (row stride = x.stride(0)).
    If ``out`` is given the last layer writes there (row stride ld_out) instead.  ``keep`` [n_seq, n_tok] (bool / uint8, 1 = keep):
    attention mask of every layer (avf_encoder_stack_fwd_masked)."""
    _cuda(x, "x")
    if x.dtype != torch.float32 or x.stride(-1) != 1:
        raise TypeError("encoder_stack_fwd_: x must be a float32 residual stream with unit column stride")
    L = _lib.lib()
    need = L.avf_encoder_workspace_bytes(ctypes.byref(shape), packed.mode)
    ws = workspace(need, x.device)
    if keep is None:
        check(L.avf_encoder_stack_fwd(packed.mode, ctypes.byref(shape), packed.array, _ptr(x), x.stride(0), _ptr(out), ld_out,
                                      _ptr(ws), ws.numel(), _stream()), "encoder_stack_fwd")
    else:
        check(L.avf_encoder_stack_fwd_masked(packed.mode, ctypes.byref(shape), packed.array, _keep_ptr(keep, shape.n_seq, shape.n_tok), _ptr(x),
                                             x.stride(0), _ptr(out), ld_out, _ptr(ws), ws.numel(), _stream()), "encoder_stack_fwd_masked")
    return x if out is None else out


def token_stack_fwd_(x: torch.Tensor, packed: PackedStack, shape: StackShape, pos: Optional[torch.Tensor] = None,
                     out: Optional[torch.Tensor] = None, ld_out: int = 0, w_last: Optional[torch.Tensor] = None, want_decisions: bool = False):
    """encoder_stack_fwd_ of a token head: + pos [n_tok, dim] first (if given); with w_last [12, dim] (12 tokens per sequence) the
    AU logits of the result follow and [n_seq, 21] logits (+ [n_seq, 12] int32 decisions) are returned, else the tokens.  In bf16
    mode a fused-kernel stack is one launch.  x is scratch whenever out or w_last is given."""
    _cuda(x, "x")
    if x.dtype != torch.float32 or x.stride(-1) != 1:
        raise TypeError("token_stack_fwd_: x must be a float32 residual stream with unit column stride")
    L = _lib.lib()
    ws = workspace(L.avf_encoder_workspace_bytes(ctypes.byref(shape), packed.mode), x.device)
    out21 = dec = None
    if w_last is not None:
        out21 = torch.empty((shape.n_seq, 21), dtype=torch.float32, device=x.device)
        dec = torch.empty((shape.n_seq, 12), dtype=torch.int32, device=x.device) if want_decisions else None
    check(L.avf_token_stack_fwd(packed.mode, ctypes.byref(shape), packed.array, _ptr(x), x.stride(0), _ptr(None if pos is None else _f32c(pos)),
                                _ptr(out), ld_out, _ptr(None if w_last is None else _f32c(w_last)), _ptr(out21), _ptr(dec), _ptr(ws), ws.numel(),
                                _stream()), "token_stack_fwd")
    if w_last is not None:
        return (out21, dec) if want_decisions else out21
    return x if out is None else out


def layernorm_fwd(x: torch.Tensor, gamma: torch.Tensor, beta: torch.Tensor, precision="bf16") -> torch.Tensor:
    x = _f32c(_cuda(x, "x"))
    rows, dim = x.numel() // x.shape[-1], x.shape[-1]
    mode = _mode(precision)
    y = torch.empty(x.shape, dtype=torch.bfloat16 if mode == AVF_BF16 else torch.float32, device=x.device)
    check(_lib.lib().avf_layernorm_fwd(mode, _ptr(x), dim, _ptr(_f32c(gamma)), _ptr(_f32c(beta)), _ptr(y), rows, dim, _stream()), "layernorm_fwd")
    return y


def linear_fwd(a: torch.Tensor, w: torch.Tensor, bias: Optional[torch.Tensor] = None, residual: Optional[torch.Tensor] = None,
               gelu: bool = False, out_dtype: torch.dtype = torch.float32, precision="bf16") -> torch.Tensor:
    """epi(a @ w.T): a [M,K], w [N,K] (both bf16 for precision 'bf16', both fp32 for 'fp32')."""
    mode = _mode(precision)
    want = torch.bfloat16 if mode == AVF_BF16 else torch.float32
    _cuda(a, "a")
    if a.dtype != want or w.dtype != want:
        raise TypeError(f"linear_fwd({precision}): operands must be {want}, got {a.dtype} / {w.dtype}")
    a, w = a.contiguous(), w.contiguous()
    m, k = a.shape
    n = w.shape[0]
    c = torch.empty((m, n), dtype=out_dtype, device=a.device)
    flags = (1 if bias is not None else 0) | (2 if gelu else 0) | (4 if residual is not None else 0)
    if residual is not None:
        residual = _f32c(residual)
    if bias is not None:
        bias = _f32c(bias)
    check(_lib.lib().avf_linear_fwd(mode, _ptr(a), k, _ptr(w), _ptr(bias), _ptr(residual), n, _ptr(c), n, _io_mode(c), m, n, k, flags,
                                    _stream()), "linear_fwd")
    return c


def attention_fwd(qkv: torch.Tensor, n_seq: int, n_tok: int, heads: int, dim_head: int, keep: Optional[torch.Tensor] = None) -> torch.Tensor:
    """softmax(q k^T / sqrt(dh)) v per (sequence, head); ``keep`` [n_seq, n_tok] (bool / uint8, 1 = keep) masks the scores."""
    qkv = _cuda(qkv, "qkv").contiguous()
    out = torch.empty((n_seq * n_tok, heads * dim_head), dtype=qkv.dtype, device=qkv.device)
    if keep is None:
        check(_lib.lib().avf_attention_fwd(_io_mode(qkv), _ptr(qkv), _ptr(out), n_seq, n_tok, heads, dim_head, _stream()), "attention_fwd")
    else:
        check(_lib.lib().avf_attention_fwd_masked(_io_mode(qkv), _ptr(qkv), _ptr(out), n_seq, n_tok, heads, dim_head, _keep_ptr(keep, n_seq, n_tok),
                                                  _stream()), "attention_fwd_masked")
    return out


# ------------------------------------------------------------------------------------------------
# a6 / a7 / a8 / a9 / a11 / a12
# ------------------------------------------------------------------------------------------------
def sformer_fwd(fmap: torch.Tensor, pos: torch.Tensor, packed: PackedStack, heads: int, dim_head: int, mlp_dim: int,
                out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """models/vformer.py:245-259 on a stage-3 map [F, C, H, W] (fp32 or bf16, NCHW-contiguous)."""
    fmap = _cuda(fmap, "fmap").contiguous()
    F_, C, H, W = fmap.shape
    shape = make_shape(F_, H * W, C, heads, dim_head, mlp_dim, packed.depth)
    L = _lib.lib()
    need = L.avf_sformer_workspace_bytes(ctypes.byref(shape), packed.mode)
    ws = workspace(need, fmap.device)
    if out is None:
        out = torch.empty_like(fmap)
    elif out.shape != fmap.shape or out.dtype != fmap.dtype or not out.is_contiguous():
        raise ValueError("sformer_fwd: `out` must be a contiguous tensor with the shape and dtype of the input map")
    check(L.avf_sformer_fwd(packed.mode, _io_mode(fmap), ctypes.byref(shape), packed.array, _ptr(_f32c(pos)), _ptr(fmap), _ptr(out),
                            _ptr(ws), ws.numel(), _stream()), "sformer_fwd")
    return out


def tformer_embed(frames: torch.Tensor, cls_token: torch.Tensor, pos: torch.Tensor, n_frames: int) -> torch.Tensor:
    frames = _cuda(frames, "frames").contiguous()
    dim = frames.shape[-1]
    n_clips = frames.numel() // (n_frames * dim)
    x = torch.empty((n_clips * (n_frames + 1), dim), dtype=torch.float32, device=frames.device)
    check(_lib.lib().avf_tformer_embed(_io_mode(frames), _ptr(frames), _ptr(_f32c(cls_token)), _ptr(_f32c(pos)), _ptr(x), n_clips, n_frames,
                                       dim, _stream()), "tformer_embed")
    return x


def tformer_fwd(frames: torch.Tensor, cls_token: torch.Tensor, pos: torch.Tensor, packed: PackedStack, shape: StackShape,
                keep: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Inference TFormer in one call: frames [n_clips*T, dim] -> cls features [n_clips, dim] fp32 (last layer on the cls rows only).
    ``keep`` [n_clips, T+1] (bool / uint8, 1 = keep; column 0 is the cls token): attention mask of every layer."""
    frames = _cuda(frames, "frames").contiguous()
    cls = torch.empty((shape.n_seq, shape.dim), dtype=torch.float32, device=frames.device)
    L = _lib.lib()
    ws = workspace(L.avf_tformer_workspace_bytes(ctypes.byref(shape), packed.mode), frames.device)
    if keep is None:
        check(L.avf_tformer_fwd(packed.mode, _io_mode(frames), ctypes.byref(shape), packed.array, _ptr(frames), _ptr(_f32c(cls_token)), _ptr(_f32c(pos)),
                                _ptr(cls), _ptr(ws), ws.numel(), _stream()), "tformer_fwd")
    else:
        check(L.avf_tformer_fwd_masked(packed.mode, _io_mode(frames), ctypes.byref(shape), packed.array, _keep_ptr(keep, shape.n_seq, shape.n_tok),
                                       _ptr(frames), _ptr(_f32c(cls_token)), _ptr(_f32c(pos)), _ptr(cls), _ptr(ws), ws.numel(), _stream()),
              "tformer_fwd_masked")
    return cls


def tformer_fwd_indexed(bank: torch.Tensor, index: torch.Tensor, cls_token: torch.Tensor, pos: torch.Tensor, packed: PackedStack,
                        shape: StackShape) -> torch.Tensor:
    """Inference TFormer on clips gathered from a frame bank in one call (avf_tformer_fwd_indexed): bank [n_bank, dim] fp32 / bf16,
    index [n_clips, T] int32 contiguous on the bank's device, an entry outside [0, n_bank) = a missing frame, masked out of every
    layer -> cls features [n_clips, dim] fp32."""
    bank = _cuda(bank, "bank").contiguous()
    if index.dtype != torch.int32 or not index.is_contiguous() or tuple(index.shape) != (shape.n_seq, shape.n_tok - 1):
        raise ValueError(f"tformer_fwd_indexed: index must be a contiguous int32 tensor [{shape.n_seq}, {shape.n_tok - 1}], "
                         f"got {index.dtype} {tuple(index.shape)}")
    _cuda(index, "index")
    cls = torch.empty((shape.n_seq, shape.dim), dtype=torch.float32, device=bank.device)
    L = _lib.lib()
    ws = workspace(L.avf_tformer_indexed_workspace_bytes(ctypes.byref(shape), packed.mode), bank.device)
    check(L.avf_tformer_fwd_indexed(packed.mode, _io_mode(bank), ctypes.byref(shape), packed.array, _ptr(bank), bank.shape[0], _ptr(index),
                                    _ptr(_f32c(cls_token)), _ptr(_f32c(pos)), _ptr(cls), _ptr(ws), ws.numel(), _stream()), "tformer_fwd_indexed")
    return cls


def tformer_cls_extract(x: torch.Tensor, n_clips: int, n_tok: int) -> torch.Tensor:
    dim = x.shape[-1]
    cls = torch.empty((n_clips, dim), dtype=torch.float32, device=x.device)
    check(_lib.lib().avf_tformer_cls_extract(_ptr(x), _ptr(cls), n_clips, n_tok, dim, _stream()), "tformer_cls_extract")
    return cls


def au_former_front(emb: torch.Tensor, ld_emb: int, n_clips: int, bn: Sequence[torch.Tensor], w_cat: torch.Tensor, b_cat: torch.Tensor,
                    pos: Optional[torch.Tensor], mode: int) -> torch.Tensor:
    """BN(eval) + 12 stacked Linear(512,128) + pos -> fp32 tokens [n_clips*12, 128] (models/heads.py:293-323); pos None: no add."""
    _cuda(emb, "emb")
    in_dim, emb_dim = w_cat.shape[1], w_cat.shape[0] // 12
    x = torch.empty((n_clips * 12, emb_dim), dtype=torch.float32, device=emb.device)
    ws = workspace(n_clips * in_dim * 4 + 256, emb.device)
    g, b, mu, var = (_f32c(t) for t in bn)
    check(_lib.lib().avf_au_former_front_fwd(mode, _ptr(emb), ld_emb, _ptr(g), _ptr(b), _ptr(mu), _ptr(var), _ptr(w_cat), _ptr(b_cat),
                                             _ptr(None if pos is None else _f32c(pos)), _ptr(x), n_clips, in_dim, emb_dim, _ptr(ws), ws.numel(), _stream()),
          "au_former_front_fwd")
    return x


def token_front(emb: torch.Tensor, ld_emb: int, n_clips: int, n_tok: int, bn: Sequence[torch.Tensor], w_cat: torch.Tensor, b_cat: torch.Tensor,
                pos: Optional[torch.Tensor], mode: int) -> torch.Tensor:
    """au_former_front for any token count: BN(eval) + n_tok stacked Linear + pos (if given) -> fp32 tokens [n_clips*n_tok, emb_dim]
    (n_tok = 2: VA_former, models/heads.py:354-364)."""
    _cuda(emb, "emb")
    in_dim, emb_dim = w_cat.shape[1], w_cat.shape[0] // n_tok
    x = torch.empty((n_clips * n_tok, emb_dim), dtype=torch.float32, device=emb.device)
    ws = workspace(n_clips * in_dim * 4 + 256, emb.device)
    g, b, mu, var = (_f32c(t) for t in bn)
    check(_lib.lib().avf_token_front_fwd(mode, _ptr(emb), ld_emb, _ptr(g), _ptr(b), _ptr(mu), _ptr(var), _ptr(w_cat), _ptr(b_cat),
                                         _ptr(None if pos is None else _f32c(pos)), _ptr(x), n_clips, in_dim, emb_dim, n_tok, _ptr(ws), ws.numel(), _stream()),
          "token_front_fwd")
    return x


def au_logits(x: torch.Tensor, w_last: torch.Tensor, n_clips: int, want_decisions: bool = False):
    """Tail of the fusion head: [B,21] zero-padded output (+ int32 decisions)."""
    _cuda(x, "x")
    out = torch.empty((n_clips, 21), dtype=torch.float32, device=x.device)
    dec = torch.empty((n_clips, 12), dtype=torch.int32, device=x.device) if want_decisions else None
    check(_lib.lib().avf_au_logits_fwd(_ptr(x), x.stride(0), _ptr(w_last), _ptr(out), _ptr(dec), n_clips, x.shape[-1], _stream()), "au_logits_fwd")
    return (out, dec) if want_decisions else out


def au_bce_loss(y_pred: torch.Tensor, y_true: torch.Tensor, pos_weight: torch.Tensor, want_grad: bool = False):
    """AULoss (models/loss.py:75-103) on logits y_pred[:, :12]; returns (loss scalar tensor, n_valid, dlogits|None)."""
    _cuda(y_pred, "y_pred")
    if y_pred.dtype != torch.float32 or y_pred.stride(-1) != 1:
        y_pred = y_pred.float().contiguous()
    y_true = _f32c(_cuda(y_true, "y_true"))
    n = y_pred.shape[0]
    res = torch.empty(2, dtype=torch.float32, device=y_pred.device)
    grad = torch.empty((n, 12), dtype=torch.float32, device=y_pred.device) if want_grad else None
    check(_lib.lib().avf_au_bce_loss(_ptr(y_pred), y_pred.stride(0), _ptr(y_true), _ptr(_f32c(pos_weight)), _ptr(res), _ptr(grad), n, _stream()),
          "au_bce_loss")
    return res[0], res[1], grad


def add_row_periodic_(x: torch.Tensor, pos: torch.Tensor, period: int) -> torch.Tensor:
    check(_lib.lib().avf_add_row_periodic(_ptr(x), x.stride(0), _ptr(_f32c(pos)), x.shape[0], x.shape[1], period, _stream()), "add_row_periodic")
    return x


def device_info() -> Dict[str, int]:
    a, b, c = _lib._i32(), _lib._i32(), _lib._i32()
    check(_lib.lib().avf_device_info(ctypes.byref(a), ctypes.byref(b), ctypes.byref(c)), "device_info")
    return {"sm_count": a.value, "cc": b.value, "has_tcgen05": c.value}


def set_fused_enabled(enabled: bool) -> bool:
    """Toggle the one-kernel-per-stack tcgen05 path (dim 256 / 128, 8x32 stacks); returns the previous setting."""
    return bool(_lib.lib().avf_set_fused_enabled(1 if enabled else 0))


def encoder_fused_supported(shape: StackShape, precision="bf16") -> bool:
    return bool(_lib.lib().avf_encoder_fused_supported(ctypes.byref(shape), _mode(precision)))


# ------------------------------------------------------------------------------------------------
# training: tape forward, backward, optimiser (include/avformer_b200.h, section "training")
# ------------------------------------------------------------------------------------------------
WEIGHTS_EPOCH = 0          # global "every packed copy is stale" switch (bump_weights_epoch); FusedAdam uses the per-parameter _avf_wver instead


def bump_weights_epoch() -> None:
    """Tell every packed (bf16 / stacked) weight copy that the fp32 master parameters changed underneath it."""
    global WEIGHTS_EPOCH
    WEIGHTS_EPOCH += 1


def _act_dtype(mode: int) -> torch.dtype:
    return torch.bfloat16 if mode == AVF_BF16 else torch.float32


def gemm(a: torch.Tensor, b: torch.Tensor, trans_a: bool = False, trans_b: bool = False, m: Optional[int] = None, n: Optional[int] = None,
         k: Optional[int] = None, bias=None, residual=None, aux=None, flags: int = 0, out_dtype=torch.float32, precision="bf16") -> torch.Tensor:
    """C[M,N] = epi(op(A) op(B)) — see avf_gemm.  a / b are 2-D contiguous; trans_* say the reduction index is the ROW index."""
    mode = _mode(precision)
    _cuda(a, "a")
    a, b = a.contiguous(), b.contiguous()
    m = m if m is not None else (a.shape[1] if trans_a else a.shape[0])
    k = k if k is not None else (a.shape[0] if trans_a else a.shape[1])
    n = n if n is not None else (b.shape[1] if trans_b else b.shape[0])
    c = torch.empty((m, n), dtype=out_dtype, device=a.device)
    L = _lib.lib()
    need = L.avf_gemm_workspace_bytes(mode, int(trans_a), int(trans_b), m, n, k)
    ws = workspace(max(need, 256), a.device)
    check(L.avf_gemm(mode, int(trans_a), int(trans_b), _ptr(a), a.stride(0), _ptr(b), b.stride(0), _ptr(bias), _ptr(residual),
                     residual.stride(0) if residual is not None else 0, _ptr(aux), aux.stride(0) if aux is not None else 0, _ptr(c), n,
                     _io_mode(c), m, n, k, flags, _ptr(ws), ws.numel(), _stream()), "gemm")
    return c


def colsum(x: torch.Tensor) -> torch.Tensor:
    """Column sums of a 2-D fp32 / bf16 matrix (unit column stride) -> fp32 [cols]."""
    _cuda(x, "x")
    rows, cols = x.shape
    out = torch.empty(cols, dtype=torch.float32, device=x.device)
    L = _lib.lib()
    ws = workspace(L.avf_colsum_workspace_bytes(rows, cols), x.device)
    check(L.avf_colsum(_io_mode(x), _ptr(x), x.stride(0), rows, cols, _ptr(out), _ptr(ws), ws.numel(), _stream()), "colsum")
    return out


def layernorm_bwd_(x: torch.Tensor, gamma: torch.Tensor, dy_norm: torch.Tensor, dres: torch.Tensor, want_bf16: bool = False):
    """In place on dres [rows, dim] (fp32): dres += LN'(dy_norm).  Returns (dres, dx_bf16|None, dgamma, dbeta, dbias)."""
    rows, dim = dres.shape
    dev = dres.device
    dg, db, dbias = (torch.empty(dim, dtype=torch.float32, device=dev) for _ in range(3))
    xb = torch.empty((rows, dim), dtype=torch.bfloat16, device=dev) if want_bf16 else None
    L = _lib.lib()
    ws = workspace(L.avf_layernorm_bwd_workspace_bytes(rows, dim), dev)
    check(L.avf_layernorm_bwd(_ptr(x), x.stride(0), _ptr(_f32c(gamma)), _ptr(dy_norm), _ptr(dres), dres.stride(0), _ptr(xb), _ptr(dg), _ptr(db),
                              _ptr(dbias), rows, dim, _ptr(ws), ws.numel(), _stream()), "layernorm_bwd")
    return dres, xb, dg, db, dbias


def attention_bwd(qkv: torch.Tensor, dout: torch.Tensor, n_seq: int, n_tok: int, heads: int, dim_head: int,
                  keep: Optional[torch.Tensor] = None) -> torch.Tensor:
    """dqkv of attention_fwd (softmax recomputed); ``keep`` must be the mask of the forward."""
    qkv, dout = _cuda(qkv, "qkv").contiguous(), dout.contiguous()
    dqkv = torch.empty_like(qkv)
    if keep is None:
        check(_lib.lib().avf_attention_bwd(_io_mode(qkv), _ptr(qkv), _ptr(dout), _ptr(dqkv), n_seq, n_tok, heads, dim_head, _stream()), "attention_bwd")
    else:
        check(_lib.lib().avf_attention_bwd_masked(_io_mode(qkv), _ptr(qkv), _ptr(dout), _ptr(dqkv), n_seq, n_tok, heads, dim_head,
                                                  _keep_ptr(keep, n_seq, n_tok), _stream()), "attention_bwd_masked")
    return dqkv


def encoder_stack_fwd_train(x: torch.Tensor, packed: PackedStack, shape: StackShape, dropout_p: float = 0.0, dropout_seed: int = 0,
                            dropout_salt: Optional[torch.Tensor] = None, keep: Optional[torch.Tensor] = None):
    """Forward of a whole stack that keeps the activations the backward needs.  x [n_seq*n_tok, dim] fp32 is left
    untouched; returns (y, tape).  dropout_p > 0 applies the reference's three dropout sites per layer with masks derived from
    dropout_seed (give the same pair to encoder_stack_bwd_).  ``keep`` [n_seq, n_tok] (bool / uint8, 1 = keep): attention mask of
    every layer; give the same tensor to encoder_stack_bwd_."""
    _cuda(x, "x")
    if x.dtype != torch.float32 or x.stride(-1) != 1:
        raise TypeError("encoder_stack_fwd_train: x must be a float32 residual stream with unit column stride")
    L = _lib.lib()
    tape = torch.empty(L.avf_encoder_tape_bytes(ctypes.byref(shape), packed.mode), dtype=torch.uint8, device=x.device)
    y = torch.empty((x.shape[0], shape.dim), dtype=torch.float32, device=x.device)
    if keep is None:
        check(L.avf_encoder_stack_fwd_train(packed.mode, ctypes.byref(shape), packed.array, _ptr(x), x.stride(0), _ptr(y), shape.dim, _ptr(tape),
                                            tape.numel(), float(dropout_p), int(dropout_seed), _ptr(dropout_salt), _stream()), "encoder_stack_fwd_train")
    else:
        check(L.avf_encoder_stack_fwd_train_masked(packed.mode, ctypes.byref(shape), packed.array, _keep_ptr(keep, shape.n_seq, shape.n_tok), _ptr(x),
                                                   x.stride(0), _ptr(y), shape.dim, _ptr(tape), tape.numel(), float(dropout_p), int(dropout_seed),
                                                   _ptr(dropout_salt), _stream()), "encoder_stack_fwd_train_masked")
    return y, tape


def encoder_stack_bwd_(dx: torch.Tensor, packed: PackedStack, shape: StackShape, tape: torch.Tensor, want: Sequence[bool],
                       dropout_p: float = 0.0, dropout_seed: int = 0, dropout_salt: Optional[torch.Tensor] = None,
                       into: Optional[Sequence[Optional[torch.Tensor]]] = None, keep: Optional[torch.Tensor] = None):
    """dx [rows, dim] fp32 dense: dL/dy on entry, dL/dx on return.  ``want`` has 11*depth flags in avf_layer_weights
    order; returns the matching list of fp32 gradient tensors (None where not wanted).

    ``into`` (optional, same order): existing fp32 contiguous gradient buffers — typically the ``p.grad`` views of the
    optimiser's flat bucket.  When every wanted gradient has one, the kernels ACCUMULATE straight into them and the returned
    list holds None throughout (nothing left for autograd to add).  ``keep``: the attention mask of the forward, if it had one."""
    from ._lib import LayerGrads
    names = [n for n, _ in LayerWeights._fields_]
    n_par = packed.depth * len(names)
    direct = into is not None and all((not want[i]) or (into[i] is not None and into[i].dtype == torch.float32 and into[i].is_contiguous()
                                                         and into[i].is_cuda) for i in range(n_par))
    grads: List[Optional[torch.Tensor]] = []
    arr = (LayerGrads * packed.depth)()
    for l in range(packed.depth):
        for j, name in enumerate(names):
            i = l * len(names) + j
            g = None
            if want[i]:
                g = into[i] if direct else torch.empty(packed.sources[i].shape, dtype=torch.float32, device=dx.device)
            grads.append(None if direct else g)
            setattr(arr[l], name, g.data_ptr() if g is not None else None)
    L = _lib.lib()
    ws = workspace(L.avf_encoder_bwd_workspace_bytes(ctypes.byref(shape), packed.mode), dx.device)
    if keep is None:
        check(L.avf_encoder_stack_bwd(packed.mode, ctypes.byref(shape), packed.array, _ptr(tape), tape.numel(), _ptr(dx), dx.stride(0), arr,
                                      1 if direct else 0, _ptr(ws), ws.numel(), float(dropout_p), int(dropout_seed), _ptr(dropout_salt), _stream()),
              "encoder_stack_bwd")
    else:
        check(L.avf_encoder_stack_bwd_masked(packed.mode, ctypes.byref(shape), packed.array, _keep_ptr(keep, shape.n_seq, shape.n_tok), _ptr(tape),
                                             tape.numel(), _ptr(dx), dx.stride(0), arr, 1 if direct else 0, _ptr(ws), ws.numel(), float(dropout_p),
                                             int(dropout_seed), _ptr(dropout_salt), _stream()), "encoder_stack_bwd_masked")
    return dx, grads


def sformer_tokens_pack(fmap: torch.Tensor, pos: Optional[torch.Tensor]) -> torch.Tensor:
    """[F,C,H,W] -> fp32 tokens [F*H*W, C] (+ pos [H*W, C]); pos=None is the plain transpose."""
    fmap = _cuda(fmap, "fmap").contiguous()
    F_, C, H, W = fmap.shape
    x = torch.empty((F_ * H * W, C), dtype=torch.float32, device=fmap.device)
    check(_lib.lib().avf_sformer_tokens_pack(_io_mode(fmap), _ptr(fmap), _ptr(_f32c(pos)) if pos is not None else None, _ptr(x), F_, C, H * W,
                                             _stream()), "sformer_tokens_pack")
    return x


def sformer_tokens_unpack(x: torch.Tensor, shape4, dtype: torch.dtype) -> torch.Tensor:
    F_, C, H, W = shape4
    fmap = torch.empty((F_, C, H, W), dtype=dtype, device=x.device)
    check(_lib.lib().avf_sformer_tokens_unpack(_io_mode(fmap), _ptr(x), _ptr(fmap), F_, C, H * W, _stream()), "sformer_tokens_unpack")
    return fmap


def au_former_front_train(emb: torch.Tensor, n_clips: int, bn_w, bn_b, run_mean, run_var, batch_stats: bool, momentum: float,
                          w_cat: torch.Tensor, b_cat: torch.Tensor, pos: torch.Tensor, mode: int):
    """BN (batch or running statistics) + 12 stacked projections + pos, keeping what the backward needs.
    emb [n_clips, in_dim] fp32 with unit column stride (any row stride).  Returns (tokens [n_clips*12, emb_dim], tape)."""
    _cuda(emb, "emb")
    in_dim, emb_dim = w_cat.shape[1], w_cat.shape[0] // 12
    L = _lib.lib()
    tape = torch.empty(L.avf_au_former_front_tape_bytes(mode, n_clips, in_dim), dtype=torch.uint8, device=emb.device)
    x = torch.empty((n_clips * 12, emb_dim), dtype=torch.float32, device=emb.device)
    check(L.avf_au_former_front_fwd_train(mode, _ptr(emb), emb.stride(0), _ptr(_f32c(bn_w)), _ptr(_f32c(bn_b)), _ptr(run_mean), _ptr(run_var),
                                          int(batch_stats), float(momentum), _ptr(w_cat), _ptr(b_cat), _ptr(_f32c(pos)), _ptr(x), n_clips, in_dim,
                                          emb_dim, _ptr(tape), tape.numel(), _stream()), "au_former_front_fwd_train")
    return x, tape


def au_former_front_bwd(emb: torch.Tensor, n_clips: int, bn_w, run_mean, run_var, batch_stats: bool, w_cat: torch.Tensor, tape: torch.Tensor,
                        dx: torch.Tensor, mode: int, want_emb=True, want_bn=True, want_w=True):
    """-> (demb [n_clips,in_dim] | None, dbn_gamma, dbn_beta | None, dw_cat [12*emb,in] | None, db_cat [12*emb] (== dpos))."""
    in_dim, emb_dim = w_cat.shape[1], w_cat.shape[0] // 12
    dev = dx.device
    dx = dx.contiguous()
    demb = torch.empty((n_clips, in_dim), dtype=torch.float32, device=dev) if want_emb else None
    dg = torch.empty(in_dim, dtype=torch.float32, device=dev) if want_bn else None
    db = torch.empty(in_dim, dtype=torch.float32, device=dev) if want_bn else None
    dw = torch.empty((12 * emb_dim, in_dim), dtype=torch.float32, device=dev) if want_w else None
    dbc = torch.empty(12 * emb_dim, dtype=torch.float32, device=dev)
    L = _lib.lib()
    ws = workspace(L.avf_au_former_front_bwd_workspace_bytes(mode, n_clips, in_dim, emb_dim), dev)
    check(L.avf_au_former_front_bwd(mode, _ptr(emb), emb.stride(0), _ptr(_f32c(bn_w)), _ptr(run_mean), _ptr(run_var), int(batch_stats), _ptr(w_cat),
                                    _ptr(tape), tape.numel(), _ptr(dx), _ptr(demb), in_dim, _ptr(dg), _ptr(db), _ptr(dw), _ptr(dbc), n_clips, in_dim,
                                    emb_dim, _ptr(ws), ws.numel(), _stream()), "au_former_front_bwd")
    return demb, dg, db, dw, dbc


def au_logits_bwd(dlogits: torch.Tensor, x: torch.Tensor, w_last: torch.Tensor, n_clips: int, want_dx=True, want_dw=True):
    """dlogits [n_clips, >=12] fp32 (row stride free) -> (dx [n_clips*12, dim] | None, dw_last [12, dim] | None)."""
    dim = w_last.shape[1]
    dx = torch.empty((n_clips * 12, dim), dtype=torch.float32, device=x.device) if want_dx else None
    dw = torch.empty((12, dim), dtype=torch.float32, device=x.device) if want_dw else None
    check(_lib.lib().avf_au_logits_bwd(_ptr(dlogits), dlogits.stride(0), _ptr(x), x.stride(0), _ptr(w_last), _ptr(dx), dim, _ptr(dw), n_clips, dim,
                                       _stream()), "au_logits_bwd")
    return dx, dw


def adam_step_(p: torch.Tensor, g: torch.Tensor, m: torch.Tensor, v: torch.Tensor, step: int, lr: float, beta1: float, beta2: float, eps: float,
               weight_decay: float, decoupled: bool = False, grad_scale: float = 1.0, shadow: Optional[torch.Tensor] = None) -> None:
    """One fused Adam / AdamW step over flat fp32 buckets (in place on p, m, v)."""
    _cuda(p, "params")
    check(_lib.lib().avf_adam_step(_ptr(p), _ptr(g), _ptr(m), _ptr(v), _ptr(shadow), p.numel(), lr, beta1, beta2, eps, weight_decay, step,
                                   int(decoupled), grad_scale, _stream()), "adam_step")


def dropout_mask(dropout_p: float, dropout_seed: int, layer: int, site: int, rows: int, cols: int, device,
                 dropout_salt: Optional[torch.Tensor] = None) -> torch.Tensor:
    """The scaled keep-mask (0 or 1/(1-p)) the kernels apply at one dropout site (0 to_out, 1 GELU, 2 net.3) of one layer."""
    out = torch.empty((rows, cols), dtype=torch.float32, device=device)
    check(_lib.lib().avf_dropout_mask(float(dropout_p), int(dropout_seed), _ptr(dropout_salt), layer, site, rows, cols, _ptr(out), _stream()),
          "dropout_mask")
    return out
