"""Loader / builder for libavformer_b200.so (the C ABI declared in include/avformer_b200.h).

The library is built in-tree with nvcc for sm_100a only.  There is no fallback of any kind: if the
library cannot be built or loaded, or there is no CUDA device, every compute call raises.
"""
from __future__ import annotations

import ctypes
import glob
import os
import shutil
import subprocess
import threading

_PKG = os.path.dirname(os.path.abspath(__file__))
_ROOT = os.path.dirname(_PKG)
_CSRC = os.path.join(_PKG, "csrc")
LIB_PATH = os.path.join(_PKG, "libavformer_b200.so")
# Developer A/B runs: AVF_LIB_OVERRIDE=<path of an alternative build of the same sources> is loaded as is (never built here).
_OVERRIDE = os.environ.get("AVF_LIB_OVERRIDE", "")

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
    "-Xcompiler", "-fPIC", "-shared", "-cudart", "static", "-t", "0",
]

AVF_FP32, AVF_BF16 = 0, 1
EPI_BIAS, EPI_GELU, EPI_RESIDUAL, EPI_DGELU, EPI_SAVE_PRE = 1, 2, 4, 8, 16

_c_p = ctypes.c_void_p
_i32 = ctypes.c_int32
_sz = ctypes.c_size_t


class LayerWeights(ctypes.Structure):
    """struct avf_layer_weights (include/avformer_b200.h)."""
    _fields_ = [(n, _c_p) for n in ("ln1_gamma", "ln1_beta", "w_qkv", "w_out", "b_out", "ln2_gamma", "ln2_beta",
                                    "w_ff1", "b_ff1", "w_ff2", "b_ff2")]


class LayerGrads(ctypes.Structure):
    """struct avf_layer_grads: fp32 gradient destinations, NULL = not wanted."""
    _fields_ = LayerWeights._fields_


class StackShape(ctypes.Structure):
    """struct avf_stack_shape."""
    _fields_ = [(n, _i32) for n in ("n_seq", "n_tok", "dim", "heads", "dim_head", "mlp_dim", "depth")]


# name -> (restype, argtypes); mirrors include/avformer_b200.h one to one
SIGNATURES = {
    "avf_abi_version": (ctypes.c_int, []),
    "avf_last_error": (ctypes.c_char_p, []),
    "avf_launch_count": (ctypes.c_uint64, []),
    "avf_device_info": (ctypes.c_int, [ctypes.POINTER(_i32)] * 3),
    "avf_set_fused_enabled": (ctypes.c_int, [ctypes.c_int]),
    "avf_encoder_fused_supported": (ctypes.c_int, [ctypes.POINTER(StackShape), ctypes.c_int]),
    "avf_debug_fused_prof": (ctypes.c_int, [ctypes.POINTER(ctypes.c_uint64), ctypes.c_int]),
    "avf_encoder_workspace_bytes": (_sz, [ctypes.POINTER(StackShape), ctypes.c_int]),
    "avf_encoder_stack_fwd": (ctypes.c_int, [ctypes.c_int, ctypes.POINTER(StackShape), ctypes.POINTER(LayerWeights), _c_p, _i32,
                                             _c_p, _i32, _c_p, _sz, _c_p]),
    "avf_token_stack_fwd": (ctypes.c_int, [ctypes.c_int, ctypes.POINTER(StackShape), ctypes.POINTER(LayerWeights), _c_p, _i32, _c_p,
                                           _c_p, _i32, _c_p, _c_p, _c_p, _c_p, _sz, _c_p]),
    "avf_layernorm_fwd": (ctypes.c_int, [ctypes.c_int, _c_p, _i32, _c_p, _c_p, _c_p, _i32, _i32, _c_p]),
    "avf_linear_fwd": (ctypes.c_int, [ctypes.c_int, _c_p, _i32, _c_p, _c_p, _c_p, _i32, _c_p, _i32, ctypes.c_int, _i32, _i32, _i32,
                                      ctypes.c_int, _c_p]),
    "avf_attention_fwd": (ctypes.c_int, [ctypes.c_int, _c_p, _c_p, _i32, _i32, _i32, _i32, _c_p]),
    "avf_sformer_tokens_pack": (ctypes.c_int, [ctypes.c_int, _c_p, _c_p, _c_p, _i32, _i32, _i32, _c_p]),
    "avf_sformer_tokens_unpack": (ctypes.c_int, [ctypes.c_int, _c_p, _c_p, _i32, _i32, _i32, _c_p]),
    "avf_sformer_workspace_bytes": (_sz, [ctypes.POINTER(StackShape), ctypes.c_int]),
    "avf_sformer_fwd": (ctypes.c_int, [ctypes.c_int, ctypes.c_int, ctypes.POINTER(StackShape), ctypes.POINTER(LayerWeights), _c_p, _c_p,
                                       _c_p, _c_p, _sz, _c_p]),
    "avf_tformer_embed": (ctypes.c_int, [ctypes.c_int, _c_p, _c_p, _c_p, _c_p, _i32, _i32, _i32, _c_p]),
    "avf_tformer_workspace_bytes": (_sz, [ctypes.POINTER(StackShape), ctypes.c_int]),
    "avf_tformer_fwd": (ctypes.c_int, [ctypes.c_int, ctypes.c_int, ctypes.POINTER(StackShape), ctypes.POINTER(LayerWeights), _c_p, _c_p, _c_p, _c_p,
                                       _c_p, _sz, _c_p]),
    "avf_tformer_cls_extract": (ctypes.c_int, [_c_p, _c_p, _i32, _i32, _i32, _c_p]),
    "avf_au_former_front_fwd": (ctypes.c_int, [ctypes.c_int, _c_p, _i32, _c_p, _c_p, _c_p, _c_p, _c_p, _c_p, _c_p, _c_p, _i32, _i32, _i32,
                                               _c_p, _sz, _c_p]),
    "avf_token_front_fwd": (ctypes.c_int, [ctypes.c_int, _c_p, _i32, _c_p, _c_p, _c_p, _c_p, _c_p, _c_p, _c_p, _c_p, _i32, _i32, _i32, _i32,
                                           _c_p, _sz, _c_p]),
    "avf_au_logits_fwd": (ctypes.c_int, [_c_p, _i32, _c_p, _c_p, _c_p, _i32, _i32, _c_p]),
    "avf_au_bce_loss": (ctypes.c_int, [_c_p, _i32, _c_p, _c_p, _c_p, _c_p, _i32, _c_p]),
    "avf_au_confusion_update": (ctypes.c_int, [_c_p, _i32, ctypes.c_float, _c_p, _i32, ctypes.c_float, _c_p, _i32, _c_p]),
    "avf_peer_gather_bytes": (_sz, [_i32, _sz]),
    "avf_logits_push": (ctypes.c_int, [_c_p, _sz, _c_p, _i32, _i32, _c_p, _c_p]),
    "avf_logits_wait": (ctypes.c_int, [_c_p, _sz, _i32, _c_p, ctypes.c_uint64, _c_p]),
    "avf_peer_allreduce_bytes": (_sz, [_i32, _sz]),
    "avf_grad_allreduce": (ctypes.c_int, [_c_p, _sz, _i32, _i32, _c_p, ctypes.c_uint64, _c_p]),
    "avf_adam_allreduce_step": (ctypes.c_int, [_c_p, _sz, _i32, _i32, _c_p, ctypes.c_uint64, _c_p, _c_p, _c_p, _c_p] + [ctypes.c_float] * 5
                                + [_i32, ctypes.c_int, ctypes.c_float, _c_p]),
    "avf_cast_f32_to_bf16": (ctypes.c_int, [_c_p, _c_p, _sz, _c_p]),
    "avf_cast_bf16_to_f32": (ctypes.c_int, [_c_p, _c_p, _sz, _c_p]),
    "avf_add_row_periodic": (ctypes.c_int, [_c_p, _i32, _c_p, _i32, _i32, _i32, _c_p]),
    # ---- training ----
    "avf_gemm_workspace_bytes": (_sz, [ctypes.c_int, ctypes.c_int, ctypes.c_int, _i32, _i32, _i32]),
    "avf_gemm": (ctypes.c_int, [ctypes.c_int, ctypes.c_int, ctypes.c_int, _c_p, _i32, _c_p, _i32, _c_p, _c_p, _i32, _c_p, _i32, _c_p, _i32,
                                ctypes.c_int, _i32, _i32, _i32, ctypes.c_int, _c_p, _sz, _c_p]),
    "avf_encoder_tape_bytes": (_sz, [ctypes.POINTER(StackShape), ctypes.c_int]),
    "avf_encoder_bwd_workspace_bytes": (_sz, [ctypes.POINTER(StackShape), ctypes.c_int]),
    "avf_encoder_stack_fwd_train": (ctypes.c_int, [ctypes.c_int, ctypes.POINTER(StackShape), ctypes.POINTER(LayerWeights), _c_p, _i32, _c_p, _i32,
                                                   _c_p, _sz, ctypes.c_float, ctypes.c_uint64, _c_p, _c_p]),
    "avf_encoder_stack_bwd": (ctypes.c_int, [ctypes.c_int, ctypes.POINTER(StackShape), ctypes.POINTER(LayerWeights), _c_p, _sz, _c_p, _i32,
                                             ctypes.POINTER(LayerGrads), ctypes.c_int, _c_p, _sz, ctypes.c_float, ctypes.c_uint64, _c_p, _c_p]),
    "avf_dropout_mask": (ctypes.c_int, [ctypes.c_float, ctypes.c_uint64, _c_p, _i32, _i32, _i32, _i32, _c_p, _c_p]),
    "avf_set_sm_cap": (ctypes.c_int, [ctypes.c_int]),
    "avf_set_pdl_enabled": (ctypes.c_int, [ctypes.c_int]),
    "avf_debug_set_trap_buffer": (ctypes.c_int, [_c_p]),
    "avf_debug_gemm_prof": (ctypes.c_int, [ctypes.POINTER(ctypes.c_uint64)]),
    "avf_debug_tmap_cache": (ctypes.c_int, [ctypes.POINTER(ctypes.c_uint64), ctypes.POINTER(ctypes.c_uint64)]),
    "avf_colsum_workspace_bytes": (_sz, [_i32, _i32]),
    "avf_colsum": (ctypes.c_int, [ctypes.c_int, _c_p, _sz, _i32, _i32, _c_p, _c_p, _sz, _c_p]),
    "avf_layernorm_bwd_workspace_bytes": (_sz, [_i32, _i32]),
    "avf_layernorm_bwd": (ctypes.c_int, [_c_p, _i32, _c_p, _c_p, _c_p, _i32, _c_p, _c_p, _c_p, _c_p, _i32, _i32, _c_p, _sz, _c_p]),
    "avf_attention_bwd": (ctypes.c_int, [ctypes.c_int, _c_p, _c_p, _c_p, _i32, _i32, _i32, _i32, _c_p]),
    "avf_au_former_front_tape_bytes": (_sz, [ctypes.c_int, _i32, _i32]),
    "avf_au_former_front_fwd_train": (ctypes.c_int, [ctypes.c_int, _c_p, _i32, _c_p, _c_p, _c_p, _c_p, ctypes.c_int, ctypes.c_float, _c_p, _c_p,
                                                     _c_p, _c_p, _i32, _i32, _i32, _c_p, _sz, _c_p]),
    "avf_au_former_front_bwd_workspace_bytes": (_sz, [ctypes.c_int, _i32, _i32, _i32]),
    "avf_au_former_front_bwd": (ctypes.c_int, [ctypes.c_int, _c_p, _i32, _c_p, _c_p, _c_p, ctypes.c_int, _c_p, _c_p, _sz, _c_p, _c_p, _i32,
                                               _c_p, _c_p, _c_p, _c_p, _i32, _i32, _i32, _c_p, _sz, _c_p]),
    "avf_au_logits_bwd": (ctypes.c_int, [_c_p, _i32, _c_p, _i32, _c_p, _c_p, _i32, _c_p, _i32, _i32, _c_p]),
    "avf_adam_step": (ctypes.c_int, [_c_p, _c_p, _c_p, _c_p, _c_p, _sz] + [ctypes.c_float] * 5 + [_i32, ctypes.c_int, ctypes.c_float, _c_p]),
    # ---- attention masks (keep: device uint8 [n_seq, n_tok]) ----
    "avf_attention_fwd_masked": (ctypes.c_int, [ctypes.c_int, _c_p, _c_p, _i32, _i32, _i32, _i32, _c_p, _c_p]),
    "avf_attention_bwd_masked": (ctypes.c_int, [ctypes.c_int, _c_p, _c_p, _c_p, _i32, _i32, _i32, _i32, _c_p, _c_p]),
    "avf_encoder_stack_fwd_masked": (ctypes.c_int, [ctypes.c_int, ctypes.POINTER(StackShape), ctypes.POINTER(LayerWeights), _c_p, _c_p, _i32,
                                                    _c_p, _i32, _c_p, _sz, _c_p]),
    "avf_encoder_stack_fwd_train_masked": (ctypes.c_int, [ctypes.c_int, ctypes.POINTER(StackShape), ctypes.POINTER(LayerWeights), _c_p, _c_p, _i32,
                                                          _c_p, _i32, _c_p, _sz, ctypes.c_float, ctypes.c_uint64, _c_p, _c_p]),
    "avf_encoder_stack_bwd_masked": (ctypes.c_int, [ctypes.c_int, ctypes.POINTER(StackShape), ctypes.POINTER(LayerWeights), _c_p, _c_p, _sz, _c_p,
                                                    _i32, ctypes.POINTER(LayerGrads), ctypes.c_int, _c_p, _sz, ctypes.c_float, ctypes.c_uint64, _c_p,
                                                    _c_p]),
    "avf_tformer_fwd_masked": (ctypes.c_int, [ctypes.c_int, ctypes.c_int, ctypes.POINTER(StackShape), ctypes.POINTER(LayerWeights), _c_p, _c_p,
                                              _c_p, _c_p, _c_p, _c_p, _sz, _c_p]),
    # ---- whole-video inference: TFormer clips gathered from a frame bank ----
    "avf_tformer_indexed_workspace_bytes": (_sz, [ctypes.POINTER(StackShape), ctypes.c_int]),
    "avf_tformer_fwd_indexed": (ctypes.c_int, [ctypes.c_int, ctypes.c_int, ctypes.POINTER(StackShape), ctypes.POINTER(LayerWeights), _c_p, _i32, _c_p,
                                               _c_p, _c_p, _c_p, _c_p, _sz, _c_p]),
    # ---- training over a frame bank: the indexed embed and its backward ----
    "avf_tformer_embed_indexed": (ctypes.c_int, [ctypes.c_int, _c_p, _i32, _c_p, _c_p, _c_p, _c_p, _c_p, _i32, _i32, _i32, _c_p]),
    "avf_tformer_embed_indexed_bwd_workspace_bytes": (_sz, [_i32, _i32, _i32]),
    "avf_tformer_embed_indexed_bwd": (ctypes.c_int, [ctypes.c_int, _c_p, _c_p, _i32, _i32, _i32, _i32, _c_p, _c_p, _sz, _c_p]),
    # ---- attention maps (probs: device fp32 [depth, n_seq, heads, n_tok, n_tok]) ----
    "avf_attention_fwd_probs": (ctypes.c_int, [ctypes.c_int, _c_p, _c_p, _i32, _i32, _i32, _i32, _c_p, _c_p, _c_p]),
    "avf_encoder_stack_fwd_probs": (ctypes.c_int, [ctypes.c_int, ctypes.POINTER(StackShape), ctypes.POINTER(LayerWeights), _c_p, _c_p, _i32, _c_p,
                                                   _c_p, _i32, _c_p, _c_p, _sz, _c_p]),
    "avf_tformer_fwd_probs": (ctypes.c_int, [ctypes.c_int, ctypes.c_int, ctypes.POINTER(StackShape), ctypes.POINTER(LayerWeights), _c_p, _c_p,
                                             _c_p, _c_p, _c_p, _c_p, _c_p, _sz, _c_p]),
    "avf_tformer_fwd_indexed_probs": (ctypes.c_int, [ctypes.c_int, ctypes.c_int, ctypes.POINTER(StackShape), ctypes.POINTER(LayerWeights), _c_p,
                                                     _i32, _c_p, _c_p, _c_p, _c_p, _c_p, _c_p, _sz, _c_p]),
    # ---- attention relevance (gmaps: device fp32 [depth, n_seq, heads, n_tok, n_tok]; R: [n_seq, n_tok, n_tok]) ----
    "avf_attention_bwd_gradmaps": (ctypes.c_int, [ctypes.c_int, _c_p, _c_p, _c_p, _i32, _i32, _i32, _i32, _c_p, _c_p, _c_p]),
    "avf_encoder_stack_bwd_gradmaps": (ctypes.c_int, [ctypes.c_int, ctypes.POINTER(StackShape), ctypes.POINTER(LayerWeights), _c_p, _c_p, _sz, _c_p,
                                                      _i32, ctypes.POINTER(LayerGrads), ctypes.c_int, _c_p, _sz, ctypes.c_float, ctypes.c_uint64,
                                                      _c_p, _c_p, _c_p]),
    "avf_attention_rollout": (ctypes.c_int, [_c_p, _i32, _i32, _i32, _i32, _c_p, _c_p]),
}

_lock = threading.Lock()
_lib = None


def sources():
    return sorted(glob.glob(os.path.join(_CSRC, "*.cu")))


def _stale() -> bool:
    if not os.path.exists(LIB_PATH):
        return True
    t = os.path.getmtime(LIB_PATH)
    deps = sources() + glob.glob(os.path.join(_CSRC, "*.cuh")) + glob.glob(os.path.join(_CSRC, "*.h")) + \
        [os.path.join(_ROOT, "include", "avformer_b200.h")]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False, out: str = "") -> str:
    """Compile csrc/*.cu into libavformer_b200.so for sm_100a (nvcc cross-compiles without a GPU).  `out` = alternative
    output path for developer variants (with AVF_NVCC_EXTRA), loaded through AVF_LIB_OVERRIDE."""
    if out:
        force = True
    if not force and not _stale():
        return LIB_PATH
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        raise RuntimeError("avformer_b200: nvcc not found and libavformer_b200.so is missing/stale; cannot build the CUDA path")
    extra = os.environ.get("AVF_NVCC_EXTRA", "").split()          # e.g. -DAVF_FUSED_PROF (developer builds)
    cmd = [nvcc] + NVCC_FLAGS + extra + (["-Xptxas", "-v"] if verbose else []) + ["-o", out or LIB_PATH] + sources()
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("avformer_b200: nvcc failed\n" + res.stdout + res.stderr)
    if verbose:
        print(res.stderr)
    return out or LIB_PATH


def lib() -> ctypes.CDLL:
    """The loaded library (built on first use if the in-tree .so is missing or older than its sources)."""
    global _lib
    if _lib is not None:
        return _lib
    with _lock:
        if _lib is None:
            if _OVERRIDE:
                handle = ctypes.CDLL(_OVERRIDE)
            else:
                try:
                    build()
                except RuntimeError:
                    if not os.path.exists(LIB_PATH):
                        raise
                handle = ctypes.CDLL(LIB_PATH)
            for name, (res, args) in SIGNATURES.items():
                fn = getattr(handle, name)       # AttributeError here = header/library mismatch: fail loudly
                fn.restype, fn.argtypes = res, args
            if os.environ.get("AVF_PDL", "") in ("0", "off"):
                handle.avf_set_pdl_enabled(0)
            if handle.avf_abi_version() != 1:
                raise RuntimeError("avformer_b200: ABI version mismatch")
            _lib = handle
    return _lib


def check(rc: int, what: str = "") -> None:
    if rc != 0:
        msg = lib().avf_last_error().decode("utf-8", "replace")
        raise RuntimeError(f"avformer_b200 {what} failed (code {rc}): {msg}")
