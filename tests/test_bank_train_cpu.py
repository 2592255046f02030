"""Training over a frame bank without a device: the indexed embed and its scatter-add backward refuse to compute instead of falling
back, and their symbols are exported."""
import pytest
import torch

import avformer_b200 as A


def test_bank_training_symbols_are_exported():
    L = A._lib.lib()
    for name in ("avf_tformer_embed_indexed", "avf_tformer_embed_indexed_bwd_workspace_bytes", "avf_tformer_embed_indexed_bwd"):
        assert hasattr(L, name), name


def test_scatter_workspace_is_positive():
    L = A._lib.lib()
    assert L.avf_tformer_embed_indexed_bwd_workspace_bytes(256, 16, 300) >= 4 * (301 + 2 * 256 * 16)
    assert L.avf_tformer_embed_indexed_bwd_workspace_bytes(1, 8, 0) > 0
    assert L.avf_tformer_embed_indexed_bwd_workspace_bytes(0, 8, 10) == 0


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-device behaviour")
def test_bank_training_without_a_device_is_an_error_not_a_fallback():
    L = A._lib.lib()
    rc = L.avf_tformer_embed_indexed(A._lib.AVF_FP32, None, 0, None, None, None, None, None, 4, 16, 512, None)
    assert rc == -2                                                       # AVF_ENODEVICE
    assert b"no CPU fallback" in L.avf_last_error()
    rc = L.avf_tformer_embed_indexed_bwd(A._lib.AVF_FP32, None, None, 4, 16, 512, 20, None, None, 0, None)
    assert rc == -2
    assert b"no CPU fallback" in L.avf_last_error()
    tf = A.TFormer(num_patches=16).train()
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        tf.forward_indexed(torch.zeros(20, 512, requires_grad=True), torch.zeros(4, 16, dtype=torch.int64))
