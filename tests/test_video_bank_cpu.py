"""Whole-video inference without a device: the frame-bank TFormer entry point refuses to compute instead of falling back."""
import ctypes

import pytest
import torch

import avformer_b200 as A


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-device behaviour")
def test_indexed_tformer_without_a_device_is_an_error_not_a_fallback():
    L = A._lib.lib()
    shape = A._lib.StackShape(4, 17, 512, 8, 64, 1024, 3)
    assert L.avf_tformer_indexed_workspace_bytes(ctypes.byref(shape), A._lib.AVF_BF16) > L.avf_tformer_workspace_bytes(ctypes.byref(shape), A._lib.AVF_BF16)
    layers = (A._lib.LayerWeights * 3)()
    rc = L.avf_tformer_fwd_indexed(A._lib.AVF_BF16, A._lib.AVF_FP32, ctypes.byref(shape), layers, None, 0, None, None, None, None, None, 0, None)
    assert rc == -2                                                       # AVF_ENODEVICE
    assert b"no CPU fallback" in L.avf_last_error()
    tf = A.TFormer(num_patches=16).eval()
    with pytest.raises(RuntimeError, match="no CPU fallback"), torch.no_grad():
        tf.cls_features_indexed(torch.zeros(20, 512), torch.zeros(4, 16, dtype=torch.int64))
