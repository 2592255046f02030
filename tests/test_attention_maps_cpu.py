"""CPU-side checks of the attention-map entry points: exported with the declared signatures, and without a device an error, never a
CPU computation."""
import ctypes

import pytest
import torch

import avformer_b200 as A

NEW = ("avf_attention_fwd_probs", "avf_encoder_stack_fwd_probs", "avf_tformer_fwd_probs", "avf_tformer_fwd_indexed_probs")


def test_map_entry_points_are_exported():
    lib = ctypes.CDLL(A._lib.build())
    for name in NEW:
        assert hasattr(lib, name) and name in A._lib.SIGNATURES, name
    assert A._lib.lib().avf_abi_version() == 1


def test_python_map_calls_exist():
    assert callable(A.functional.attention_fwd_probs) and callable(A.functional.encoder_stack_probs_)
    for cls, names in ((A.Transformer, ("attention_maps",)), (A.TFormer, ("attention_maps", "attention_maps_indexed")),
                       (A.TwoStreamAuralVisualFormer, ("attention_maps",))):
        for n in names:
            assert callable(getattr(cls, n)), f"{cls.__name__}.{n}"
    assert A.TwoStreamAuralVisualFormer.MAP_STACKS == ("sformer", "tformer", "audio_au_former", "video_au_former", "fusion_head")


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-device behaviour")
def test_maps_without_a_device_are_an_error():
    L = A._lib.lib()
    assert L.avf_attention_fwd_probs(1, None, None, 1, 12, 8, 32, None, None, None) == -2          # AVF_ENODEVICE
    assert b"no CPU fallback" in L.avf_last_error()
    with pytest.raises(RuntimeError, match="no CPU fallback"), torch.no_grad():
        A.Transformer(128, 1, 8, 32, 256).eval().attention_maps(torch.zeros(1, 12, 128))
