"""CPU-side checks of continuous-batching inference: argument validation in Decoder.inference_continuous and the C-ABI
workspace size (include/genvox_b200.h, gvx_dec_infer_continuous_workspace_bytes)."""
import ctypes as C

import pytest
import torch


def _decoder(precision="fp32"):
    import genvox_b200
    dec = genvox_b200.Decoder(80, 512, 1024, 256, 1000, 0.5, 0.1, 0.1, 1024, 128, 32, 31).eval()
    dec.precision = precision
    return dec


def test_inference_continuous_rejects_bad_arguments():
    dec = _decoder("bf16")
    mem, lens = torch.zeros(3, 5, 512), torch.tensor([5, 4, 3])
    for slots in (0, -1, 129):
        with pytest.raises(ValueError, match="slots"):
            dec.inference_continuous(mem, lens, slots=slots)
    dec.precision = "fp32"
    for caps in ([0, 5, 5], [5, 1001, 5], [5, 5]):
        with pytest.raises(ValueError, match="frame_caps"):
            dec.inference_continuous(mem, lens, slots=2, frame_caps=torch.tensor(caps))
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        dec.inference_continuous(mem, lens, slots=2, frame_caps=[1, 1000, 7])
    dec.train()
    with pytest.raises(RuntimeError, match="eval mode"):
        dec.inference_continuous(mem, lens, slots=2)


def test_continuous_workspace_size():
    from genvox_b200 import _native
    lib = _native.load()
    dec = _decoder()
    d = dec._dims()
    size = lambda U, N=150, S=64: lib.gvx_dec_infer_continuous_workspace_bytes(C.byref(d), U, N, S)
    assert 0 < size(64) < size(512) < size(4096)
    # one slot block plus the processed memory of the whole queue, [ceil(U/S)*S, N, att_dim] floats
    assert size(4096) - size(64) == (4096 - 64) * 150 * 128 * 4
    assert size(0) == 0 and size(64, N=0) == 0 and size(64, S=0) == 0
    dec.precision = "bf16"
    d = dec._dims()
    assert size(64, S=128) > 0 and size(64, S=129) == 0
