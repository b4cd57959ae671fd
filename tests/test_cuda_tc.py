"""GPU tests of the tcgen05 / TMEM / TMA gate-GEMM engine (genvox_b200/csrc/gvx_tc.cuh) on its own:
out = X . W^T with bf16-rounded operands and fp32 accumulation, against an fp64 matmul of the same
bf16-rounded operands (so the only difference is the accumulation order: tolerance 2e-6 of max|ref|)."""
import ctypes as C

import pytest
import torch

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("B,M,K,KS", [(64, 128, 64, 1), (64, 256, 128, 1), (16, 128, 64, 1), (64, 4096, 1792, 4),
                                      (64, 4096, 2560, 4), (5, 81, 1536, 3), (128, 1792, 4096, 10), (32, 200, 100, 2),
                                      (64, 2560, 4096, 7), (64, 128, 1024, 8), (3, 1024, 128, 2)])
def test_tc_gemm_matches_bf16_matmul(cuda_device, B, M, K, KS):
    from genvox_b200 import _native
    from genvox_b200.decoder import _ptr, _stream
    lib = _native.load()
    g = torch.Generator().manual_seed(B * 7919 + M * 31 + K)
    W = (torch.rand(M, K, generator=g) - 0.5).to(cuda_device)
    X = (torch.rand(B, K, generator=g) - 0.5).mul(4).to(cuda_device)
    out = torch.full((B, M), float("nan"), device=cuda_device)
    _native.check(lib.gvx_test_tc_gemm(_ptr(W), _ptr(X), B, M, K, KS, _ptr(out), _stream()), "gvx_test_tc_gemm")
    ref = X.bfloat16().double() @ W.bfloat16().double().t()
    err = float((out.double() - ref).abs().max() / ref.abs().max())
    assert err < 2e-6, err


@pytest.mark.parametrize("M,N,K,mode", [(128, 128, 64, 0), (300, 200, 136, 0), (4096, 256, 512, 0), (1000, 81, 1536, 0),
                                        (256, 512, 2048, 1), (4096, 1792, 3208, 1), (128, 1024, 6400, 1),
                                        # long K with few tiles: the deterministic split-K path (partial tiles + fixed-order reduction)
                                        (128, 1024, 16384, 1), (256, 768, 8192, 0), (88, 1536, 12800, 1),
                                        # the weight gradients of training at configs[2] (K = T*B = 51200), with the split counts
                                        # training selects: decoder-LSTM W_ih part and whole [W_ih | W_hh], attention LSTM, query
                                        (4096, 1536, 51200, 1), (4096, 2560, 51200, 1), (4096, 1792, 51200, 1), (128, 1024, 51200, 1)])
def test_nt_gemm_matches_torch(cuda_device, M, N, K, mode):
    """The tcgen05 GEMM of the time-batched contractions (csrc/gvx_nt_gemm.cuh): tails in M, N and K, the transposed
    (weight-gradient) path, split-K with its fixed-order reduction, bit-exact run to run."""
    import ctypes as C
    import torch
    from genvox_b200 import _native
    lib = _native.load()
    # operands and the fp64 reference on the device: the production shapes are 0.5 TFLOP in fp64
    g = torch.Generator(device=cuda_device).manual_seed(M * 7 + N * 3 + K)
    if mode == 1:       # MN-major operands A^T [K, M], B^T [K, N]
        a_dev = torch.randn(K, M, generator=g, device=cuda_device)
        b_dev = torch.randn(K, N, generator=g, device=cuda_device)
        ref = a_dev.bfloat16().double().t() @ b_dev.bfloat16().double()
    else:
        a_dev = torch.randn(M, K, generator=g, device=cuda_device)
        b_dev = torch.randn(N, K, generator=g, device=cuda_device)
        ref = a_dev.bfloat16().double() @ b_dev.bfloat16().double().t()
    outs = []
    for _ in range(2):
        Cd = torch.full((M, N), float("nan"), device=cuda_device)
        _native.check(lib.gvx_test_nt_gemm(C.c_void_p(a_dev.data_ptr()), C.c_void_p(b_dev.data_ptr()), M, N, K, mode,
                                           C.c_void_p(Cd.data_ptr()), C.c_void_p(torch.cuda.current_stream().cuda_stream)), "gvx_test_nt_gemm")
        torch.cuda.synchronize()
        outs.append(Cd)
    assert torch.equal(outs[0], outs[1])
    err = float((outs[0].double() - ref).abs().max() / ref.abs().max())
    # fp32 accumulation over K products: 2.2e-5 of max|ref| at K = 51200 (B200); one K block of 64 dropped or repeated moves an
    # element by ~7e-3 of max|ref|
    assert err < (2e-5 if K <= 16384 else 5e-5), err
