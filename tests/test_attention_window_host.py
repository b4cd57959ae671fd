"""CPU checks of the attention constraint (Decoder.attention_window, gvx_dec_*_windowed): argument validation in Python and
in the C ABI, and the rule itself on the windowed oracle (tests/attention_window_oracle.py, built on oracle/decoder_oracle.py),
which the GPU tests compare the kernels with.

Rule: at step t, last = argmax_n w_{t-1}[b, n] (lowest index on ties; all-zero w_{t-1} at t = 0 gives 0), and tokens
outside [last - backward, last + forward) get energy -inf, so weight exactly 0."""
import ctypes as C

import numpy as np
import pytest
import torch

import genvox_b200
from genvox_b200 import _native, synthesis
import attention_window_oracle as WO
from oracle import decoder_oracle as O
from oracle import synth

BAD_WINDOWS = [(-1, 3), (0, 0), (1, -2), (1,), (1, 2, 3), 5, "ab", (1.5, 3), (True, 3), (1, 2 ** 31), (None, 3)]


def _dec():
    return genvox_b200.Decoder(**synth.SMALL_DIMS.kwargs()).eval()


# --------------------------------------------------------------------------- Python API
def test_attribute_defaults_to_none_and_stays_out_of_the_state_dict():
    dec = _dec()
    assert dec.attention_window is None
    keys = set(dec.state_dict())
    dec.attention_window = (1, 3)
    assert set(dec.state_dict()) == keys
    dec.load_state_dict(_dec().state_dict())                                 # loading a checkpoint leaves it alone
    assert dec.attention_window == (1, 3)


@pytest.mark.parametrize("window", BAD_WINDOWS)
def test_bad_windows_raise_value_error(window):
    dec = _dec()
    memory = torch.zeros(2, 5, synth.SMALL_DIMS.encoder_embedding_dim)
    with pytest.raises(ValueError, match="attention_window"):
        dec.inference(memory, attention_window=window)
    with pytest.raises(ValueError, match="attention_window"):
        dec.inference_continuous(memory, None, slots=2, attention_window=window)
    with pytest.raises(ValueError, match="attention_window"):
        dec.session(5, slots=2, attention_window=window)
    dec.attention_window = window                                            # through the attribute too
    with pytest.raises(ValueError, match="attention_window"):
        dec.inference(memory)
    with pytest.raises(ValueError, match="attention_window"):
        dec.inference_continuous(memory, None, slots=2)
    with pytest.raises(ValueError, match="attention_window"):
        dec.session(5, slots=2)


@pytest.mark.parametrize("window", [None, (0, 1), (1, 3), (np.int64(2), 7), (2 ** 31 - 1, 2 ** 31 - 1)])
def test_good_windows_reach_the_device_check(window):
    """valid windows pass validation; with CPU tensors the call then fails on the missing device, as without a window"""
    dec = _dec()
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        dec.inference(torch.zeros(1, 5, synth.SMALL_DIMS.encoder_embedding_dim), attention_window=window)


def test_batched_inference_passes_the_window_only_when_given():
    seen = []

    class Dec(torch.nn.Module):
        def inference(self, memory, memory_lengths=None, ignore_gate=False, max_decoder_steps=None, **kw):
            seen.append(kw)
            B, N, _ = memory.shape
            self.last_n_frames = torch.full((B,), 2, dtype=torch.int32)
            return torch.zeros(B, 3, 2), torch.zeros(B, 2), torch.zeros(B, 2, N)

    model = torch.nn.Module()
    model.embedding = torch.nn.Embedding(10, 4)
    model.encoder = type("E", (torch.nn.Module,), {"inference": lambda self, x: x.transpose(1, 2)})()
    model.decoder = Dec()
    model.postnet = lambda m: m
    synthesis.batched_inference(model, [[1, 2, 3]])
    synthesis.batched_inference(model, [[1, 2, 3]], attention_window=(1, 3))
    synthesis.batched_inference(model, [[1, 2, 3]], attention_window=None)
    assert seen == [{}, {"attention_window": (1, 3)}, {"attention_window": None}]


# --------------------------------------------------------------------------- C ABI refusals
def _c_args():
    d = _dims()
    w = _native.GvxWeights()
    fake = C.c_void_p(16)             # never dereferenced: the window is refused first
    return d, w, fake


def _dims():
    return _dec()._dims()


@pytest.mark.parametrize("back,fwd,what", [(-1, 3, "att_backward"), (1, -1, "att_forward"), (-5, -5, "att_backward")])
def test_c_abi_refuses_negative_windows(back, fwd, what):
    lib = _native.load()
    d, w, p = _c_args()
    ran, ran_ll = C.c_int(0), C.c_longlong(0)
    assert lib.gvx_dec_infer_windowed(C.byref(d), C.byref(w), p, p, None, 2, 5, 10, 0.5, 0, 1, 0, 0, p, p, p, p, C.byref(ran),
                                      back, fwd, p, None) != 0
    assert what.encode() in lib.gvx_last_error()
    assert lib.gvx_dec_infer_continuous_windowed(C.byref(d), C.byref(w), p, p, None, 3, 5, 2, 10, None, 0.5, 0, 1, 0, p, p, p, p,
                                                 C.byref(ran_ll), back, fwd, p, None) != 0
    assert what.encode() in lib.gvx_last_error()
    s = _native.GvxSession()
    s.N, s.slots, s.capacity, s.max_steps = 5, 2, 4, 10
    assert lib.gvx_dec_session_step_windowed(C.byref(d), C.byref(w), p, C.byref(s), 4, p, p, p, p, p, C.byref(ran), back, fwd,
                                             p, None) != 0
    assert what.encode() in lib.gvx_last_error()


# --------------------------------------------------------------------------- the rule, on the oracle
def _oracle_run(window, dims=synth.SMALL_DIMS, B=3, N=24, steps=20, dtype=torch.float64, peaks=None):
    W = synth.make_decoder_weights(21, dims)
    mem, _, lens = synth.make_inputs(5, B, N, 0, dims)
    return WO.inference(O.as_params(W, dtype), torch.from_numpy(mem).to(dtype), lens, steps, 0.5, True, 77, False,
                       window=window, peaks=peaks), lens


@pytest.mark.parametrize("dtype,bf16", [(torch.float64, False), (torch.float32, False), (torch.float32, True)])
def test_windowed_oracle_without_a_window_is_the_oracle(dtype, bf16):
    """window=None: exactly oracle/decoder_oracle.py's inference, gate-stopped and ragged, in its fp32 / fp64 / bf16 modes"""
    dims = synth.SMALL_DIMS
    W = synth.make_decoder_weights(21, dims)
    mem, _, lens = synth.make_inputs(5, 3, 24, 0, dims)
    P, memory = O.as_params(W, dtype), torch.from_numpy(mem).to(dtype)
    args = (P, memory, lens, 20, 0.5, False, 77, False, 0.1, 0.1, 2)
    if bf16:
        with O.bf16_semantics():
            want, got = O.inference(*args), WO.inference(*args)
    else:
        want, got = O.inference(*args), WO.inference(*args)
    for x, y in zip(want, got):
        assert torch.equal(x, y)


def test_oracle_window_covering_everything_is_bit_identical_to_none():
    (m0, g0, a0, n0), _ = _oracle_run(None)
    (m1, g1, a1, n1), _ = _oracle_run((24, 24))
    assert torch.equal(m0, m1) and torch.equal(g0, g1) and torch.equal(a0, a1) and torch.equal(n0, n1)


def _check_support_and_step_bound(align, lens, back, fwd):
    """align [B, T, N]: weights exactly 0 outside [p_{t-1} - back, p_{t-1} + fwd), p_{-1} = 0, and past each length"""
    B, T, N = align.shape
    p = align.argmax(-1)
    prev = torch.cat([torch.zeros(B, 1, dtype=p.dtype), p[:, :-1]], dim=1)
    n = torch.arange(N)[None, None, :]
    outside = (n < prev[..., None] - back) | (n >= prev[..., None] + fwd) | (n >= torch.as_tensor(lens)[:, None, None])
    assert not bool(align[outside].any())
    step = p - prev
    assert int(step.min()) >= -back and int(step.max()) <= fwd - 1, (int(step.min()), int(step.max()))


@pytest.mark.parametrize("window", [(1, 3), (0, 1), (2, 5)])
def test_oracle_support_and_step_bound(window):
    (m, g, a, _), lens = _oracle_run(window)
    _check_support_and_step_bound(a, lens, *window)
    (_, _, a0, _), _ = _oracle_run(None)
    assert not torch.equal(a, a0)                                            # the constraint really changed the decode
    if window == (0, 1):
        assert torch.equal(a.argmax(-1), torch.zeros_like(a.argmax(-1)))     # never leaves token 0: all weight there
        assert torch.equal(a[..., 0], torch.ones_like(a[..., 0]))


def test_oracle_forced_peaks_equal_its_own_argmax():
    (m, g, a, n), _ = _oracle_run((1, 3))
    B, T, N = a.shape
    peaks = [torch.zeros(B, dtype=torch.int64)] + [a[:, t - 1].argmax(-1) for t in range(1, T)]
    (m1, g1, a1, n1), _ = _oracle_run((1, 3), peaks=peaks)
    assert torch.equal(m, m1) and torch.equal(a, a1)


def test_oracle_tie_takes_the_lowest_index():
    dims = synth.SMALL_DIMS
    P = O.as_params(synth.make_decoder_weights(21, dims), torch.float64)
    B, N = 4, 12
    mem = torch.from_numpy(synth.make_inputs(5, B, N, 0, dims)[0]).double()
    pm = torch.nn.functional.linear(mem, P["attention_layer.memory_layer.linear_layer.weight"])
    w_prev = torch.zeros(B, N, dtype=torch.float64)
    w_prev[1, [3, 7]] = 0.5                                                  # tie: 3 wins
    w_prev[2, [9, 10, 11]] = 1.0 / 3                                         # tie: 9 wins
    w_prev[3, 5] = 0.25
    w_prev[3, 6] = 0.25 + 1e-12                                              # no tie: 6 wins
    h = torch.from_numpy(synth.uniform01(3, 1, B * dims.attention_rnn_dim).reshape(B, -1) - 0.5)
    _, w = WO.attention(P, h, mem, pm, w_prev, torch.zeros(B, N, dtype=torch.float64), None, window=(0, 1))
    assert w.argmax(-1).tolist() == [0, 3, 9, 6]
    assert torch.equal(w.sum(-1), torch.ones(B, dtype=torch.float64)) and int((w != 0).sum()) == B
    assert torch.equal(w_prev.argmax(-1), torch.tensor([0, 3, 9, 6]))        # the rule is torch.argmax's
