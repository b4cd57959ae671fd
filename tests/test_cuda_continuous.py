"""Continuous-batching inference (Decoder.inference_continuous, gvx_dec_infer_continuous) on the GPU.

The contract is an exact identity: utterance u, whichever slot it ran in and whatever the other slots held, decodes
bit-identically to row r of a static `inference` call with the same S rows, N, seed and precision, u in row r and
dropout_row_offset = u + row_offset - r; its frame count is that row's stop step.  A slot reset that misses any piece of
recurrent state, or a prenet that draws the wrong dropout row or frame, breaks the identity at the first refill."""
import numpy as np
import pytest
import torch

import genvox_b200
from genvox_b200 import _native, synthesis
from oracle import decoder_oracle as O
from oracle import synth
from test_cuda_parity import argmax_agrees, make_decoder
from test_cuda_synthesis import _model

pytestmark = pytest.mark.gpu

SEED = 4242
STEPS = 24
GVX_STOP_POLL = 16         # include/genvox_b200.h: the host reads the active-slot count every 16 steps
GATE_BIAS = -0.15          # SMALL_DIMS, weights seed 21: stops at frames 1 .. 3 and runs to the step limit, mixed


def _decoder(dev, precision, dims=synth.SMALL_DIMS, gate_bias=GATE_BIAS):
    W = synth.make_decoder_weights(21, dims)
    W["gate_layer.linear_layer.bias"][:] = gate_bias
    dec = make_decoder(dims, W, dev, False)
    dec.precision = precision
    return dec, W


def _queue(dev, U, N, dims=synth.SMALL_DIMS, seed=5):
    """U ragged utterances (9 .. N tokens), zero past each length as synthesis pads them."""
    mem, _, _ = synth.make_inputs(seed, U, N, 0, dims, ragged=False)
    lens = (9 + np.floor(synth.uniform01(seed + 1, 1, U) * (N - 8))).astype(np.int64)
    lens[0] = N
    for u, n in enumerate(lens):
        mem[u, n:] = 0
    return torch.from_numpy(mem).to(dev), torch.from_numpy(lens).to(dev)


def _sync():
    torch.cuda.synchronize()
    genvox_b200.check_device_errors()


def _continuous(dec, memory, lens, S, caps=None, ignore_gate=False, row_offset=0, return_alignments=True):
    dec.dropout_row_offset = row_offset
    dec.set_dropout_seed(SEED)
    out = dec.inference_continuous(memory, lens, slots=S, max_decoder_steps=STEPS, frame_caps=caps, ignore_gate=ignore_gate,
                                   return_alignments=return_alignments)
    dec.dropout_row_offset = 0
    _sync()
    return out, dec.last_n_frames.long().cpu()


def _static(dec, memory, lens, u0, S, row_offset=0):
    """utterances u0 .. u0+S-1 in rows 0 .. S-1 (a short last group is padded with copies of utterance 0)"""
    idx = [u if u < memory.shape[0] else 0 for u in range(u0, u0 + S)]
    dec.dropout_row_offset = u0 + row_offset
    dec.set_dropout_seed(SEED)
    out = dec.inference(memory[idx].contiguous(), memory_lengths=lens[idx].contiguous(), ignore_gate=True, max_decoder_steps=STEPS)
    dec.dropout_row_offset = 0
    _sync()
    return out


def _stop_frames(gate, cap, thr):
    """first frame whose sigmoid(gate) > thr (frame included), else the cap"""
    fired = torch.nonzero(torch.sigmoid(gate[:cap]) > thr)
    return int(fired[0]) + 1 if len(fired) and int(fired[0]) < cap else cap


def _check_against_static(dec, memory, lens, S, caps=None, row_offset=0, ignore_gate=False):
    U = memory.shape[0]
    (mel, gate, align), nf = _continuous(dec, memory, lens, S, caps, ignore_gate, row_offset)
    capv = [STEPS if caps is None else min(STEPS, int(caps[u])) for u in range(U)]
    assert mel.shape[2] == int(nf.max())
    for u0 in range(0, U, S):
        smel, sgate, salign = _static(dec, memory, lens, u0, S, row_offset)
        for r, u in enumerate(range(u0, min(u0 + S, U))):
            n = int(nf[u])
            want = capv[u] if ignore_gate else _stop_frames(sgate[r].cpu(), capv[u], dec.gate_threshold)
            assert n == want, (u, n, want)
            assert torch.equal(mel[u, :, :n], smel[r, :, :n]), ("mel", u)
            assert torch.equal(gate[u, :n], sgate[r, :n]), ("gate", u)
            assert torch.equal(align[u, :n], salign[r, :n]), ("align", u)
            assert not bool(mel[u, :, n:].any()) and not bool(gate[u, n:].any()) and not bool(align[u, n:].any()), ("tail", u)
    return nf


# --------------------------------------------------------------------------- 1. bit-exact against static inference
@pytest.mark.parametrize("precision,row_offset", [("fp32", 0), ("bf16", 0), ("fp32", 37), ("bf16", 37)])
def test_bit_exact_against_static(cuda_device, precision, row_offset):
    dec, _ = _decoder(cuda_device, precision)
    memory, lens = _queue(cuda_device, 23, 64)
    caps = torch.full((23,), STEPS, dtype=torch.int32)
    caps[[1, 4, 8, 13, 20]] = torch.tensor([5, 9, 2, 17, 11], dtype=torch.int32)
    nf = _check_against_static(dec, memory, lens, 4, caps, row_offset)
    assert len(set(nf.tolist())) >= 4, nf                        # stops really are spread, so slots refill at different steps
    assert dec.last_steps_run < (23 + 3) // 4 * STEPS


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_bit_exact_at_full_size(cuda_device, precision):
    """Reference dims (the two-CTA cluster attention kernel, which prefetches the processed memory and reads the lengths
    before it waits on the previous kernel); the frame caps make the slots refill whatever the random-init gate does."""
    dims = synth.DecoderDims()
    dec, _ = _decoder(cuda_device, precision, dims, gate_bias=-0.2)
    memory, lens = _queue(cuda_device, 10, 64, dims)
    caps = torch.tensor([3, 7, 1, 12, 5, 9, 2, 16, 4, 11], dtype=torch.int32)
    _check_against_static(dec, memory, lens, 4, caps, row_offset=5)


def test_many_slots_take_the_unfused_prenet(cuda_device):
    """fp32 with more than 64 slots: the prenet runs as two GEMMs whose epilogue reads the per-row frame and row"""
    dec, _ = _decoder(cuda_device, "fp32")
    memory, lens = _queue(cuda_device, 150, 32, seed=9)
    caps = torch.from_numpy((1 + np.floor(synth.uniform01(12, 1, 150) * STEPS)).astype(np.int32))
    _check_against_static(dec, memory, lens, 72, caps)


# --------------------------------------------------------------------------- 2. against the oracle (fp32)
def test_matches_oracle_fp32(cuda_device):
    dec, W = _decoder(cuda_device, "fp32")
    memory, lens = _queue(cuda_device, 23, 64)
    (mel, gate, align), nf = _continuous(dec, memory, lens, 4)
    P = O.as_params(W)
    for u in (0, 5, 11, 22):
        rm, rg, ra, rn = O.inference(P, memory[u:u + 1].cpu(), lens[u:u + 1].cpu(), STEPS, dec.gate_threshold, False, SEED,
                                     False, dec.p_attention_dropout, dec.p_decoder_dropout, row_offset=u)
        n = int(rn[0])
        assert int(nf[u]) == n, (u, int(nf[u]), n)
        scale = float(rm.abs().max())
        assert float((mel[u, :, :n].cpu() - rm[0, :, :n]).abs().max()) <= 1e-4 * scale, u
        assert float((gate[u, :n].cpu() - rg[0, :n]).abs().max()) <= 1e-4 * max(float(rg.abs().max()), 1e-30), u
        ok, _ = argmax_agrees(align[u, :n].cpu().numpy(), ra[0, :n].numpy())
        assert ok, u


# --------------------------------------------------------------------------- 3. edges
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_fewer_utterances_than_slots(cuda_device, precision):
    dec, _ = _decoder(cuda_device, precision)
    memory, lens = _queue(cuda_device, 3, 64)
    _check_against_static(dec, memory, lens, 8)
    _check_against_static(dec, memory[:1].contiguous(), lens[:1].contiguous(), 8)


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_one_slot_equals_one_utterance_at_a_time(cuda_device, precision):
    dec, _ = _decoder(cuda_device, precision)
    memory, lens = _queue(cuda_device, 7, 64)
    caps = torch.tensor([24, 3, 24, 8, 1, 24, 12], dtype=torch.int32)
    _check_against_static(dec, memory, lens, 1, caps)


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_every_utterance_stops_at_frame_one(cuda_device, precision):
    """a slot is admitted at every step"""
    dec, _ = _decoder(cuda_device, precision)
    memory, lens = _queue(cuda_device, 23, 64)
    nf = _check_against_static(dec, memory, lens, 4, torch.ones(23, dtype=torch.int32))
    assert nf.tolist() == [1] * 23
    assert dec.last_steps_run <= GVX_STOP_POLL
    dec.gate_layer.linear_layer.bias.data.fill_(30.0)              # the gate fires at frame 1 of every utterance
    dec.invalidate_packed()
    nf = _check_against_static(dec, memory, lens, 4)
    assert nf.tolist() == [1] * 23


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_without_alignments_and_repeated(cuda_device, precision):
    dec, _ = _decoder(cuda_device, precision)
    memory, lens = _queue(cuda_device, 23, 64)
    (m1, g1, a1), n1 = _continuous(dec, memory, lens, 4)
    (m2, g2, a2), n2 = _continuous(dec, memory, lens, 4, return_alignments=False)
    (m3, g3, a3), n3 = _continuous(dec, memory, lens, 4)
    assert a2 is None
    assert torch.equal(n1, n2) and torch.equal(n1, n3)
    assert torch.equal(m1, m2) and torch.equal(g1, g2)
    assert torch.equal(m1, m3) and torch.equal(g1, g3) and torch.equal(a1, a3)


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_ignore_gate_stops_at_the_caps(cuda_device, precision):
    dec, _ = _decoder(cuda_device, precision, gate_bias=30.0)      # the gate would fire at once
    memory, lens = _queue(cuda_device, 9, 64)
    caps = torch.tensor([4, 24, 1, 7, 13, 2, 24, 5, 9], dtype=torch.int32)
    nf = _check_against_static(dec, memory, lens, 4, caps, ignore_gate=True)
    assert nf.tolist() == caps.tolist()


# --------------------------------------------------------------------------- 4. launch budget
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_launches_per_step_equal_static(cuda_device, precision):
    lib = _native.load()
    dec, _ = _decoder(cuda_device, precision, gate_bias=-30.0)     # the gate never fires: the static run takes every step
    memory, lens = _queue(cuda_device, 8, 64)

    def launches(fn):
        fn()                                                        # warm (weight packing)
        _sync()
        c0 = lib.gvx_launch_count()
        fn()
        _sync()
        return lib.gvx_launch_count() - c0

    def static(steps):
        return launches(lambda: dec.inference(memory[:4], memory_lengths=lens[:4], max_decoder_steps=steps))

    def continuous(cap):
        def run():
            dec.inference_continuous(memory, lens, slots=4, max_decoder_steps=STEPS,
                                     frame_caps=torch.full((8,), cap, dtype=torch.int32))
            run.steps = dec.last_steps_run
        n = launches(run)
        return n, run.steps

    per_static = (static(20) - static(10)) / 10
    (c1, s1), (c2, s2) = continuous(8), continuous(16)           # two rounds of 4 slots, ending on a host poll
    assert (s1, s2) == (16, 32)
    assert (c2 - c1) / (s2 - s1) == per_static


# --------------------------------------------------------------------------- 5. synthesis wrapper
def test_continuous_inference_equals_one_utterance_at_a_time(cuda_device):
    m = _model(cuda_device, max_steps=24)
    g = torch.Generator().manual_seed(5)
    rows = [torch.randint(0, 40, (n,), generator=g).tolist() for n in (37, 9, 64, 23, 50, 12, 64)]
    m.decoder.gate_layer.linear_layer.bias.data.fill_(-0.2)
    m.decoder._next_seed = lambda: 1234
    cont = synthesis.continuous_inference(m, rows, slots=3)
    stops = []
    for i, r in enumerate(rows):
        m.decoder.dropout_row_offset = i
        single = m.inference({"tokens": torch.tensor(r, dtype=torch.int32, device=cuda_device).unsqueeze(0)})
        m.decoder.dropout_row_offset = 0
        stops.append(single["mel_outputs"].shape[2])
        for k, v in single.items():
            assert cont[i][k].shape == v.shape, (i, k, cont[i][k].shape, v.shape)
            err = float((cont[i][k] - v).abs().max() / v.abs().max().clamp_min(1e-30))
            assert err < 1e-4, (i, k, err)
    assert len(set(stops)) > 1 or stops[0] == 24
    _sync()

