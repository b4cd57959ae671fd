"""Decoder sessions (Decoder.session, gvx_dec_session_*, synthesis.SynthesisSession) on the GPU.

The contract is the continuous one: utterance `id` decodes bit-identically to row r of a static `inference` call with the
same S rows, N, seed and precision, id in row r and dropout_row_offset = id + row_offset - r, whatever the submission
times, the step counts per call and the other slots were.  A state word that does not survive between calls (the output
ring, the slot ping-pong, the h / c halves, the prenet barrier), or a head admission that misses part of a slot's reset,
breaks the identity at the first call boundary."""
import numpy as np
import pytest
import torch

from genvox_b200 import _native, synthesis
from oracle import decoder_oracle as O
from oracle import synth
from test_cuda_continuous import SEED, STEPS, _continuous, _decoder, _queue, _static, _stop_frames, _sync
from test_cuda_parity import argmax_agrees
from test_cuda_synthesis import _model

pytestmark = pytest.mark.gpu


def _session(dec, N, S, capacity=64, row_offset=0, ignore_gate=False, return_alignments=True):
    dec.dropout_row_offset = row_offset
    dec.set_dropout_seed(SEED)
    sess = dec.session(N, slots=S, capacity=capacity, max_decoder_steps=STEPS, ignore_gate=ignore_gate,
                       return_alignments=return_alignments)
    dec.dropout_row_offset = 0
    return sess


def _drive(sess, memory, lens, caps, plan):
    """plan: ("submit", lo, hi) queues utterances lo .. hi-1 (their ids must be lo .. hi-1), ("step", k) runs one step
    call, ("drain", k) runs step calls of k until nothing is active or queued.  Returns {id: (mel, gate, align, n)}."""
    parts, fin = {}, {}

    def absorb(res):
        chunks, done = res
        for i, c in chunks.items():
            assert i not in fin, ("frames after the last one", i)
            parts.setdefault(i, []).append(c)
        for i, n in done.items():
            fin[i] = n

    for op, *args in plan:
        if op == "submit":
            lo, hi = args
            ids = sess.submit(memory[lo:hi], lens[lo:hi], caps[lo:hi] if caps is not None else None)
            assert ids == list(range(lo, hi)), ids
        elif op == "step":
            absorb(sess.step(args[0]))
        else:
            while sess.active or sess.pending:
                absorb(sess.step(args[0]))
    _sync()
    out = {}
    for i, ps in parts.items():
        mel = torch.cat([p[0] for p in ps], dim=1)
        gate = torch.cat([p[1] for p in ps])
        align = torch.cat([p[2] for p in ps]) if ps[0][2] is not None else None
        n = fin.get(i)
        assert n is None or mel.shape[1] == n, (i, mel.shape, n)      # the chunks add up to the frame count
        out[i] = (mel, gate, align, n)
    return out


def _check_static(dec, memory, lens, S, out, caps=None, row_offset=0, ignore_gate=False):
    U = memory.shape[0]
    assert sorted(out) == list(range(U)) and all(out[u][3] is not None for u in range(U))
    for u0 in range(0, U, S):
        smel, sgate, salign = _static(dec, memory, lens, u0, S, row_offset)
        for r, u in enumerate(range(u0, min(u0 + S, U))):
            mel, gate, align, n = out[u]
            cap = STEPS if caps is None else min(STEPS, int(caps[u]))
            want = cap if ignore_gate else _stop_frames(sgate[r].cpu(), cap, dec.gate_threshold)
            assert n == want, (u, n, want)
            assert torch.equal(mel, smel[r, :, :n]), ("mel", u)
            assert torch.equal(gate, sgate[r, :n]), ("gate", u)
            if align is not None:
                assert torch.equal(align, salign[r, :n]), ("align", u)


def _spread_caps(U, seed):
    return torch.from_numpy((1 + np.floor(synth.uniform01(seed, 1, U) * STEPS)).astype(np.int32))


def _staggered(U, S, chunk=7):
    """busy slots, then some idle, then fully idle, then the rest"""
    a, b, c = S + 2, S + 2 + S // 2 + 1, 2 * S + 4
    return [("submit", 0, a), ("step", chunk), ("submit", a, b), ("step", chunk), ("step", chunk), ("submit", b, c),
            ("drain", chunk), ("submit", c, U), ("drain", chunk)]


# --------------------------------------------------------------------------- 1. the same queue gives the same result
@pytest.mark.parametrize("precision,row_offset", [("fp32", 0), ("bf16", 0), ("fp32", 37), ("bf16", 37)])
def test_whole_queue_up_front_equals_inference_continuous(cuda_device, precision, row_offset):
    dec, _ = _decoder(cuda_device, precision)
    memory, lens = _queue(cuda_device, 23, 64)
    caps = torch.full((23,), STEPS, dtype=torch.int32)
    caps[[1, 4, 8, 13, 20]] = torch.tensor([5, 9, 2, 17, 11], dtype=torch.int32)
    (mel, gate, align), nf = _continuous(dec, memory, lens, 4, caps, row_offset=row_offset)
    for chunk in (1, 7, 16, 64):
        sess = _session(dec, 64, 4, capacity=32, row_offset=row_offset)
        out = _drive(sess, memory, lens, caps, [("submit", 0, 23), ("drain", chunk)])
        assert sess.steps_run == dec.last_steps_run or chunk != 16, (chunk, sess.steps_run, dec.last_steps_run)
        for u in range(23):
            m, g, a, n = out[u]
            assert n == int(nf[u]), (chunk, u, n, int(nf[u]))
            assert torch.equal(m, mel[u, :, :n]) and torch.equal(g, gate[u, :n]) and torch.equal(a, align[u, :n]), (chunk, u)


# --------------------------------------------------------------------------- 2. staggered submission
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_staggered_submission_is_bit_exact_against_static(cuda_device, precision):
    dec, _ = _decoder(cuda_device, precision)
    memory, lens = _queue(cuda_device, 23, 64)
    caps = _spread_caps(23, 31)
    sess = _session(dec, 64, 4, row_offset=3)
    out = _drive(sess, memory, lens, caps, _staggered(23, 4))
    assert len({o[3] for o in out.values()}) >= 4                 # stops really are spread: slots refill at different steps
    _check_static(dec, memory, lens, 4, out, caps, row_offset=3)
    assert sess.active == 0 and sess.pending == 0 and sess.idle == 4


def test_partial_chunks_are_prefixes(cuda_device):
    dec, _ = _decoder(cuda_device, "fp32")
    memory, lens = _queue(cuda_device, 9, 64)
    caps = _spread_caps(9, 41)
    sess = _session(dec, 64, 4)
    sess.submit(memory[:6], lens[:6], caps[:6])
    seen, late = {}, False
    while sess.active or sess.pending or not late:
        chunks, _ = sess.step(3)
        for i, (m, g, a) in chunks.items():
            seen[i] = torch.cat([seen[i], m], dim=1) if i in seen else m
            assert m.shape[1] <= 3
        if not late and (sess.steps_run >= 6 or not (sess.active or sess.pending)):
            sess.submit(memory[6:], lens[6:], caps[6:])
            late = True
    smel, _, _ = _static(dec, memory, lens, 0, 4)
    for r in range(4):
        assert torch.equal(seen[r], smel[r, :, :seen[r].shape[1]])


# --------------------------------------------------------------------------- 3. / 4. other kernels of the step
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_reference_dims(cuda_device, precision):
    """the two-CTA cluster attention kernel reads lengths and prefetches processed memory before it waits"""
    dims = synth.DecoderDims()
    dec, _ = _decoder(cuda_device, precision, dims, gate_bias=-0.2)
    memory, lens = _queue(cuda_device, 10, 64, dims)
    caps = torch.tensor([3, 7, 1, 12, 5, 9, 2, 16, 4, 11], dtype=torch.int32)
    sess = _session(dec, 64, 4, row_offset=5)
    out = _drive(sess, memory, lens, caps, [("submit", 0, 5), ("step", 4), ("submit", 5, 8), ("drain", 16), ("submit", 8, 10),
                                            ("drain", 5)])
    _check_static(dec, memory, lens, 4, out, caps, row_offset=5)


def test_many_slots_take_the_unfused_prenet(cuda_device):
    dec, _ = _decoder(cuda_device, "fp32")
    memory, lens = _queue(cuda_device, 150, 32, seed=9)
    caps = _spread_caps(150, 12)
    sess = _session(dec, 32, 72, capacity=160)
    out = _drive(sess, memory, lens, caps, [("submit", 0, 80), ("step", 5), ("submit", 80, 150), ("drain", 16)])
    _check_static(dec, memory, lens, 72, out, caps)


# --------------------------------------------------------------------------- 5. ring wrap-around
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_ring_wraps_around(cuda_device, precision):
    dec, _ = _decoder(cuda_device, precision)
    S, cap, U = 4, 8, 30
    memory, lens = _queue(cuda_device, U, 64, seed=17)
    caps = _spread_caps(U, 23)
    sess = _session(dec, 64, S, capacity=cap)
    sess.submit(memory[:cap], lens[:cap], caps[:cap])
    with pytest.raises(RuntimeError, match="ring is full"):
        sess.submit(memory[cap:cap + 1], lens[cap:cap + 1], caps[cap:cap + 1])
    parts, fin, nxt = {}, {}, cap
    while len(fin) < U:
        chunks, done = sess.step(5)
        for i, c in chunks.items():
            parts.setdefault(i, []).append(c)
        fin.update(done)
        room = cap - sess.pending
        if nxt < U and room > 0:                                       # the session is still usable after the refusal
            hi = min(U, nxt + room)
            assert sess.submit(memory[nxt:hi], lens[nxt:hi], caps[nxt:hi]) == list(range(nxt, hi))
            nxt = hi
    _sync()
    out = {i: (torch.cat([p[0] for p in ps], 1), torch.cat([p[1] for p in ps]), torch.cat([p[2] for p in ps]), fin[i])
           for i, ps in parts.items()}
    _check_static(dec, memory, lens, S, out, caps)


# --------------------------------------------------------------------------- 6. an admission at every step
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_admission_at_every_step(cuda_device, precision):
    dec, _ = _decoder(cuda_device, precision)
    memory, lens = _queue(cuda_device, 23, 64)
    ones = torch.ones(23, dtype=torch.int32)
    out = _drive(_session(dec, 64, 4), memory, lens, ones, [("submit", 0, 10), ("step", 2), ("submit", 10, 23), ("drain", 3)])
    assert [out[u][3] for u in range(23)] == [1] * 23
    _check_static(dec, memory, lens, 4, out, ones)
    dec.gate_layer.linear_layer.bias.data.fill_(30.0)                 # the gate fires at frame 1 of every utterance
    dec.invalidate_packed()
    out = _drive(_session(dec, 64, 4), memory, lens, None, [("submit", 0, 23), ("drain", 7)])
    assert [out[u][3] for u in range(23)] == [1] * 23
    _check_static(dec, memory, lens, 4, out)


# --------------------------------------------------------------------------- 7. against the oracle (fp32)
def test_matches_oracle_fp32(cuda_device):
    dec, W = _decoder(cuda_device, "fp32")
    memory, lens = _queue(cuda_device, 23, 64)
    out = _drive(_session(dec, 64, 4), memory, lens, None, [("submit", 0, 12), ("step", 9), ("submit", 12, 23), ("drain", 16)])
    P = O.as_params(W)
    for u in (0, 5, 11, 22):
        rm, rg, ra, rn = O.inference(P, memory[u:u + 1].cpu(), lens[u:u + 1].cpu(), STEPS, dec.gate_threshold, False, SEED,
                                     False, dec.p_attention_dropout, dec.p_decoder_dropout, row_offset=u)
        mel, gate, align, n = out[u]
        assert n == int(rn[0]), (u, n, int(rn[0]))
        scale = float(rm.abs().max())
        assert float((mel.cpu() - rm[0, :, :n]).abs().max()) <= 1e-4 * scale, u
        assert float((gate.cpu() - rg[0, :n]).abs().max()) <= 1e-4 * max(float(rg.abs().max()), 1e-30), u
        ok, _ = argmax_agrees(align.cpu().numpy(), ra[0, :n].numpy())
        assert ok, u


# --------------------------------------------------------------------------- 8. launch budget
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_launches_per_step_equal_static(cuda_device, precision):
    lib = _native.load()
    dec, _ = _decoder(cuda_device, precision, gate_bias=-30.0)     # the gate never fires: the static run takes every step
    memory, lens = _queue(cuda_device, 8, 64)

    def launches(fn):
        _sync()
        c0 = lib.gvx_launch_count()
        fn()
        _sync()
        return lib.gvx_launch_count() - c0

    def static(steps):
        return launches(lambda: dec.inference(memory[:4], memory_lengths=lens[:4], max_decoder_steps=steps))

    static(10)                                                      # warm (weight packing)
    per_static = (static(20) - static(10)) / 10
    sess = _session(dec, 64, 4)
    sess.submit(memory, lens)
    for k in (16, 5):                                               # every slot busy throughout both calls
        n = launches(lambda: sess.step(k))
        assert n == k * per_static + 1, (k, n, per_static)           # + the head-of-call admission


# --------------------------------------------------------------------------- 9. refusals, and an idle session
def test_refusals_and_idle_session(cuda_device):
    lib = _native.load()
    dec, _ = _decoder(cuda_device, "fp32")
    memory, lens = _queue(cuda_device, 6, 64)
    sess = _session(dec, 64, 4)
    c0 = lib.gvx_launch_count()
    assert sess.step(16) == ({}, {}) and sess.steps_run == 0
    assert lib.gvx_launch_count() == c0                              # nothing queued, nothing running: nothing launched
    with pytest.raises(ValueError, match="wider"):
        sess.submit(torch.zeros(1, 65, memory.shape[2], device=cuda_device), None)
    with pytest.raises(ValueError, match="frame_caps"):
        sess.submit(memory[:2], lens[:2], [0, 5])
    with pytest.raises(ValueError, match="frame_caps"):
        sess.submit(memory[:2], lens[:2], [5, STEPS + 1])
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        sess.submit(memory[:2].cpu(), lens[:2])
    narrow = memory[:2, :40].contiguous()                           # zero-padded to N by submit
    assert sess.submit(narrow, torch.clamp(lens[:2], max=40)) == [0, 1]
    sess.step(4)
    with torch.no_grad():
        dec.prenet.layers[0].linear_layer.weight.mul_(1.0)           # a parameter update (its version counter moves)
    with pytest.raises(RuntimeError, match="changed"):
        sess.step(4)
    with pytest.raises(RuntimeError, match="changed"):
        sess.submit(memory[2:3], lens[2:3])
    sess2 = _session(dec, 64, 4)
    dec.precision = "bf16"
    with pytest.raises(RuntimeError, match="changed"):
        sess2.step(4)
    dec.precision = "fp32"
    dec.train()
    with pytest.raises(RuntimeError, match="changed"):
        sess2.step(4)
    dec.eval()
    sess2.submit(memory[:1], lens[:1])
    chunks, done = sess2.step(STEPS)
    assert sorted(chunks) == [0] and 0 in done
    _sync()
    c0 = lib.gvx_launch_count()
    assert sess2.step(8) == ({}, {}) and lib.gvx_launch_count() == c0     # drained: idle and empty again


# --------------------------------------------------------------------------- 10. synthesis
def test_synthesis_session_equals_continuous_inference(cuda_device):
    m = _model(cuda_device, max_steps=24)
    g = torch.Generator().manual_seed(5)
    rows = [torch.randint(0, 40, (n,), generator=g).tolist() for n in (37, 9, 64, 23, 50, 12, 64)]
    m.decoder.gate_layer.linear_layer.bias.data.fill_(-0.2)
    m.decoder._next_seed = lambda: 1234
    cont = synthesis.continuous_inference(m, rows, slots=3)
    ss = synthesis.SynthesisSession(m, 64, slots=3)
    got, partial = {}, {}
    assert ss.submit(rows[:4]) == [0, 1, 2, 3]
    for call in range(100):
        chunks, done = ss.step(5)
        for i, c in chunks.items():
            partial[i] = torch.cat([partial[i], c], dim=2) if i in partial else c
        got.update(done)
        if call == 1:
            assert ss.submit(rows[4:]) == [4, 5, 6]
        if len(got) == len(rows):
            break
    _sync()
    for i, want in enumerate(cont):
        assert torch.equal(partial[i], want["mel_outputs"]), i
        for k, v in want.items():
            assert torch.equal(got[i][k], v), (i, k)
