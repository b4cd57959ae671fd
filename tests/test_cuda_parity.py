"""GPU parity tests: the CUDA path (through the C ABI, via genvox_b200.Decoder / ctypes) against
  * the committed golden outputs of the UNMODIFIED reference (tests/golden/, fp64 run = yardstick),
  * the CPU oracle (oracle/decoder_oracle.py) on the same seeded inputs,
  * size-independent properties at BASELINE.json's full sizes.

Tolerances (north_star): mel / gate / alignments within 1e-4 of max|ref| in fp32; alignment argmax
and stop steps exact (tie-aware: wherever the fp64 reference's top-2 margin exceeds 1e-5).
Gradients: 2e-4 of max|ref| per tensor.
"""
import ctypes as C

import numpy as np
import pytest
import torch

from conftest import golden_tags, load_golden, rel_err
from oracle import decoder_oracle as O
from oracle import philox, synth

pytestmark = pytest.mark.gpu

FWD_TOL = 1e-4
GRAD_TOL = 2e-4


def _tol(z, key, base):
    k32, k64 = key.replace("{p}", "f32"), key.replace("{p}", "f64")
    return max(base, 4.0 * rel_err(z[k32], z[k64]))


def make_decoder(dims, W, device, training):
    import genvox_b200
    dec = genvox_b200.Decoder(**dims.kwargs())
    dec.load_state_dict({k: torch.from_numpy(np.ascontiguousarray(v)) for k, v in W.items()}, strict=True)
    return dec.to(device).train(training)


def argmax_agrees(align, ref64, margin=1e-5):
    """argmax equal wherever the reference's top-1/top-2 gap is above `margin` (relative to the max)."""
    ref64 = np.asarray(ref64, dtype=np.float64)
    srt = np.sort(ref64, axis=-1)
    clear = (srt[..., -1] - srt[..., -2]) > margin * srt[..., -1] if ref64.shape[-1] > 1 else np.ones(ref64.shape[:-1], bool)
    same = np.asarray(align).argmax(-1) == ref64.argmax(-1)
    return bool(same[clear].all()), float(clear.mean())


# --------------------------------------------------------------------------- library / device
def test_library_runs_on_sm100(cuda_device):
    from genvox_b200 import _native
    lib = _native.load()
    sm, major, minor = C.c_int(), C.c_int(), C.c_int()
    _native.check(lib.gvx_device_info(C.byref(sm), C.byref(major), C.byref(minor)), "gvx_device_info")
    assert major.value == 10, f"built for sm_100a, device is sm_{major.value}{minor.value}"
    assert sm.value >= 100


# --------------------------------------------------------------------------- single phases
def _native_bits(dec):
    from genvox_b200 import _native
    params = [p.detach() for p in dec._ordered_params()]
    dims, weights, packed = dec._native_state(params)
    return _native.load(), dims, weights, packed, params


@pytest.mark.parametrize("B,F", [(5, 3), (64, 2), (1, 4)])
def test_phase_prenet(cuda_device, B, F):
    from genvox_b200 import _native
    from genvox_b200.decoder import _ptr, _stream
    dims = synth.DecoderDims()
    W = synth.make_decoder_weights(3, dims)
    dec = make_decoder(dims, W, cuda_device, True)
    lib, gd, gw, packed, _ = _native_bits(dec)
    frames = (synth.uniform01(5, 1, F * B * dims.n_mels).astype(np.float32) - 0.5).reshape(F, B, dims.n_mels) * 4
    x = torch.from_numpy(frames).to(cuda_device)
    tmp = torch.empty(F, B, dims.prenet_dim, device=cuda_device)
    out = torch.empty(F, B, dims.prenet_dim, device=cuda_device)
    _native.check(lib.gvx_prenet_fwd(C.byref(gd), C.byref(gw), _ptr(x), F, B, 77, 5, 2, _ptr(tmp), _ptr(out), _stream()),
                  "gvx_prenet_fwd")
    ref = O.prenet(O.as_params(W), torch.from_numpy(frames), 77, t0=5, row_offset=2)
    assert rel_err(out.cpu(), ref) < 1e-5
    assert float((out == 0).float().mean()) > 0.5          # dropout p=.5 after ReLU is really on


@pytest.mark.parametrize("which,B,training", [(0, 64, True), (1, 64, True), (0, 3, False), (1, 17, True)])
def test_phase_lstm_cell(cuda_device, which, B, training):
    from genvox_b200 import _native
    from genvox_b200.decoder import _ptr, _stream
    dims = synth.DecoderDims()
    W = synth.make_decoder_weights(4, dims)
    dec = make_decoder(dims, W, cuda_device, training)
    lib, gd, gw, packed, _ = _native_bits(dec)
    hid = dims.attention_rnn_dim if which == 0 else dims.decoder_rnn_dim
    nin = (dims.prenet_dim if which == 0 else dims.attention_rnn_dim) + dims.encoder_embedding_dim
    u = lambda s, n: (synth.uniform01(9, s, n).astype(np.float32) - 0.5) * 2
    x, h, c = u(1, B * nin).reshape(B, nin), u(2, B * hid).reshape(B, hid), u(3, B * hid).reshape(B, hid)
    dx, dh, dc = (torch.from_numpy(a).to(cuda_device) for a in (x, h, c))
    h_out, c_out = torch.empty(B, hid, device=cuda_device), torch.empty(B, hid, device=cuda_device)
    gates = torch.empty(B, 4 * hid, device=cuda_device)
    _native.check(lib.gvx_lstm_step(C.byref(gd), _ptr(packed), which, _ptr(dx), _ptr(dh), _ptr(dc), B, 1234, 7,
                                    int(training), 3, _ptr(h_out), _ptr(c_out), _ptr(gates), _stream()), "gvx_lstm_step")
    P = O.as_params(W)
    pre = "attention_rnn" if which == 0 else "decoder_rnn"
    rh, rc = O.lstm_cell(torch.from_numpy(x), torch.from_numpy(h), torch.from_numpy(c), P[f"{pre}.weight_ih"],
                         P[f"{pre}.weight_hh"], P[f"{pre}.bias_ih"], P[f"{pre}.bias_hh"])
    p = dims.p_attention_dropout if which == 0 else dims.p_decoder_dropout
    rh = O.philox_dropout(rh, p, training, 1234, philox.SITE_ATT if which == 0 else philox.SITE_DEC, 7, row_offset=3)
    assert rel_err(c_out.cpu(), rc) < 1e-5
    assert rel_err(h_out.cpu(), rh) < 1e-5
    # packed gate activations: [b, 4*unit + (i,f,g,o)]; o * tanh(c') must reproduce the undropped h
    g = gates.cpu().view(B, hid, 4)
    assert rel_err(g[:, :, 3] * torch.tanh(c_out.cpu()), O.lstm_cell(
        torch.from_numpy(x), torch.from_numpy(h), torch.from_numpy(c), P[f"{pre}.weight_ih"], P[f"{pre}.weight_hh"],
        P[f"{pre}.bias_ih"], P[f"{pre}.bias_hh"])[0]) < 1e-5


@pytest.mark.parametrize("B,N,masked", [(4, 37, True), (64, 150, False), (2, 300, True)])
def test_phase_attention(cuda_device, B, N, masked):
    from genvox_b200 import _native
    from genvox_b200.decoder import _ptr, _stream
    dims = synth.DecoderDims()
    W = synth.make_decoder_weights(5, dims)
    dec = make_decoder(dims, W, cuda_device, False)
    lib, gd, gw, packed, _ = _native_bits(dec)
    mem, _, lens = synth.make_inputs(21, B, N, 0, dims, ragged=masked)
    P = O.as_params(W)
    memory = torch.from_numpy(mem)
    pm = torch.nn.functional.linear(memory, P["attention_layer.memory_layer.linear_layer.weight"])
    h = torch.from_numpy((synth.uniform01(22, 1, B * dims.attention_rnn_dim).astype(np.float32) - 0.5).reshape(B, -1))
    # a plausible previous state: normalised weights over the valid tokens, two steps of cumulation
    wp = torch.from_numpy(synth.uniform01(22, 2, B * N).astype(np.float32).reshape(B, N))
    mask = O.get_mask_from_lengths(torch.from_numpy(lens), N) if masked else None
    if masked:
        wp = wp.masked_fill(mask, 0.0)
    wp = wp / wp.sum(1, keepdim=True)
    cum = 2.0 * wp.flip(1) + wp
    ref_ctx, ref_w = O.attention(P, h, memory, pm, wp, cum, mask)
    d = lambda t: t.contiguous().to(cuda_device)
    dwp, dcum = d(wp.clone()), d(cum.clone())
    q = torch.empty(B, dims.attention_dim, device=cuda_device)
    ctx = torch.empty(B, dims.encoder_embedding_dim, device=cuda_device)
    al = torch.empty(B, N, device=cuda_device)
    dl = torch.from_numpy(lens).to(cuda_device) if masked else None
    dh, dmem, dpm = d(h), d(memory), d(pm)       # keep the device tensors alive across the call
    _native.check(lib.gvx_attention_step(C.byref(gd), C.byref(gw), _ptr(packed), _ptr(dh), _ptr(dmem), _ptr(dpm),
                                         _ptr(dl), B, N, _ptr(dwp), _ptr(dcum), _ptr(q), _ptr(ctx), _ptr(al), _stream()),
                  "gvx_attention_step")
    assert rel_err(al.cpu(), ref_w) < 2e-5
    assert rel_err(ctx.cpu(), ref_ctx) < 2e-5
    assert torch.equal(dwp.cpu(), al.cpu())                                # w_prev <- w          (tacotron2.py:345-352)
    assert rel_err(dcum.cpu(), cum + ref_w) < 2e-6                         # cum += w             (tacotron2.py:353)
    if masked:
        for b, L in enumerate(lens):
            assert float(al[b, L:].abs().max().cpu()) == 0.0 if L < N else True


# --------------------------------------------------------------------------- golden: teacher forcing + BPTT
@pytest.mark.parametrize("tag", golden_tags("forward"))
def test_forward_and_bptt_match_reference_golden(cuda_device, tag):
    meta, z = load_golden(tag)
    dims = synth.DecoderDims(**meta["dims"])
    W = synth.make_decoder_weights(meta["weight_seed"], dims, meta["weight_scale"])
    B, N, T = meta["B"], meta["N"], meta["T"]
    mem, mel, lens = synth.make_inputs(meta["input_seed"], B, N, T, dims)
    dec = make_decoder(dims, W, cuda_device, meta["training"])
    memory = torch.from_numpy(mem).to(cuda_device).requires_grad_(meta["with_grads"])
    dec.set_dropout_seed(meta["dropout_seed"])
    m, g, a = dec(memory, torch.from_numpy(mel).to(cuda_device), torch.from_numpy(lens).to(cuda_device))
    assert m.shape == (B, dims.n_mels, T) and g.shape == (B, T) and a.shape == (B, T, N)
    fr = meta.get("frames")         # long fixtures keep selected frames only (oracle/make_golden.py: keep_frames_of)
    ms, gs, as_ = (m, g, a) if fr is None else (m[:, :, fr], g[:, fr], a[:, fr])
    errs = {k: rel_err(v.detach().cpu(), z[f"{k}_f64"]) for k, v in (("mel", ms), ("gate", gs), ("align", as_))}
    print(tag, "forward rel err vs fp64 reference:", errs)
    for k, e in errs.items():
        assert e < _tol(z, k + "_{p}", FWD_TOL), (k, e)
    ok, frac = argmax_agrees(as_.detach().cpu().numpy(), z["align_f64"])
    assert ok, "alignment argmax differs from the reference where its margin is clear"
    for b, L in enumerate(lens):                        # padded tokens: exactly zero weight (tacotron2.py:125)
        if L < N:
            assert float(a[b, :, L:].abs().max().cpu()) == 0.0
    if not meta["with_grads"]:
        return
    r_mel = (synth.uniform01(meta["input_seed"], 20, B * dims.n_mels * T) - 0.5).astype(np.float32).reshape(B, dims.n_mels, T)
    r_gate = (synth.uniform01(meta["input_seed"], 21, B * T) - 0.5).astype(np.float32).reshape(B, T)
    loss = (m * torch.from_numpy(r_mel).to(cuda_device)).sum() + (g * torch.from_numpy(r_gate).to(cuda_device)).sum()
    loss.backward()
    grads = {k: p.grad.cpu().numpy() for k, p in dec.named_parameters()}
    grads["memory"] = memory.grad.cpu().numpy()
    worst = {}
    for name, gr in grads.items():
        pre = f"grad_f64|{name}"
        which = "full" if f"{pre}|full" in z else "vals"
        gtol = _tol(z, "grad_{p}|" + name + "|" + which, GRAD_TOL)
        ref = z[f"{pre}|{which}"]
        got = gr if which == "full" else gr.reshape(-1)[z[f"{pre}|idx"]]     # a fixed sample of positions
        err = float(np.abs(got - ref).max() / max(np.abs(ref).max(), 1e-30))
        worst[name] = err
        assert err <= gtol, (name, err, gtol)
        l2 = float(z[f"{pre}|l2"])
        assert abs(np.sqrt((gr.astype(np.float64) ** 2).sum()) - l2) <= 10 * gtol * max(l2, 1e-30), name
        if f"{pre}|colsum" in z:
            cs = z[f"{pre}|colsum"]
            assert np.abs(gr.astype(np.float64).sum(0) - cs).max() <= 20 * gtol * max(np.abs(cs).max(), 1e-30), name
    print(tag, "worst grad rel err:", max(worst.items(), key=lambda kv: kv[1]))


# --------------------------------------------------------------------------- golden: inference
@pytest.mark.parametrize("tag", golden_tags("decode_loop"))
def test_batched_inference_matches_reference_decode_loop(cuda_device, tag):
    meta, z = load_golden(tag)
    dims = synth.DecoderDims(**meta["dims"])
    W = synth.make_decoder_weights(meta["weight_seed"], dims, meta["weight_scale"])
    mem, _, lens = synth.make_inputs(meta["input_seed"], meta["B"], meta["N"], 0, dims)
    dec = make_decoder(dims, W, cuda_device, False)
    dec.set_dropout_seed(meta["dropout_seed"])
    m, g, a = dec.inference(torch.from_numpy(mem).to(cuda_device),
                            memory_lengths=torch.from_numpy(lens).to(cuda_device) if meta["masked"] else None,
                            ignore_gate=True, max_decoder_steps=meta["steps"])
    assert m.shape[2] == meta["steps"] and dec.last_n_frames.tolist() == [meta["steps"]] * meta["B"]
    for k, v in (("mel", m), ("gate", g), ("align", a)):
        e = rel_err(v.cpu(), z[f"{k}_f64"])
        assert e < _tol(z, k + "_{p}", FWD_TOL), (k, e)
    ok, _ = argmax_agrees(a.cpu().numpy(), z["align_f64"])
    assert ok


@pytest.mark.parametrize("tag", golden_tags("decode_stops"))
def test_batched_inference_rows_stop_at_different_steps(cuda_device, tag):
    """Per-row stop rule (tacotron2.py:405 / :407) on a batch whose rows fire at different steps: `last_n_frames` exact,
    every row's frames up to its own stop step equal to the reference's."""
    meta, z = load_golden(tag)
    dims = synth.DecoderDims(**{**meta["dims"], "gate_threshold": meta["gate_threshold"], "max_decoder_steps": meta["steps"]})
    W = synth.make_decoder_weights(meta["weight_seed"], dims, meta["weight_scale"])
    mem, _, lens = synth.make_inputs(meta["input_seed"], meta["B"], meta["N"], 0, dims)
    nf = meta["n_frames"]
    assert len(set(nf)) >= 3 and max(nf) == meta["steps"]
    for precision in ("fp32", "bf16"):
        dec = make_decoder(dims, W, cuda_device, False)
        dec.precision = precision
        dec.set_dropout_seed(meta["dropout_seed"])
        m, g, a = dec.inference(torch.from_numpy(mem).to(cuda_device), memory_lengths=torch.from_numpy(lens).to(cuda_device))
        if precision == "fp32":
            assert dec.last_n_frames.tolist() == nf                                  # stop steps exact
        assert m.shape[2] == max(dec.last_n_frames.tolist())
        tol = FWD_TOL if precision == "fp32" else 3e-2
        for b, n in enumerate(nf if precision == "fp32" else dec.last_n_frames.tolist()):
            n = min(n, nf[b])
            for k, v in (("mel", m[b, :, :n]), ("gate", g[b, :n]), ("align", a[b, :n])):
                ref = z[f"{k}_f64"][b][..., :n] if k != "align" else z["align_f64"][b, :n]
                e = float(np.abs(v.cpu().numpy() - ref).max() / max(np.abs(z[f"{k}_f64"]).max(), 1e-30))
                assert e < max(tol, _tol(z, k + "_{p}", tol)), (precision, b, k, e)


@pytest.mark.parametrize("tag", golden_tags("public_inference"))
def test_gate_stopped_inference_matches_reference_public_api(cuda_device, tag, capsys):
    meta, z = load_golden(tag)
    dims = synth.DecoderDims(**meta["dims"])
    W = synth.make_decoder_weights(meta["weight_seed"], dims, meta["weight_scale"])
    mem, _, _ = synth.make_inputs(meta["input_seed"], 1, meta["N"], 0, dims, ragged=False)
    dec = make_decoder(dims, W, cuda_device, False)
    dec.set_dropout_seed(meta["dropout_seed"])
    m, g, a = dec.inference(torch.from_numpy(mem).to(cuda_device))
    assert dec.last_n_frames.tolist() == [meta["n_frames"]]           # stop step exact (tacotron2.py:405)
    assert m.shape == (1, dims.n_mels, meta["n_frames"])
    for k, v in (("mel", m), ("gate", g), ("align", a)):
        e = rel_err(v.cpu(), z[f"{k}_f64"])
        assert e < _tol(z, k + "_{p}", FWD_TOL), (k, e)
    assert "max decoder steps" not in capsys.readouterr().out


def test_max_decoder_steps_guard_prints_the_reference_warning(cuda_device, capsys):
    dims = synth.DecoderDims(max_decoder_steps=5, gate_threshold=0.999999)
    W = synth.make_decoder_weights(7, dims)
    mem, _, _ = synth.make_inputs(3, 2, 11, 0, dims, ragged=False)
    dec = make_decoder(dims, W, cuda_device, False)
    m, g, a = dec.inference(torch.from_numpy(mem).to(cuda_device))
    assert m.shape[2] == 5 and dec.last_n_frames.tolist() == [5, 5]
    assert "Reached max decoder steps" in capsys.readouterr().out       # tacotron2.py:408


def test_invalidate_packed_after_data_edit(cuda_device):
    """In-place edits through `.data` do not bump autograd's version counter: `invalidate_packed()` is the documented way to make
    the kernels see them; ordinary optimizer steps / `copy_` on the parameter itself are picked up without it."""
    dims = synth.DecoderDims(max_decoder_steps=4, gate_threshold=0.999999)
    W = synth.make_decoder_weights(7, dims)
    mem, _, _ = synth.make_inputs(3, 2, 11, 0, dims, ragged=False)
    dec = make_decoder(dims, W, cuda_device, False)
    x = torch.from_numpy(mem).to(cuda_device)
    dec.set_dropout_seed(5)
    m0 = dec.inference(x, ignore_gate=True)[0].clone()
    dec.linear_projection.linear_layer.weight.data.mul_(2.0)
    dec.invalidate_packed()
    dec.set_dropout_seed(5)
    m1 = dec.inference(x, ignore_gate=True)[0].clone()
    assert not torch.allclose(m0[:, :, 0], m1[:, :, 0])
    with torch.no_grad():
        dec.linear_projection.linear_layer.weight.mul_(0.5)          # versioned edit: no explicit invalidation needed
    dec.set_dropout_seed(5)
    m2 = dec.inference(x, ignore_gate=True)[0]
    assert torch.allclose(m0[:, :, 0], m2[:, :, 0], rtol=1e-5, atol=1e-6)


# --------------------------------------------------------------------------- oracle at config-1 batch shape
def test_forward_backward_match_oracle_config1_shape(cuda_device):
    """B=16, N=120 (config 1's batch/token shape), T=24 frames, ragged lengths, training mode."""
    dims = synth.DecoderDims()
    B, N, T, seed = 16, 120, 24, 4242
    W = synth.make_decoder_weights(11, dims)
    mem, mel, lens = synth.make_inputs(31, B, N, T, dims)
    u = lambda s, shape: torch.from_numpy((synth.uniform01(31, s, int(np.prod(shape))) - 0.5).astype(np.float32).reshape(shape))
    r_mel, r_gate, r_align = u(20, (B, dims.n_mels, T)), u(21, (B, T)), u(22, (B, T, N))
    torch.set_num_threads(max(1, torch.get_num_threads()))
    (om, og, oa), ograds, omem = O.loss_and_grads(O.as_params(W), torch.from_numpy(mem), torch.from_numpy(mel), lens,
                                                  r_mel, r_gate, seed, True, dims.p_attention_dropout,
                                                  dims.p_decoder_dropout, r_align=r_align)
    dec = make_decoder(dims, W, cuda_device, True)
    memory = torch.from_numpy(mem).to(cuda_device).requires_grad_(True)
    dec.set_dropout_seed(seed)
    m, g, a = dec(memory, torch.from_numpy(mel).to(cuda_device), torch.from_numpy(lens).to(cuda_device))
    assert rel_err(m.detach().cpu(), om) < FWD_TOL
    assert rel_err(g.detach().cpu(), og) < FWD_TOL
    assert rel_err(a.detach().cpu(), oa) < FWD_TOL
    assert argmax_agrees(a.detach().cpu().numpy(), oa.numpy())[0]
    dv = lambda t: t.to(cuda_device)
    ((m * dv(r_mel)).sum() + (g * dv(r_gate)).sum() + (a * dv(r_align)).sum()).backward()
    worst = ("", 0.0)
    for k, p in dec.named_parameters():
        e = rel_err(p.grad.cpu(), ograds[k])
        worst = max(worst, (k, e), key=lambda kv: kv[1])
        assert e < GRAD_TOL, (k, e)
    e = rel_err(memory.grad.cpu(), omem)
    assert e < GRAD_TOL, ("memory", e)
    print("worst grad rel err vs oracle:", worst, "memory:", e)


# --------------------------------------------------------------------------- properties at full size
def test_inference_full_size_properties(cuda_device):
    """BASELINE config 2 shape: B=64, N=150, fixed steps (gate ignored).  Deterministic, prefix-stable,
    alignments are distributions, no NaN."""
    dims = synth.DecoderDims()
    W = synth.make_decoder_weights(7, dims)
    mem, _, _ = synth.make_inputs(41, 64, 150, 0, dims, ragged=False)
    dec = make_decoder(dims, W, cuda_device, False)
    memory = torch.from_numpy(mem).to(cuda_device)
    outs = []
    for steps in (200, 200, 50):
        dec.set_dropout_seed(99)
        outs.append([t.clone() for t in dec.inference(memory, ignore_gate=True, max_decoder_steps=steps)])
    for x, y in zip(outs[0], outs[1]):
        assert torch.equal(x, y)                                     # run-to-run bit-exact
    assert torch.equal(outs[0][0][:, :, :50], outs[2][0]) and torch.equal(outs[0][2][:, :50], outs[2][2])
    m, g, a = outs[0]
    assert bool(torch.isfinite(m).all()) and bool(torch.isfinite(g).all())
    assert float((a.sum(-1) - 1).abs().max().cpu()) < 1e-5 and float(a.min().cpu()) >= 0.0


def test_backward_is_linear_in_upstream_gradient(cuda_device):
    """BPTT is a linear map of (d_mel, d_gate): grads(2 r) == 2 grads(r), grads(r1 + r2) == grads(r1) + grads(r2)."""
    dims = synth.DecoderDims()
    B, N, T = 8, 50, 12
    W = synth.make_decoder_weights(13, dims)
    mem, mel, lens = synth.make_inputs(51, B, N, T, dims)
    dec = make_decoder(dims, W, cuda_device, True)
    u = lambda s, shape: torch.from_numpy((synth.uniform01(51, s, int(np.prod(shape))) - 0.5).astype(np.float32).reshape(shape)).to(cuda_device)
    r1, r2, q1, q2 = u(1, (B, dims.n_mels, T)), u(2, (B, dims.n_mels, T)), u(3, (B, T)), u(4, (B, T))

    def grads(rm, rg):
        dec.zero_grad(set_to_none=True)
        memory = torch.from_numpy(mem).to(cuda_device).requires_grad_(True)
        dec.set_dropout_seed(5)
        m, g, _ = dec(memory, torch.from_numpy(mel).to(cuda_device), torch.from_numpy(lens).to(cuda_device))
        ((m * rm).sum() + (g * rg).sum()).backward()
        return torch.cat([p.grad.flatten() for p in dec.parameters()] + [memory.grad.flatten()])

    ga, gb, gab, g2a = grads(r1, q1), grads(r2, q2), grads(r1 + r2, q1 + q2), grads(2 * r1, 2 * q1)
    scale = float(gab.abs().max().cpu())
    assert float((gab - (ga + gb)).abs().max().cpu()) < 1e-4 * scale
    assert float((g2a - 2 * ga).abs().max().cpu()) < 1e-5 * scale
