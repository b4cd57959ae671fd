"""Pin the CPU oracle (oracle/decoder_oracle.py) to outputs of the UNMODIFIED reference.

The fixtures under tests/golden/ were produced by oracle/make_golden.py from the reference's
own Decoder (tacotron2.py:258-414) in fp32 and fp64.  fp32 tolerance: 2e-6 of max|ref| (the
oracle runs the same torch CPU ops, only op fusion differs); the fp64 run bounds how far
either fp32 result is from exact arithmetic.
"""
import numpy as np
import pytest
import torch

from conftest import golden_tags, load_golden, rel_err
from oracle import decoder_oracle as O
from oracle import synth

F32_TOL = 2e-6
F64_TOL = 1e-12


def tol_of(z, key, prec, base):
    """fp32: the larger of `base` and 4x the reference's own fp32-vs-fp64 distance on this
    quantity (an ill-conditioned case — the weight_scale=3 fixtures — has a higher floor)."""
    if prec == "f64":
        return base
    k32, k64 = key.replace("{p}", "f32"), key.replace("{p}", "f64")
    return max(base, 4.0 * rel_err(z[k32], z[k64]))


def _setup(meta, dtype):
    dims = synth.DecoderDims(**meta["dims"])
    W = synth.make_decoder_weights(meta["weight_seed"], dims, meta["weight_scale"])
    return dims, O.as_params(W, dtype)


@pytest.mark.parametrize("tag", golden_tags("forward"))
@pytest.mark.parametrize("prec", ["f32", "f64"])
def test_forward_and_bptt_match_reference(tag, prec):
    meta, z = load_golden(tag)
    dtype, tol = (torch.float32, F32_TOL) if prec == "f32" else (torch.float64, F64_TOL)
    dims, P = _setup(meta, dtype)
    B, N, T = meta["B"], meta["N"], meta["T"]
    mem, mel, lens = synth.make_inputs(meta["input_seed"], B, N, T, dims)
    assert lens.tolist() == meta["lengths"]
    mem_t, mel_t = torch.from_numpy(mem).to(dtype), torch.from_numpy(mel).to(dtype)
    if not meta["with_grads"]:
        with torch.no_grad():
            m, g, a = O.forward_teacher(P, mem_t, mel_t, lens, meta["dropout_seed"], meta["training"],
                                        dims.p_attention_dropout, dims.p_decoder_dropout)
        grads = None
    else:
        r_mel = (synth.uniform01(meta["input_seed"], 20, B * dims.n_mels * T) - 0.5).astype(np.float32).reshape(B, dims.n_mels, T)
        r_gate = (synth.uniform01(meta["input_seed"], 21, B * T) - 0.5).astype(np.float32).reshape(B, T)
        (m, g, a), grads, gmem = O.loss_and_grads(P, mem_t, mel_t, lens, torch.from_numpy(r_mel).to(dtype),
                                                  torch.from_numpy(r_gate).to(dtype), meta["dropout_seed"],
                                                  meta["training"], dims.p_attention_dropout, dims.p_decoder_dropout)
        grads = dict(grads)
        grads["memory"] = gmem
    fr = meta.get("frames")         # long fixtures keep selected frames only (oracle/make_golden.py: keep_frames_of)
    ms, gs, as_ = (m, g, a) if fr is None else (m[:, :, fr], g[:, fr], a[:, fr])
    assert rel_err(ms, z[f"mel_{prec}"]) < tol_of(z, "mel_{p}", prec, tol)
    assert rel_err(gs, z[f"gate_{prec}"]) < tol_of(z, "gate_{p}", prec, tol)
    assert rel_err(as_, z[f"align_{prec}"]) < tol_of(z, "align_{p}", prec, tol)
    # padded tokens get exactly zero attention (tacotron2.py:125)
    for b, L in enumerate(lens):
        assert float(np.abs(a[b, :, L:].numpy()).max(initial=0.0)) == 0.0
    if grads is not None:
        for name, gr in grads.items():
            gr = gr.numpy()
            pre = f"grad_{prec}|{name}"
            which = "full" if f"{pre}|full" in z else "vals"
            gtol = tol_of(z, "grad_{p}|" + name + "|" + which, prec, 50 * tol)
            l2 = float(z[f"{pre}|l2"])
            assert abs(np.sqrt((gr.astype(np.float64) ** 2).sum()) - l2) <= gtol * max(l2, 1e-30), name
            if f"{pre}|full" in z:
                assert np.abs(gr - z[f"{pre}|full"]).max() <= gtol * max(np.abs(z[f"{pre}|full"]).max(), 1e-30), name
            else:           # a fixed sample of positions (oracle/make_golden.py: grad_digest)
                ref = z[f"{pre}|vals"]
                assert np.abs(gr.reshape(-1)[z[f"{pre}|idx"]] - ref).max() <= gtol * max(np.abs(ref).max(), 1e-30), name
            if f"{pre}|colsum" in z:
                cs = z[f"{pre}|colsum"]
                assert np.abs(gr.astype(np.float64).sum(0) - cs).max() <= 20 * gtol * max(np.abs(cs).max(), 1e-30), name


@pytest.mark.parametrize("tag", golden_tags("decode_loop"))
@pytest.mark.parametrize("prec", ["f32", "f64"])
def test_batched_decode_loop_matches_reference(tag, prec):
    meta, z = load_golden(tag)
    dtype, tol = (torch.float32, F32_TOL) if prec == "f32" else (torch.float64, F64_TOL)
    dims, P = _setup(meta, dtype)
    mem, _, lens = synth.make_inputs(meta["input_seed"], meta["B"], meta["N"], 0, dims)
    m, g, a, nf = O.inference(P, torch.from_numpy(mem).to(dtype), lens if meta["masked"] else None,
                              max_decoder_steps=meta["steps"], ignore_gate=True, seed=meta["dropout_seed"])
    assert nf.tolist() == [meta["steps"]] * meta["B"]
    assert rel_err(m, z[f"mel_{prec}"]) < tol_of(z, "mel_{p}", prec, tol)
    assert rel_err(g, z[f"gate_{prec}"]) < tol_of(z, "gate_{p}", prec, tol)
    assert rel_err(a, z[f"align_{prec}"]) < tol_of(z, "align_{p}", prec, tol)


@pytest.mark.parametrize("tag", golden_tags("decode_stops"))
@pytest.mark.parametrize("prec", ["f32", "f64"])
def test_batched_decode_rows_stop_at_different_steps(tag, prec):
    """The oracle's batched `inference` applies the reference stop rule (tacotron2.py:405, :407) per row."""
    meta, z = load_golden(tag)
    dtype, tol = (torch.float32, F32_TOL) if prec == "f32" else (torch.float64, F64_TOL)
    dims, P = _setup(meta, dtype)
    mem, _, lens = synth.make_inputs(meta["input_seed"], meta["B"], meta["N"], 0, dims)
    m, g, a, nf = O.inference(P, torch.from_numpy(mem).to(dtype), lens, max_decoder_steps=meta["steps"],
                              gate_threshold=meta["gate_threshold"], ignore_gate=False, seed=meta["dropout_seed"])
    assert nf.tolist() == meta["n_frames"] and len(set(meta["n_frames"])) >= 3
    n = m.shape[2]
    assert n == max(meta["n_frames"])
    assert rel_err(m, z[f"mel_{prec}"][:, :, :n]) < tol_of(z, "mel_{p}", prec, tol)
    assert rel_err(g, z[f"gate_{prec}"][:, :n]) < tol_of(z, "gate_{p}", prec, tol)
    assert rel_err(a, z[f"align_{prec}"][:, :n]) < tol_of(z, "align_{p}", prec, tol)


@pytest.mark.parametrize("tag", golden_tags("public_inference"))
@pytest.mark.parametrize("prec", ["f32", "f64"])
def test_public_inference_gate_stop_matches_reference(tag, prec):
    meta, z = load_golden(tag)
    dtype, tol = (torch.float32, F32_TOL) if prec == "f32" else (torch.float64, F64_TOL)
    dims, P = _setup(meta, dtype)
    mem, _, _ = synth.make_inputs(meta["input_seed"], 1, meta["N"], 0, dims, ragged=False)
    m, g, a, nf = O.inference(P, torch.from_numpy(mem).to(dtype), None, dims.max_decoder_steps,
                              dims.gate_threshold, False, meta["dropout_seed"])
    assert nf.tolist() == [meta["n_frames"]]          # stop step exact (tacotron2.py:405)
    assert m.shape[2] == meta["n_frames"] < dims.max_decoder_steps
    assert rel_err(m, z[f"mel_{prec}"]) < tol_of(z, "mel_{p}", prec, tol)
    assert rel_err(g, z[f"gate_{prec}"]) < tol_of(z, "gate_{p}", prec, tol)
    assert rel_err(a, z[f"align_{prec}"]) < tol_of(z, "align_{p}", prec, tol)


def test_fp32_reference_noise_floor_is_far_below_parity_tolerance():
    """fp32 vs fp64 reference: sets the floor under the 1e-4 parity bound of north_star."""
    meta, z = load_golden("fwd_default_train")
    assert rel_err(z["mel_f32"], z["mel_f64"]) < 1e-5
    assert rel_err(z["align_f32"], z["align_f64"]) < 1e-5


def test_bf16_semantics_memory_rounding_is_opt_in_and_small():
    """bf16_semantics(round_memory=True) mirrors the fused attention chain's extra rounding point (bf16 memory operand of
    the context, tacotron2.py:127); the default bf16 semantics and the fp32 oracle are untouched by it."""
    import torch

    from oracle import decoder_oracle as O
    from oracle import synth
    dims = synth.SMALL_DIMS
    W = O.as_params(synth.make_decoder_weights(5, dims))
    mem, mel, lens = synth.make_inputs(9, 3, 11, 4, dims)
    args = (W, torch.from_numpy(mem), torch.from_numpy(mel), lens)
    plain = O.forward_teacher(*args, seed=3, training=True)
    with O.bf16_semantics():
        b0 = O.forward_teacher(*args, seed=3, training=True)
    with O.bf16_semantics(round_memory=True):
        b1 = O.forward_teacher(*args, seed=3, training=True)
    again = O.forward_teacher(*args, seed=3, training=True)
    assert all(torch.equal(x, y) for x, y in zip(plain, again))               # the context managers restore the fp32 oracle
    d01 = float((b0[0] - b1[0]).abs().max() / b0[0].abs().max())
    assert 0.0 < d01 < 5e-3                                                    # one more bf16 rounding: visible but small
    assert float((b0[0] - plain[0]).abs().max() / plain[0].abs().max()) < 3e-2


def test_loss_and_grads_row_offset_selects_rows_of_one_dropout_stream():
    """Rows k.. of a batch run at row offset 0 are what the same rows compute on their own at row offset k (rows never interact;
    the dropout masks are drawn per global row): outputs and d memory equal, and the offset really changes the masks."""
    dims = synth.SMALL_DIMS
    B, N, T, k, seed = 5, 9, 4, 2, 11
    P = O.as_params(synth.make_decoder_weights(3, dims), torch.float64)
    mem, mel, lens = synth.make_inputs(5, B, N, T, dims)
    mem, mel = torch.from_numpy(mem).double(), torch.from_numpy(mel).double()
    u = lambda s, shape: torch.from_numpy(synth.uniform01(5, s, int(np.prod(shape))).reshape(shape) - 0.5)
    r_mel, r_gate = u(20, (B, dims.n_mels, T)), u(21, (B, T))
    r_mel[:k], r_gate[:k] = 0.0, 0.0
    (m, g, a), _, dm = O.loss_and_grads(P, mem, mel, lens, r_mel, r_gate, seed)
    (ms, gs, as_), _, dms = O.loss_and_grads(P, mem[k:], mel[k:], lens[k:], r_mel[k:], r_gate[k:], seed, row_offset=k)
    for x, y in ((ms, m[k:]), (gs, g[k:]), (as_, a[k:]), (dms, dm[k:])):
        assert rel_err(x, y) < 1e-12
    (m0, _, _), _, _ = O.loss_and_grads(P, mem[k:], mel[k:], lens[k:], r_mel[k:], r_gate[k:], seed)
    assert rel_err(m0, m[k:]) > 1e-2
