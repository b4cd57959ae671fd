"""TEST INFRASTRUCTURE (build container only) — write tests/golden/*.npz.

Runs the UNMODIFIED reference modules from /root/reference (oracle/ref_import.py) on
Philox-synthesised weights / inputs (oracle/synth.py) with replayable dropout masks, in
fp32 and in fp64 (`.double()`, the error yardstick), and stores the outputs.  The
reference has no golden vectors of its own (SURVEY.md §4, §8c), so these files are the pin
for oracle/decoder_oracle.py and, through it, for the CUDA path.

    python -m oracle.make_golden          # rewrites every fixture

Each fixture records the seeds and dims it was made from; tests rebuild weights/inputs
from those seeds with oracle/synth.py (no torch RNG involved) and compare.
"""
import json
import os
import sys

import numpy as np
import torch

from . import decoder_oracle as O
from . import ref_import as R
from . import synth

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")
LSTM_ROWS = [0, 1, 2, 3, 511, 1023, 1024, 1025, 2047, 2048, 2049, 3071, 3072, 3073, 4094, 4095]


def grad_digest(name, g, full_limit=70000, n_sample=1024, colsum_limit=20000):
    """What we keep of one gradient tensor: everything if small, else norms, the sum over the first axis when it has at
    most `colsum_limit` entries, and the values at a fixed sample of `n_sample` positions inside the rows LSTM_ROWS (`idx`:
    flat indices into the tensor).  The limits keep every fixture file under 1 MB (the (60, 512) sum of d memory in
    fwd_default_long would not fit)."""
    g = np.asarray(g)
    out = {f"{name}|sum": np.float64(g.astype(np.float64).sum()),
           f"{name}|l2": np.float64(np.sqrt((g.astype(np.float64) ** 2).sum()))}
    if g.size <= full_limit:
        out[f"{name}|full"] = g
        return out
    rows = np.asarray([r for r in LSTM_ROWS if r < g.shape[0]], dtype=np.int64)
    width = g.size // g.shape[0]
    pick = np.sort(np.random.default_rng(0).choice(len(rows) * width, min(n_sample, len(rows) * width), replace=False))
    idx = rows[pick // width] * width + pick % width
    out[f"{name}|idx"] = idx
    out[f"{name}|vals"] = g.reshape(-1)[idx]
    if width <= colsum_limit:
        out[f"{name}|colsum"] = g.astype(np.float64).sum(0)
    return out


def run_reference_forward(dims, W, mem, mel, lens, seed, training, dtype, r_mel=None, r_gate=None):
    dec = R.build_reference_decoder(dims, W, dtype)
    dec.train(training)
    memory = torch.from_numpy(mem).to(dtype).requires_grad_(r_mel is not None)
    with R.philox_dropout_patch(seed, "forward"):
        m, g, a = dec(memory, torch.from_numpy(mel).to(dtype), torch.from_numpy(lens))
    grads = None
    if r_mel is not None:
        loss = (m * torch.from_numpy(r_mel).to(dtype)).sum() + (g * torch.from_numpy(r_gate).to(dtype)).sum()
        loss.backward()     # the BPTT of tacotron2.py:520 restricted to the decoder graph
        grads = {k: v.grad.detach().numpy() for k, v in dec.named_parameters()}
        grads["memory"] = memory.grad.numpy()
    return m.detach().numpy(), g.detach().numpy(), a.detach().numpy(), grads


def run_reference_decode_loop(dims, W, mem, lens, seed, steps, dtype):
    """B >= 1 inference by driving the reference's own initialize_decoder_states / prenet / decode
    (tacotron2.py:303,:140,:333) — the public `inference` is B = 1 only (:405)."""
    ref = R.import_reference()
    dec = R.build_reference_decoder(dims, W, dtype)
    dec.eval()
    memory = torch.from_numpy(mem).to(dtype)
    mask = None if lens is None else ref.get_mask_from_lengths(torch.from_numpy(lens))
    mels, gates, aligns = [], [], []
    with torch.no_grad(), R.philox_dropout_patch(seed, "inference"):
        dec.initialize_decoder_states(memory, mask=mask)
        x = memory.new_zeros(memory.shape[0], dims.n_mels)
        for _ in range(steps):
            m, g, a = dec.decode(dec.prenet(x))
            mels.append(m), gates.append(g.squeeze(1)), aligns.append(a)
            x = m
        m, g, a = dec.parse_decoder_outputs(mels, gates, aligns)
    return m.numpy(), g.numpy(), a.numpy()


def keep_frames_of(T, head=12, stride=13, tail=12):
    """Frames a long fixture keeps (the file stays small): the first `head`, every `stride`-th, the last `tail`."""
    return sorted(set(range(min(head, T))) | set(range(0, T, stride)) | set(range(max(0, T - tail), T)))


def case_forward(tag, dims, B, N, T, wseed, iseed, dseed, training=True, with_grads=True, wscale=1.0, subsample=False,
                 full_limit=70000):
    W = synth.make_decoder_weights(wseed, dims, wscale)
    mem, mel, lens = synth.make_inputs(iseed, B, N, T, dims)
    r_mel = (synth.uniform01(iseed, 20, B * dims.n_mels * T) - 0.5).astype(np.float32).reshape(B, dims.n_mels, T)
    r_gate = (synth.uniform01(iseed, 21, B * T) - 0.5).astype(np.float32).reshape(B, T)
    out = {}
    for dtype, sfx in ((torch.float32, "f32"), (torch.float64, "f64")):
        m, g, a, grads = run_reference_forward(dims, W, mem, mel, lens, dseed, training, dtype,
                                               r_mel if with_grads else None, r_gate)
        if subsample:       # long sequences: selected frames only (tests slice their outputs with meta["frames"])
            fr = keep_frames_of(T)
            m, g, a = m[:, :, fr], g[:, fr], a[:, fr]
        out[f"mel_{sfx}"], out[f"gate_{sfx}"], out[f"align_{sfx}"] = m, g, a
        if grads is not None:
            for k, v in grads.items():
                for kk, vv in grad_digest(k, v, full_limit).items():
                    out[f"grad_{sfx}|{kk}"] = vv
    meta = dict(kind="forward", dims=dims.kwargs(), B=B, N=N, T=T, weight_seed=wseed, input_seed=iseed,
                dropout_seed=dseed, training=training, weight_scale=wscale, lengths=lens.tolist(),
                with_grads=with_grads, r_mel_stream=20, r_gate_stream=21,
                source="reference Decoder.forward (tacotron2.py:365-388) + autograd (:520)")
    if subsample:
        meta["frames"] = keep_frames_of(T)
    save(tag, meta, out)


def case_decode_stops(tag, dims, B, N, steps, wseed, iseed, dseed, wscale=1.0, margin=2e-3):
    """Batched decode whose rows stop at DIFFERENT steps.  The reference's public loop is B = 1 only (:405 raises for
    B > 1), so its decode() is driven for B rows (as in case_decode_loop) and the reference stop rule of :405 - first
    frame with sigmoid(gate) > threshold, that frame included - is applied per row to the reference's own gate logits.
    The threshold is chosen so that the rows' stop steps differ, at least one row never fires (-> max steps, :407), and
    every logit is at least `margin` away from the threshold (the stop steps then do not hinge on fp32 rounding)."""
    W = synth.make_decoder_weights(wseed, dims, wscale)
    mem, _, lens = synth.make_inputs(iseed, B, N, 0, dims)
    out, gates = {}, {}
    for dtype, sfx in ((torch.float32, "f32"), (torch.float64, "f64")):
        m, g, a = run_reference_decode_loop(dims, W, mem, lens, dseed, steps, dtype)
        out[f"mel_{sfx}"], out[f"gate_{sfx}"], out[f"align_{sfx}"] = m, g, a
        gates[sfx] = g.astype(np.float64)

    def stops(g, logit_thr):
        fired = g > logit_thr
        return [int(np.argmax(fired[b])) + 1 if fired[b].any() else steps for b in range(B)]

    best = None
    vals = np.unique(gates["f64"].reshape(-1))
    for cand in 0.5 * (vals[1:] + vals[:-1]):        # every threshold between two neighbouring logits
        if np.abs(gates["f64"] - cand).min() < margin or np.abs(gates["f32"] - cand).min() < margin:
            continue
        st = stops(gates["f64"], cand)
        score = (len(set(st)), st.count(steps) >= 1, -abs(st.count(steps) - 1))
        if st == stops(gates["f32"], cand) and min(st) >= 2 and (best is None or score > best[0]):
            best = (score, float(cand), st)
    assert best is not None and best[0][0] >= 3 and best[0][1], best
    logit_thr, n_frames = best[1], best[2]
    meta = dict(kind="decode_stops", dims=dims.kwargs(), B=B, N=N, steps=steps, weight_seed=wseed, input_seed=iseed,
                dropout_seed=dseed, masked=True, weight_scale=wscale, lengths=lens.tolist(),
                gate_threshold=float(1.0 / (1.0 + np.exp(-logit_thr))), gate_logit_threshold=logit_thr, n_frames=n_frames,
                source="reference initialize_decoder_states/prenet/decode driven for B rows (tacotron2.py:303,:140,:333); "
                       "per-row stop rule of :405 / :407 applied to the reference's gate logits")
    save(tag, meta, out)


def case_decode_loop(tag, dims, B, N, steps, wseed, iseed, dseed, masked, wscale=1.0):
    W = synth.make_decoder_weights(wseed, dims, wscale)
    mem, _, lens = synth.make_inputs(iseed, B, N, 0, dims)
    out = {}
    for dtype, sfx in ((torch.float32, "f32"), (torch.float64, "f64")):
        m, g, a = run_reference_decode_loop(dims, W, mem, lens if masked else None, dseed, steps, dtype)
        out[f"mel_{sfx}"], out[f"gate_{sfx}"], out[f"align_{sfx}"] = m, g, a
    meta = dict(kind="decode_loop", dims=dims.kwargs(), B=B, N=N, steps=steps, weight_seed=wseed, input_seed=iseed,
                dropout_seed=dseed, masked=masked, weight_scale=wscale, lengths=lens.tolist(),
                source="reference initialize_decoder_states/prenet/decode driven for B rows (tacotron2.py:303,:140,:333)")
    save(tag, meta, out)


def case_public_inference(tag, dims, N, wseed, iseed, dseed, wscale=1.0, probe_steps=40):
    """The reference's public Decoder.inference (B = 1) with a gate threshold chosen so the stop
    test (:405) fires mid-way: first step k >= 3 whose gate logit is a strict running maximum."""
    W = synth.make_decoder_weights(wseed, dims, wscale)
    mem, _, _ = synth.make_inputs(iseed, 1, N, 0, dims, ragged=False)
    _, g, _ = run_reference_decode_loop(dims, W, mem, None, dseed, probe_steps, torch.float32)
    g = g[0].astype(np.float64)
    k = next(k for k in range(3, probe_steps) if g[k] > g[:k].max() + 1e-4)
    logit_thr = 0.5 * (g[k] + g[:k].max())
    thr = float(1.0 / (1.0 + np.exp(-logit_thr)))
    d2 = synth.DecoderDims(**{**dims.kwargs(), "gate_threshold": thr, "max_decoder_steps": probe_steps})
    out = {}
    for dtype, sfx in ((torch.float32, "f32"), (torch.float64, "f64")):
        dec = R.build_reference_decoder(d2, W, dtype)
        dec.eval()
        with torch.no_grad(), R.philox_dropout_patch(dseed, "inference"):
            m, gg, a = dec.inference(torch.from_numpy(mem).to(dtype))
        assert m.shape[2] == k + 1, (m.shape, k)
        out[f"mel_{sfx}"], out[f"gate_{sfx}"], out[f"align_{sfx}"] = m.numpy(), gg.numpy(), a.numpy()
    meta = dict(kind="public_inference", dims=d2.kwargs(), B=1, N=N, weight_seed=wseed, input_seed=iseed,
                dropout_seed=dseed, weight_scale=wscale, n_frames=k + 1,
                source="reference Decoder.inference (tacotron2.py:390-414), B = 1, gate-stopped")
    save(tag, meta, out)


def save(tag, meta, arrays):
    os.makedirs(GOLDEN_DIR, exist_ok=True)
    path = os.path.join(GOLDEN_DIR, f"{tag}.npz")
    meta["torch"] = torch.__version__
    np.savez_compressed(path, meta=np.frombuffer(json.dumps(meta).encode(), dtype=np.uint8), **arrays)
    print(f"{tag}: {os.path.getsize(path) / 1e6:.2f} MB  {meta['kind']}")


def main():
    torch.set_num_threads(8)
    D, S = synth.DecoderDims(), synth.SMALL_DIMS
    if "--new" in sys.argv:      # only the fixtures added in round 2 (the others regenerate bit-identically)
        if "--stops-only" not in sys.argv:
            case_forward("fwd_default_long", D, B=4, N=60, T=400, wseed=7, iseed=19, dseed=131, subsample=True, full_limit=8192)
        case_decode_stops("stops_default_masked", D, B=6, N=33, steps=24, wseed=8, iseed=21, dseed=132, wscale=2.0)
        return 0
    case_forward("fwd_small_train", S, B=3, N=11, T=7, wseed=7, iseed=11, dseed=123, wscale=3.0)
    case_forward("fwd_small_eval", S, B=2, N=9, T=5, wseed=8, iseed=12, dseed=124, training=False, wscale=3.0)
    case_forward("fwd_default_train", D, B=4, N=37, T=10, wseed=7, iseed=11, dseed=123, full_limit=8192)
    case_forward("fwd_default_eval_b1", D, B=1, N=16, T=6, wseed=9, iseed=13, dseed=125, training=False, with_grads=False)
    case_decode_loop("loop_default_nomask", D, B=3, N=23, steps=12, wseed=7, iseed=14, dseed=126, masked=False)
    case_decode_loop("loop_default_masked", D, B=5, N=40, steps=9, wseed=7, iseed=15, dseed=127, masked=True)
    case_decode_loop("loop_small_masked", S, B=4, N=13, steps=15, wseed=8, iseed=16, dseed=128, masked=True, wscale=3.0)
    case_public_inference("infer_default_b1_gate", D, N=29, wseed=7, iseed=17, dseed=129)
    case_public_inference("infer_small_b1_gate", S, N=10, wseed=8, iseed=18, dseed=130, wscale=3.0)
    case_forward("fwd_default_long", D, B=4, N=60, T=400, wseed=7, iseed=19, dseed=131, subsample=True, full_limit=8192)
    case_decode_stops("stops_default_masked", D, B=6, N=33, steps=24, wseed=8, iseed=21, dseed=132, wscale=2.0)


if __name__ == "__main__":
    sys.exit(main())
