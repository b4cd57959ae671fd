"""GPU tests of the drop-in wiring on a whole Tacotron2 model (oracle/standin.py: the reference model's interface, its
decoder the CPU oracle that tests/test_oracle_golden.py pins to the unmodified reference): that model on the CPU is the
yardstick, the same model with `genvox_b200.install`ed decoder on the B200 is the subject.

  * `model_train_step` vs `Tacotron2.train_step` (tacotron2.py:515-522) on the same batch: same loss items, same gradient for
    every parameter of the model (embedding, encoder, decoder, postnet - the encoder's come through d memory);
  * `batched_inference` / `wiring.tts_batch` vs `Tacotron2.inference` (tacotron2.py:483-499) run once per utterance.
Both decoders draw the same counter-based Philox dropout masks (same seed and row offset)."""
import numpy as np
import pytest
import torch

import genvox_b200
from conftest import rel_err
from genvox_b200 import synthesis
from genvox_b200.training import model_train_step
from oracle import standin, synth

pytestmark = pytest.mark.gpu


def _model(seed):
    return standin.Tacotron2(synth.DecoderDims(), seed=seed)


def _batch(B, n_tok, T, seed):
    g = torch.Generator().manual_seed(seed)
    lens = torch.sort(torch.randint(n_tok // 2, n_tok + 1, (B,), generator=g), descending=True).values      # collate order (:32)
    lens[0] = n_tok
    tok = torch.randint(1, 64, (B, n_tok), generator=g)
    for b in range(B):
        tok[b, lens[b]:] = 0
    mel = torch.randn(B, 80, T, generator=g)
    gate = torch.zeros(B, T)
    gate[:, -1] = 1.0
    return {"token_padded": tok, "token_lengths": lens, "mel_padded": mel, "gate_padded": gate,
            "mel_lengths": torch.full((B,), T, dtype=torch.int64)}


def test_model_train_step_matches_reference_train_step(cuda_device):
    B, n_tok, T, seed = 6, 23, 14, 321
    # the encoder / postnet stay stock PyTorch on the GPU: keep cuDNN / cuBLAS out of TF32 so that they are comparable with the CPU
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    ref = _model(2)
    ours = genvox_b200.install(_model(2)).to(cuda_device)
    for m in (ref, ours):
        m.train()                   # decoder: LSTM-state dropout on, like a training step
    batch = _batch(B, n_tok, T, 5)
    # ---- reference: its own train_step on the CPU
    crit, opt = ref.get_criterion(), ref.get_optimizer()
    ref.decoder.set_dropout_seed(seed)
    ref.train_step(batch={k: v.clone() for k, v in batch.items()}, criterion=crit, optimizer=opt)
    ref_grads = {k: p.grad.clone() for k, p in ref.named_parameters()}
    # ---- installed model on the GPU through the data-parallel-ready step (no group: single process)
    ours.decoder.set_dropout_seed(seed)
    gb = ours.prepare_batch({k: v.clone() for k, v in batch.items()}, device=cuda_device)
    items = model_train_step(ours, gb, ours.get_criterion(), ours.get_optimizer())
    torch.cuda.synchronize()
    genvox_b200.check_device_errors()
    for k, v in ref.loss_items.items():
        assert abs(float(items[k]) - v) <= 2e-5 * max(abs(v), 1.0), (k, float(items[k]), v)
    assert abs(float(ours.grad_norm_val) - ref.grad_norm_val) <= 1e-4 * ref.grad_norm_val
    worst = ("", 0.0)
    for k, p in ours.named_parameters():
        e = rel_err(p.grad.cpu(), ref_grads[k])
        worst = max(worst, (k, e), key=lambda kv: kv[1])
        assert e < (2e-4 if k.startswith("decoder.") else 1e-3), (k, e)
    print("worst gradient rel err over the whole model:", worst)


def test_batched_synthesis_matches_reference_inference_per_utterance(cuda_device):
    seed, steps = 77, 10
    torch.backends.cudnn.allow_tf32 = False         # the postnet runs on the GPU on one side: no TF32 convolutions
    ref = _model(4).eval()
    ours = genvox_b200.install(_model(4)).to(cuda_device).eval()
    for m in (ref, ours):
        m.decoder.max_decoder_steps = steps
        m.decoder.gate_threshold = 0.999999            # random-init gate logits: every utterance runs to max_decoder_steps
    g = torch.Generator().manual_seed(9)
    rows = [torch.randint(1, 64, (n,), generator=g).tolist() for n in (17, 9, 26, 12)]
    ours.decoder.set_dropout_seed(seed)
    outs = synthesis.batched_inference(ours, rows)
    torch.cuda.synchronize()
    genvox_b200.check_device_errors()
    order = sorted(range(len(rows)), key=lambda i: -len(rows[i]))             # batched_inference decodes longest first
    for slot, i in enumerate(order):
        ref.decoder.set_dropout_seed(seed)
        ref.decoder.dropout_row_offset = slot                                    # the row the utterance has in the batch
        r = ref.inference(inputs={"tokens": torch.IntTensor(rows[i]).unsqueeze(0)})
        o = outs[i]
        assert set(o.keys()) == set(r.keys())
        for k in r:
            assert tuple(o[k].shape) == tuple(r[k].shape), (k, o[k].shape, r[k].shape)
            assert rel_err(o[k].cpu(), r[k]) < 1e-4, (i, k, rel_err(o[k].cpu(), r[k]))
        assert o["mel_outputs"].shape[2] == steps
