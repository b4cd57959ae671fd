"""TEST INFRASTRUCTURE — a small stand-in for the reference Tacotron2 model (tacotron2.py:416-615) around a CPU decoder.

The wiring tests need a whole model to install the B200 decoder into: an embedding, an encoder with `inference`, a
decoder, a postnet, and the model methods the reference Trainer and Synthesizer call (`get_criterion`, `get_optimizer`,
`train_step`, `get_checkpoint_statedicts`, `load_checkpoint_statedicts`, `inference`).  The reference ships no such
model with this repository, so `Tacotron2` here has those names and call signatures, small deterministic torch modules
for everything outside the decoder, and `OracleDecoder` as its decoder: the reference Decoder's constructor, attributes
and state_dict (they are genvox_b200.Decoder's) with forward / inference computed by oracle/decoder_oracle.py on the
host - the oracle that tests/test_oracle_golden.py pins to outputs of the unmodified reference.  Dropout masks come from
the shared Philox stream (`set_dropout_seed`, `dropout_row_offset`), as in the CUDA decoder.
"""
import types

import torch
import torch.nn as nn
import torch.nn.functional as F

import genvox_b200

from . import decoder_oracle as O


class OracleDecoder(genvox_b200.Decoder):
    """Reference-layout decoder whose forward / inference run the CPU oracle (fp32, torch autograd for BPTT)."""

    def forward(self, memory, decoder_inputs, memory_lengths):
        P = dict(self.named_parameters())
        return O.forward_teacher(P, memory, decoder_inputs, memory_lengths, self._next_seed(), self.training,
                                 self.p_attention_dropout, self.p_decoder_dropout, self.dropout_row_offset)

    @torch.no_grad()
    def inference(self, memory, memory_lengths=None, ignore_gate=False, max_decoder_steps=None):
        steps = int(max_decoder_steps if max_decoder_steps is not None else self.max_decoder_steps)
        m, g, a, n_frames = O.inference(dict(self.named_parameters()), memory, memory_lengths, steps, self.gate_threshold,
                                        ignore_gate, self._next_seed(), self.training, self.p_attention_dropout,
                                        self.p_decoder_dropout, self.dropout_row_offset)
        self.last_n_frames = n_frames
        return m, g, a


class Encoder(nn.Module):
    """[B, sym, n_tok] -> [B, n_tok, enc]; `inference` ignores lengths like the reference's (tacotron2.py:248-256)."""

    def __init__(self, sym, enc):
        super().__init__()
        self.conv = nn.Conv1d(sym, enc, 5, padding=2)

    def forward(self, x, lengths=None):
        return torch.tanh(self.conv(x)).transpose(1, 2)

    inference = forward


def tacotron2_loss(batch, outputs):
    """Tacotron2Loss (tacotron2.py:598-615)."""
    mel_loss = F.mse_loss(outputs["mel_outputs"], batch["mel_padded"]) + \
        F.mse_loss(outputs["mel_outputs_postnet"], batch["mel_padded"])
    gate_loss = F.binary_cross_entropy_with_logits(outputs["gate_outputs"].reshape(-1, 1), batch["gate_padded"].reshape(-1, 1))
    return {"loss": mel_loss + gate_loss, "mel_loss": mel_loss, "gate_loss": gate_loss}


class Tacotron2(nn.Module):
    """Same construction under the same torch seed => same parameters, so two instances are replicas."""

    def __init__(self, dims, n_tokens=64, sym=32, seed=0):
        super().__init__()
        torch.manual_seed(seed)
        self.embedding = nn.Embedding(n_tokens, sym)
        self.encoder = Encoder(sym, dims.encoder_embedding_dim)
        self.decoder = OracleDecoder(**dims.kwargs())
        self.postnet = nn.Sequential(nn.Conv1d(dims.n_mels, 64, 5, padding=2), nn.Tanh(),
                                     nn.Conv1d(64, dims.n_mels, 5, padding=2))
        self.model_config = types.SimpleNamespace(grad_clip_thresh=1.0, learning_rate=1e-3, weight_decay=1e-6)

    def prepare_batch(self, batch, device=None):
        return {k: v.to(device if device is not None else next(self.parameters()).device) for k, v in batch.items()}

    def forward(self, batch):                                             # tacotron2.py:450-481
        emb = self.embedding(batch["token_padded"]).transpose(1, 2)
        enc = self.encoder(emb, batch["token_lengths"])
        mel, gate, align = self.decoder(enc, batch["mel_padded"], batch["token_lengths"])
        return {"mel_outputs": mel, "mel_outputs_postnet": mel + self.postnet(mel), "gate_outputs": gate, "alignments": align}

    @torch.no_grad()
    def inference(self, inputs):                                          # tacotron2.py:483-499 (B = 1)
        tokens = inputs["tokens"].to(next(self.parameters()).device)
        emb = self.embedding(tokens).transpose(1, 2)
        mel, gate, align = self.decoder.inference(self.encoder.inference(emb))
        return {"mel_outputs": mel, "mel_outputs_postnet": mel + self.postnet(mel), "gate_outputs": gate, "alignments": align}

    def get_criterion(self):
        return {"loss": tacotron2_loss}

    def get_optimizer(self):
        return {"optimizer": torch.optim.Adam(self.parameters(), lr=self.model_config.learning_rate,
                                              weight_decay=self.model_config.weight_decay)}

    def train_step(self, batch, criterion, optimizer):                   # tacotron2.py:515-522
        optimizer["optimizer"].zero_grad()
        loss = criterion["loss"](batch, self.forward(batch=batch))
        self.loss_items = {key: val.item() for key, val in loss.items()}
        loss["loss"].backward()
        self.grad_norm_val = torch.nn.utils.clip_grad_norm_(self.parameters(), self.model_config.grad_clip_thresh).item()
        optimizer["optimizer"].step()

    def get_checkpoint_statedicts(self, optimizer=None):
        return {"model_statedict": self.state_dict(),
                "optimizer_statedict": optimizer["optimizer"].state_dict() if optimizer is not None else None}

    def load_checkpoint_statedicts(self, statedicts, save_optimizer_dict, optimizer):
        self.load_state_dict(statedicts["model_statedict"])
        if save_optimizer_dict:
            optimizer["optimizer"].load_state_dict(statedicts["optimizer_statedict"])
