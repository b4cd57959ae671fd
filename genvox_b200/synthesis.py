"""Batched synthesis around the B200-native decoder (SURVEY.md §8f N1).

The reference synthesises ONE utterance per call: `Synthesizer.tts` builds `tokens [1, n_tok]`
(/root/reference/core/synthesizer.py:33-38) and `Tacotron2.inference` (/root/reference/models/tts/tacotron2.py:483-499)
runs embedding -> `Encoder.inference` -> `Decoder.inference` -> postnet with a host sync per decoder step (:405).
`Decoder.inference` of this package decodes B rows at once (per-row gate stop on the device, `memory_lengths` mask), so
the batch is built AROUND it while everything that is not row-independent in the reference stays per utterance:

  * `Encoder.inference` ignores lengths (tacotron2.py:248-256), so padded tokens would change the encoder output of
    the shorter utterances: the encoder runs per utterance and its OUTPUTS are zero-padded to the longest one;
  * the postnet's conv stack sees zero padding past the last frame of a B = 1 call: it runs per utterance on the
    frames up to that row's stop step.

`batched_inference(model, token_rows)` therefore returns, for every utterance, exactly the dictionary
`Tacotron2.inference` returns for it alone (same keys, leading batch dimension of 1), up to fp32 rounding of the
decoder (the token split over the two CTAs of a row depends on the padded length).  `sharded_inference` is the
multi-GPU form: utterances are sharded over ranks, no collective (BASELINE configs[3]).  `continuous_inference` returns
the same dictionaries from one continuous-batching call (`Decoder.inference_continuous`): a decoder row whose utterance
stops takes the next utterance of the queue instead of idling until its batch ends.  `SynthesisSession` is the serving
form (`Decoder.session`): token rows are submitted whenever they arrive, and each `step` returns partial mel chunks and,
for every utterance that finished, the same dictionary.
"""
import torch

from .decoder import FROM_ATTRIBUTE
from .training import shard_rows


def _as_rows(token_rows, device):
    rows = []
    for r in token_rows:
        t = torch.as_tensor(r, dtype=torch.int32, device=device).reshape(-1)
        if t.numel() == 0:
            raise ValueError("genvox_b200.synthesis: empty token sequence")
        rows.append(t)
    return rows


@torch.no_grad()
def batched_inference(model, token_rows, max_batch=64, ignore_gate=False, max_decoder_steps=None, attention_window=FROM_ATTRIBUTE):
    """`model`: a reference Tacotron2 whose decoder was swapped by `genvox_b200.install` (needs `.embedding`,
    `.encoder.inference`, `.decoder.inference`, `.postnet`).  `token_rows`: sequence of 1-D integer token-id sequences.
    Returns a list (input order) of dicts with the reference's keys (tacotron2.py:492-498):
    mel_outputs [1,n_mels,T_i], mel_outputs_postnet [1,n_mels,T_i], gate_outputs [1,T_i], alignments [1,T_i,n_tok_i].
    attention_window goes to `Decoder.inference` (left out: the decoder's `attention_window` attribute)."""
    dev = next(model.parameters()).device
    rows = _as_rows(token_rows, dev)
    # longest first inside every decoder batch (the decoder's mask only needs lengths; sorting keeps batches dense)
    order = sorted(range(len(rows)), key=lambda i: -rows[i].numel())
    out = [None] * len(rows)
    win = {} if attention_window is FROM_ATTRIBUTE else {"attention_window": attention_window}   # decoders without the option work
    for lo in range(0, len(order), max_batch):
        idx = order[lo:lo + max_batch]
        enc = []
        for i in idx:   # Encoder.inference per utterance: [1, n_tok] -> [1, n_tok, enc_dim]   (tacotron2.py:486-487)
            emb = model.embedding(rows[i].unsqueeze(0)).transpose(1, 2)
            enc.append(model.encoder.inference(emb))
        lengths = torch.tensor([e.shape[1] for e in enc], dtype=torch.int64, device=dev)
        n_max = int(lengths.max())
        memory = torch.zeros(len(idx), n_max, enc[0].shape[2], dtype=torch.float32, device=dev)
        for r, e in enumerate(enc):
            memory[r, :e.shape[1]] = e[0]
        mel, gate, align = model.decoder.inference(memory, memory_lengths=lengths, ignore_gate=ignore_gate,
                                                   max_decoder_steps=max_decoder_steps, **win)
        n_frames = model.decoder.last_n_frames.tolist()          # one device->host read per batch (reference: one per step)
        for r, i in enumerate(idx):
            t_i, n_i = int(n_frames[r]), int(lengths[r])
            m = mel[r:r + 1, :, :t_i].contiguous()
            out[i] = {
                "mel_outputs": m,
                "mel_outputs_postnet": m + model.postnet(m),     # tacotron2.py:490-491
                "gate_outputs": gate[r:r + 1, :t_i].contiguous(),
                "alignments": align[r:r + 1, :t_i, :n_i].contiguous(),
            }
    return out


@torch.no_grad()
def sharded_inference(model, token_rows, rank, world, **kwargs):
    """Utterances [lo, hi) of `token_rows` on this rank (contiguous shards, no collective).  Returns (lo, outputs)."""
    lo, hi = shard_rows(len(token_rows), rank, world)
    return lo, batched_inference(model, token_rows[lo:hi], **kwargs)


@torch.no_grad()
def continuous_inference(model, token_rows, slots=64, **kw):
    """Like `batched_inference`, but the decoder runs every utterance in one `Decoder.inference_continuous` call through
    `slots` rows, in the order given (utterance i draws prenet dropout row i + dropout_row_offset).  `kw` goes to
    `inference_continuous` (max_decoder_steps, frame_caps, ignore_gate, return_alignments, attention_window); "alignments"
    is None when alignments are not returned."""
    dev = next(model.parameters()).device
    rows = _as_rows(token_rows, dev)
    enc = []
    for r in rows:      # Encoder.inference per utterance (tacotron2.py:486-487), outputs zero-padded to the longest
        emb = model.embedding(r.unsqueeze(0)).transpose(1, 2)
        enc.append(model.encoder.inference(emb))
    lengths = torch.tensor([e.shape[1] for e in enc], dtype=torch.int64, device=dev)
    memory = torch.zeros(len(rows), int(lengths.max()), enc[0].shape[2], dtype=torch.float32, device=dev)
    for i, e in enumerate(enc):
        memory[i, :e.shape[1]] = e[0]
    mel, gate, align = model.decoder.inference_continuous(memory, lengths, slots=slots, **kw)
    n_frames = model.decoder.last_n_frames.tolist()
    out = []
    for i in range(len(rows)):
        t_i, n_i = int(n_frames[i]), int(lengths[i])
        m = mel[i:i + 1, :, :t_i].contiguous()
        out.append({
            "mel_outputs": m,
            "mel_outputs_postnet": m + model.postnet(m),     # tacotron2.py:490-491
            "gate_outputs": gate[i:i + 1, :t_i].contiguous(),
            "alignments": align[i:i + 1, :t_i, :n_i].contiguous() if align is not None else None,
        })
    return out


class SynthesisSession:
    """Continuous synthesis for requests that arrive over time, around a decoder session (`Decoder.session`) of
    `max_tokens` tokens per utterance and `slots` decoder rows; `kw` goes to `Decoder.session` (capacity,
    max_decoder_steps, ignore_gate, return_alignments, attention_window).  Utterance `id` draws prenet dropout row id + dropout_row_offset,
    so with the same N (= max_tokens) and seed its dictionary equals `continuous_inference`'s for the same token rows."""

    def __init__(self, model, max_tokens, slots=64, **kw):
        self.model = model
        self.session = model.decoder.session(max_tokens, slots=slots, **kw)
        self._device = next(model.parameters()).device
        self._parts = {}        # id -> (n_tokens, [(mel, gate, align)] chunks so far)

    @torch.no_grad()
    def submit(self, token_rows):
        """Runs the embedding and `Encoder.inference` per utterance (tacotron2.py:486-487) and queues the outputs.
        Returns the ids."""
        rows = _as_rows(token_rows, self._device)
        if not rows:
            return []
        enc = []
        for r in rows:
            if r.numel() > self.session.N:
                raise ValueError(f"genvox_b200.synthesis: {r.numel()} tokens, more than the session's {self.session.N}")
            emb = self.model.embedding(r.unsqueeze(0)).transpose(1, 2)
            enc.append(self.model.encoder.inference(emb))
        lengths = torch.tensor([e.shape[1] for e in enc], dtype=torch.int64, device=self._device)
        memory = torch.zeros(len(rows), self.session.N, enc[0].shape[2], dtype=torch.float32, device=self._device)
        for i, e in enumerate(enc):
            memory[i, :e.shape[1]] = e[0]
        ids = self.session.submit(memory, lengths)
        for i, n in zip(ids, lengths.tolist()):
            self._parts[i] = (n, [])
        return ids

    @torch.no_grad()
    def step(self, steps=16):
        """Runs up to `steps` decoder steps.  Returns (chunks, finished): chunks = {id: mel [1, n_mels, j]} with the new
        frames of every utterance that advanced; finished = {id: dict with the keys of Tacotron2.inference}, as
        `continuous_inference` returns it.  The postnet runs once an utterance has finished: its convolutions see the
        whole utterance."""
        new, done = self.session.step(steps)
        chunks = {}
        for i, part in new.items():
            self._parts[i][1].append(part)
            chunks[i] = part[0].unsqueeze(0)
        finished = {}
        for i in done:
            n_tok, parts = self._parts.pop(i)
            m = torch.cat([p[0] for p in parts], dim=1).unsqueeze(0).contiguous()
            align = None
            if self.session.return_alignments:
                align = torch.cat([p[2] for p in parts], dim=0)[:, :n_tok].unsqueeze(0).contiguous()
            finished[i] = {
                "mel_outputs": m,
                "mel_outputs_postnet": m + self.model.postnet(m),     # tacotron2.py:490-491
                "gate_outputs": torch.cat([p[1] for p in parts]).unsqueeze(0).contiguous(),
                "alignments": align,
            }
        return chunks, finished
