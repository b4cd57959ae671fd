"""Decoder sessions: continuous batching for utterances that arrive over time (include/genvox_b200.h, gvx_dec_session_*).

`Decoder.inference_continuous` needs its whole queue up front and returns when the queue is empty.  A `DecoderSession`
keeps `slots` decoder rows and their recurrent state alive between calls: `submit` appends utterances at any time between
calls, and `step(k)` runs up to k decoder steps and returns the frames decoded in them, so a request that arrives during
a long decode joins at the next call and its first frames leave after the call it was admitted in.

Contract (as `inference_continuous`): utterance `id` decodes bit-identically to row r of a static `Decoder.inference` call
with the same `slots` rows, the session's N, the same seed and precision, id in row r and dropout_row_offset =
id + row_offset - r, whatever the submission times, step counts and other slots were.
"""
import ctypes as C

import numpy as np
import torch

from . import _native
from .decoder import _buffer, _f32c, _ptr, _stream


class DecoderSession:
    """Made by `Decoder.session(...)`.  Eval mode only; the decoder's parameters must not change while it runs."""

    def __init__(self, dec, N, slots=64, capacity=1024, max_decoder_steps=None, ignore_gate=False, return_alignments=True):
        if dec.training:
            raise RuntimeError("genvox_b200: decoder sessions run in eval mode only (call .eval())")
        steps = int(max_decoder_steps if max_decoder_steps is not None else dec.max_decoder_steps)
        limit = 128 if dec.precision == "bf16" else None
        if int(slots) < 1 or (limit is not None and int(slots) > limit):
            raise ValueError(f"genvox_b200: slots must be in 1 .. {limit or 'inf'} in {dec.precision} mode, got {slots}")
        if int(N) < 1 or int(capacity) < 1 or steps < 1:
            raise ValueError(f"genvox_b200: N, capacity and max_decoder_steps must be positive, got {N}, {capacity}, {steps}")
        params = [p.detach() for p in dec._ordered_params()]
        if not params[0].is_cuda:
            raise RuntimeError("genvox_b200: the decoder must be on a CUDA device (there is no CPU fallback)")
        self._lib = _native.load()
        self._dec = dec
        self._dims, self._weights, self._packed = dec._native_state(params)
        self._key = dec._pack_key
        self.N, self.slots, self.max_decoder_steps = int(N), int(slots), steps
        self.return_alignments = bool(return_alignments)
        self.n_mels = dec.n_mel_channels
        self.device = params[0].device
        s = _native.GvxSession()
        s.N, s.slots, s.capacity, s.max_steps = self.N, self.slots, int(capacity), steps
        s.ignore_gate, s.with_alignments, s.row_offset = int(bool(ignore_gate)), int(self.return_alignments), dec.dropout_row_offset
        s.gate_threshold, s.seed = float(dec.gate_threshold), dec._next_seed()
        self._s = s
        nbytes = self._lib.gvx_dec_session_workspace_bytes(C.byref(self._dims), self.N, self.slots, int(capacity))
        if nbytes == 0:
            _native.check(1, "gvx_dec_session_workspace_bytes")
        self._work = _buffer(nbytes, self.device)
        _native.check(self._lib.gvx_dec_session_init(C.byref(self._dims), C.byref(s), _ptr(self._work), _stream()),
                      "gvx_dec_session_init")
        self._chunk_steps = 0

    # ------------------------------------------------------------------ state
    @property
    def pending(self):
        """utterances submitted and not yet taken into a slot (as of the end of the last step call)"""
        return self._s.submitted - self._s.admitted

    @property
    def active(self):
        return self._s.active

    @property
    def idle(self):
        return self.slots - self._s.active

    @property
    def steps_run(self):
        return self._s.steps_run

    def _check_weights(self):
        params = [p.detach() for p in self._dec._ordered_params()]
        if self._dec.training or self._dec._packed_key(params) != self._key:
            raise RuntimeError("genvox_b200: the decoder's parameters, precision or mode changed since the session began; "
                               "its utterances would no longer decode as one model (start a new session)")

    # ------------------------------------------------------------------ calls
    def submit(self, memory, lengths, frame_caps=None):
        """memory [k, n <= N, E] (zero-padded to N here), lengths [k] (None: all N), frame_caps [k] in 1 .. max_decoder_steps
        or None.  Returns the ids of the k utterances."""
        self._check_weights()
        memory = _f32c(memory, "memory")
        if memory.dim() != 3 or memory.shape[2] != self._dec.encoder_embedding_dim:
            raise ValueError(f"genvox_b200: memory must be [k, n, {self._dec.encoder_embedding_dim}], got {tuple(memory.shape)}")
        k, n, E = memory.shape
        if n > self.N:
            raise ValueError(f"genvox_b200: memory has {n} tokens, wider than the session's N = {self.N}")
        if k == 0:
            return []
        caps = None
        if frame_caps is not None:
            caps = torch.as_tensor(frame_caps).reshape(-1)
            if caps.numel() != k:
                raise ValueError(f"genvox_b200: frame_caps needs one entry per utterance ({k}), got {caps.numel()}")
            if bool((caps < 1).any()) or bool((caps > self.max_decoder_steps).any()):
                raise ValueError(f"genvox_b200: frame_caps must lie in 1 .. max_decoder_steps ({self.max_decoder_steps})")
            caps = caps.to(device=self.device, dtype=torch.int32).contiguous()
        if n < self.N:
            padded = torch.zeros(k, self.N, E, device=memory.device, dtype=torch.float32)
            padded[:, :n] = memory
            memory = padded
        lens = None
        if lengths is not None:
            lens = torch.as_tensor(lengths).reshape(-1).to(device=self.device, dtype=torch.int64).contiguous()
            if lens.numel() != k:
                raise ValueError(f"genvox_b200: lengths needs one entry per utterance ({k}), got {lens.numel()}")
        first = self._s.submitted
        _native.check(self._lib.gvx_dec_session_submit(C.byref(self._dims), C.byref(self._weights), _ptr(self._packed),
                                                       C.byref(self._s), _ptr(memory), _ptr(lens), _ptr(caps), k,
                                                       _ptr(self._work), _stream()),
                      "gvx_dec_session_submit")
        return list(range(first, first + k))

    def _chunk_buffers(self, steps):
        if steps > self._chunk_steps:
            S, dev = self.slots, self.device
            self._frames = torch.empty(steps, S, self.n_mels + 1, device=dev, dtype=torch.float32)
            self._align = torch.empty(steps, S, self.N, device=dev, dtype=torch.float32) if self.return_alignments else None
            # the int tags in one buffer, read back with one copy: utt [steps][S], frame [steps][S] (int32), last (int8)
            self._tags = torch.empty(steps * S * 9, device=dev, dtype=torch.uint8)
            self._chunk_steps = steps
        return self._frames, self._align, self._tags

    def step(self, steps=16):
        """Run up to `steps` decoder steps.  Returns (chunks, finished): chunks = {id: (mel [n_mels, j], gate [j],
        align [j, N] or None)} with the j new frames of every utterance that advanced in this call, in frame order;
        finished = {id: n_frames} for the utterances whose last frame is among them."""
        self._check_weights()
        steps = int(steps)
        if steps < 1:
            raise ValueError(f"genvox_b200: steps must be positive, got {steps}")
        frames, align, tags = self._chunk_buffers(steps)
        K, S = self._chunk_steps, self.slots
        utt, frame = tags[:4 * K * S].view(torch.int32), tags[4 * K * S:8 * K * S].view(torch.int32)
        last = tags[8 * K * S:].view(torch.int8)
        ran = C.c_int(0)
        _native.check(self._lib.gvx_dec_session_step(C.byref(self._dims), C.byref(self._weights), _ptr(self._packed),
                                                     C.byref(self._s), steps, _ptr(frames), _ptr(align), _ptr(utt),
                                                     _ptr(frame), _ptr(last), C.byref(ran), _ptr(self._work), _stream()),
                      "gvx_dec_session_step")
        n = int(ran.value) * S          # rows [step][slot] written by this call
        if n == 0:
            return {}, {}
        host = tags.cpu().numpy()
        u = host[:4 * K * S].view(np.int32)[:n]
        f = host[4 * K * S:8 * K * S].view(np.int32)[:n]
        lst = host[8 * K * S:].view(np.int8)[:n]
        rows = np.nonzero(u >= 0)[0]
        order = rows[np.lexsort((f[rows], u[rows]))]          # by (id, frame)
        ids, counts = np.unique(u[order], return_counts=True)
        perm = torch.from_numpy(order.astype(np.int64)).to(self.device)
        counts = counts.tolist()
        got = torch.split(frames.view(K * S, self.n_mels + 1).index_select(0, perm), counts)
        got_align = torch.split(align.view(K * S, self.N).index_select(0, perm), counts) if align is not None else [None] * len(counts)
        chunks = {uid: (piece[:, :self.n_mels].t(), piece[:, self.n_mels], a) for uid, piece, a in zip(ids.tolist(), got, got_align)}
        done = np.nonzero((u >= 0) & (lst != 0))[0]
        finished = {int(u[r]): int(f[r]) + 1 for r in done}
        return chunks, finished
