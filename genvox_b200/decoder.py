"""Host-side mirror of the reference Decoder (/root/reference/models/tts/tacotron2.py:258-414).

Same constructor, same `state_dict`, same `forward(memory, decoder_inputs, memory_lengths)` and
`inference(memory)` signatures and return values — but every step of the recurrence runs in the
hand-written sm_100a kernels behind the C ABI (include/genvox_b200.h).  PyTorch is used for
device memory, streams and autograd plumbing only.  There is no CPU path: non-CUDA inputs raise.
"""
import ctypes as C

import torch
from torch import nn

from . import _native
from .containers import AttentionParams, LinearParams, PrenetParams


def _ptr(t):
    return C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p(0)


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _f32c(t, name):
    if not t.is_cuda:
        raise RuntimeError(f"genvox_b200: `{name}` must be a CUDA tensor (there is no CPU fallback)")
    if t.dtype != torch.float32:
        raise RuntimeError(f"genvox_b200: `{name}` must be float32, got {t.dtype}")
    return t.contiguous()


def _buffer(nbytes, device):
    return torch.empty((nbytes + 3) // 4, dtype=torch.float32, device=device)


class _TeacherForced(torch.autograd.Function):
    """Decoder.forward (tacotron2.py:365-388) / BPTT (loss.backward(), :520) through the C ABI."""

    @staticmethod
    def forward(ctx, dec, memory, mel_in, lengths, seed, *params):
        lib = _native.load()
        B, N, _ = memory.shape
        T = mel_in.shape[2]
        dev = memory.device
        dims, weights, packed = dec._native_state(params)
        mel = torch.empty(B, dec.n_mel_channels, T, device=dev, dtype=torch.float32)
        gate = torch.empty(B, T, device=dev, dtype=torch.float32)
        align = torch.empty(B, T, N, device=dev, dtype=torch.float32)
        stash = _buffer(lib.gvx_dec_stash_bytes(C.byref(dims), B, N, T), dev)
        _native.check(lib.gvx_dec_train_fwd(C.byref(dims), C.byref(weights), _ptr(packed), _ptr(memory), _ptr(mel_in),
                                            _ptr(lengths), B, N, T, seed, int(dec.training), dec.dropout_row_offset,
                                            _ptr(mel), _ptr(gate), _ptr(align), _ptr(stash), _stream()),
                      "gvx_dec_train_fwd")
        ctx.dec, ctx.seed, ctx.training, ctx.row_offset = dec, seed, int(dec.training), dec.dropout_row_offset
        ctx.shape = (B, N, T)
        ctx.save_for_backward(memory, lengths if lengths is not None else torch.empty(0, device=dev), stash, packed, *params)
        ctx.has_lengths = lengths is not None
        ctx.set_materialize_grads(False)
        return mel, gate, align

    @staticmethod
    def backward(ctx, d_mel, d_gate, d_align):
        lib = _native.load()
        memory, lengths, stash, packed, *params = ctx.saved_tensors
        lengths = lengths if ctx.has_lengths else None
        dec = ctx.dec
        B, N, T = ctx.shape
        dev = memory.device
        dims = dec._dims()
        weights = dec._weights_struct(params)
        d_mel = _f32c(d_mel, "d_mel") if d_mel is not None else torch.zeros(B, dec.n_mel_channels, T, device=dev)
        d_gate = _f32c(d_gate, "d_gate") if d_gate is not None else torch.zeros(B, T, device=dev)
        d_align = _f32c(d_align, "d_align") if d_align is not None else None
        grads = [torch.empty_like(p) for p in params]
        gstruct = _native.GvxGrads(*[_ptr(g) for g in grads])
        d_memory = torch.empty_like(memory)
        work = _buffer(lib.gvx_dec_bwd_workspace_bytes(C.byref(dims), B, N, T), dev)
        _native.check(lib.gvx_dec_train_bwd(C.byref(dims), C.byref(weights), _ptr(packed), _ptr(memory), _ptr(lengths),
                                            B, N, T, ctx.seed, ctx.training, ctx.row_offset, _ptr(d_mel), _ptr(d_gate),
                                            _ptr(d_align), _ptr(stash), _ptr(work), C.byref(gstruct), _ptr(d_memory),
                                            _stream()),
                      "gvx_dec_train_bwd")
        return (None, d_memory, None, None, None, *grads)


class Decoder(nn.Module):
    """Drop-in for the reference `Decoder` (tacotron2.py:258-301): identical constructor arguments,
    parameter names / shapes / initialisers (so checkpoints load either way, checkpoint_manager.py:35-37)."""

    def __init__(self, n_mels, encoder_embedding_dim, decoder_rnn_dim, prenet_dim, max_decoder_steps, gate_threshold,
                 p_attention_dropout, p_decoder_dropout, attention_rnn_dim, attention_dim,
                 attention_location_n_filters, attention_location_kernel_size):
        super().__init__()
        self.n_mel_channels = n_mels
        self.encoder_embedding_dim = encoder_embedding_dim
        self.decoder_rnn_dim = decoder_rnn_dim
        self.prenet_dim = prenet_dim
        self.max_decoder_steps = max_decoder_steps
        self.gate_threshold = gate_threshold
        self.p_attention_dropout = p_attention_dropout
        self.p_decoder_dropout = p_decoder_dropout
        self.attention_rnn_dim = attention_rnn_dim
        self.attention_dim = attention_dim
        self.attention_location_n_filters = attention_location_n_filters
        self.attention_location_kernel_size = attention_location_kernel_size

        # same construction order as the reference => same parameters under the same torch seed
        self.prenet = PrenetParams(n_mels, [prenet_dim, prenet_dim])
        self.attention_rnn = nn.LSTMCell(prenet_dim + encoder_embedding_dim, attention_rnn_dim)
        self.attention_layer = AttentionParams(attention_rnn_dim, encoder_embedding_dim, attention_dim,
                                               attention_location_n_filters, attention_location_kernel_size)
        self.decoder_rnn = nn.LSTMCell(attention_rnn_dim + encoder_embedding_dim, decoder_rnn_dim, 1)
        self.linear_projection = LinearParams(decoder_rnn_dim + encoder_embedding_dim, n_mels)
        self.gate_layer = LinearParams(decoder_rnn_dim + encoder_embedding_dim, 1, bias=True, w_init_gain="sigmoid")

        # arithmetic of the recurrent GEMMs: "fp32" (FFMA, parity mode) or "bf16" (tcgen05, fp32 accumulate)
        self.precision = "fp32"
        # dropout stream control (the reference draws from torch's global RNG, tacotron2.py:143,341,358)
        self.dropout_row_offset = 0        # data parallel: first row of this rank in the global batch
        self._forced_seed = None
        self.last_dropout_seed = None
        self.last_n_frames = None
        self.last_steps_run = None      # decoder steps of the last inference_continuous call
        self._pack_key = None
        self._packed = None
        self._pack_epoch = 0          # bumped by invalidate_packed()

    # ------------------------------------------------------------------ plumbing
    def set_dropout_seed(self, seed):
        """Use exactly `seed` for the next forward()/inference() call (tests, reproducibility)."""
        self._forced_seed = int(seed)

    def _next_seed(self):
        if self._forced_seed is not None:
            seed, self._forced_seed = self._forced_seed, None
        else:   # CPU generator: follows torch.manual_seed, no device sync
            seed = int(torch.randint(0, 2 ** 62, (1,), dtype=torch.int64).item())
        self.last_dropout_seed = seed
        return seed

    def _ordered_params(self):
        sd = dict(self.named_parameters())
        return [sd[key] for _, key in _native.PARAM_FIELDS]

    def _dims(self):
        return _native.GvxDims(self.n_mel_channels, self.encoder_embedding_dim, self.attention_rnn_dim,
                               self.decoder_rnn_dim, self.prenet_dim, self.attention_dim,
                               self.attention_location_n_filters, self.attention_location_kernel_size,
                               float(self.p_attention_dropout), float(self.p_decoder_dropout),
                               {"fp32": 0, "bf16": 1}[self.precision])

    @staticmethod
    def _weights_struct(params):
        return _native.GvxWeights(*[_ptr(p) for p in params])

    def invalidate_packed(self):
        """Force a repack of the kernel-side weight images on the next call.  Needed after in-place edits that bypass autograd's
        version counter (`p.data.copy_(...)`, an EMA swap through `.data`, manual re-initialisation): the cache key is
        (data_ptr, version) per parameter and `.data` writes do not bump the version."""
        self._pack_epoch += 1

    def _last_step_gate_fired(self, gate, n_frames, steps):
        """True when every row that reached the last allowed step did so because its gate fired there (then the reference's
        loop ends through the gate `break`, tacotron2.py:405-406, without the max-steps warning)."""
        rows = n_frames >= steps
        if not bool(rows.any()):
            return True
        return bool((torch.sigmoid(gate[rows, steps - 1]) > self.gate_threshold).all())

    def _packed_key(self, params):
        """cache key of the packed weights: precision, invalidate_packed() epoch, (data_ptr, version) per parameter"""
        return (self.precision, self._pack_epoch) + tuple((p.data_ptr(), p._version) for p in params)

    def _native_state(self, params):
        """(dims, weights struct, packed weights) — repacks when any parameter changed."""
        lib = _native.load()
        for p in params:
            if not p.is_cuda or p.dtype != torch.float32 or not p.is_contiguous():
                raise RuntimeError("genvox_b200: decoder parameters must be contiguous float32 CUDA tensors")
        dims = self._dims()
        weights = self._weights_struct(params)
        key = self._packed_key(params)
        if key != self._pack_key:
            nbytes = lib.gvx_dec_packed_bytes(C.byref(dims))
            if nbytes == 0:
                _native.check(1, "gvx_dec_packed_bytes")
            # a FRESH buffer per repack: an autograd graph of an earlier forward may still hold the previous one
            # (save_for_backward), and its backward must see the weights that forward used
            self._packed = _buffer(nbytes, params[0].device)
            _native.check(lib.gvx_dec_pack_weights(C.byref(dims), C.byref(weights), _ptr(self._packed), _stream()),
                          "gvx_dec_pack_weights")
            self._pack_key = key
        return dims, weights, self._packed

    # ------------------------------------------------------------------ reference API
    def forward(self, memory, decoder_inputs, memory_lengths):
        """memory [B,N,E], decoder_inputs [B,n_mels,T], memory_lengths [B] ->
        (mel [B,n_mels,T], gate [B,T], alignments [B,T,N])   — tacotron2.py:365-388."""
        memory = _f32c(memory, "memory")
        mel_in = _f32c(decoder_inputs, "decoder_inputs")
        lengths = None
        if memory_lengths is not None:
            lengths = memory_lengths.to(device=memory.device, dtype=torch.int64).contiguous()
        params = [p if p.is_contiguous() else p.contiguous() for p in self._ordered_params()]
        return _TeacherForced.apply(self, memory, mel_in, lengths, self._next_seed(), *params)

    @torch.no_grad()
    def inference(self, memory, memory_lengths=None, ignore_gate=False, max_decoder_steps=None):
        """Autoregressive decoding, tacotron2.py:390-414, for B >= 1 rows.  Returns the reference's triple
        (mel [B,n_mels,Tmax], gate [B,Tmax], alignments [B,Tmax,N]) with Tmax = max over rows of the per-row
        frame count; the per-row counts are left in `self.last_n_frames` (int32 [B], device)."""
        lib = _native.load()
        memory = _f32c(memory, "memory")
        B, N, _ = memory.shape
        dev = memory.device
        steps = int(max_decoder_steps if max_decoder_steps is not None else self.max_decoder_steps)
        lengths = None
        if memory_lengths is not None:
            lengths = memory_lengths.to(device=dev, dtype=torch.int64).contiguous()
        params = [p.detach() for p in self._ordered_params()]
        dims, weights, packed = self._native_state(params)
        mel = torch.empty(B, self.n_mel_channels, steps, device=dev, dtype=torch.float32)
        gate = torch.empty(B, steps, device=dev, dtype=torch.float32)
        align = torch.empty(B, steps, N, device=dev, dtype=torch.float32)
        n_frames = torch.empty(B, device=dev, dtype=torch.int32)
        work = _buffer(lib.gvx_dec_infer_workspace_bytes(C.byref(dims), B, N, steps), dev)
        ran = C.c_int(0)
        _native.check(lib.gvx_dec_infer(C.byref(dims), C.byref(weights), _ptr(packed), _ptr(memory), _ptr(lengths), B, N,
                                        steps, float(self.gate_threshold), int(bool(ignore_gate)), self._next_seed(),
                                        int(self.training), self.dropout_row_offset, _ptr(mel), _ptr(gate), _ptr(align),
                                        _ptr(n_frames), C.byref(ran), _ptr(work), _stream()),
                      "gvx_dec_infer")
        self.last_n_frames = n_frames
        tmax = steps if ignore_gate else int(n_frames.max().item())
        # tacotron2.py:405-409 breaks on the gate BEFORE it tests the step count: a row whose gate fires on the last allowed
        # step does not warn.  `ran` counts the decoder steps executed: the loop ran out only if no stop ended it.
        if not ignore_gate and tmax >= steps and int(ran.value) >= steps and not self._last_step_gate_fired(gate, n_frames, steps):
            print("Warning! Reached max decoder steps")      # tacotron2.py:408
        return mel[:, :, :tmax], gate[:, :tmax], align[:, :tmax]

    @torch.no_grad()
    def inference_continuous(self, memory, memory_lengths, slots=64, max_decoder_steps=None, frame_caps=None, ignore_gate=False,
                             return_alignments=True):
        """Continuous batching: decode the U utterances of `memory` [U,N,E] through `slots` decoder rows; a row whose utterance
        stops takes the next one of the queue on the device (include/genvox_b200.h, gvx_dec_infer_continuous).  Utterance u
        stops at its first gate over the threshold or after min(max_decoder_steps, frame_caps[u]) frames, and draws the prenet
        dropout of row u + dropout_row_offset.  Returns (mel [U,n_mels,Tmax], gate [U,Tmax], alignments [U,Tmax,N] or None)
        with Tmax = max over utterances of the frame count; frames past an utterance's count are zero.  The counts are left
        in `self.last_n_frames` (int32 [U], device).  Eval mode only."""
        lib = _native.load()
        steps = int(max_decoder_steps if max_decoder_steps is not None else self.max_decoder_steps)
        if self.training:
            raise RuntimeError("genvox_b200: inference_continuous runs in eval mode only (call .eval())")
        limit = 128 if self.precision == "bf16" else None
        if int(slots) < 1 or (limit is not None and int(slots) > limit):
            raise ValueError(f"genvox_b200: slots must be in 1 .. {limit or 'inf'} in {self.precision} mode, got {slots}")
        if steps < 1:
            raise ValueError(f"genvox_b200: max_decoder_steps must be positive, got {steps}")
        caps = None
        if frame_caps is not None:
            caps = torch.as_tensor(frame_caps).reshape(-1)
            if caps.numel() != memory.shape[0]:
                raise ValueError(f"genvox_b200: frame_caps needs one entry per utterance ({memory.shape[0]}), got {caps.numel()}")
            if bool((caps < 1).any()) or bool((caps > steps).any()):
                raise ValueError(f"genvox_b200: frame_caps must lie in 1 .. max_decoder_steps ({steps})")
        memory = _f32c(memory, "memory")
        U, N, _ = memory.shape
        dev = memory.device
        lengths = None
        if memory_lengths is not None:
            lengths = memory_lengths.to(device=dev, dtype=torch.int64).contiguous()
        if caps is not None:
            caps = caps.to(device=dev, dtype=torch.int32).contiguous()
        params = [p.detach() for p in self._ordered_params()]
        dims, weights, packed = self._native_state(params)
        mel = torch.zeros(U, self.n_mel_channels, steps, device=dev, dtype=torch.float32)
        gate = torch.zeros(U, steps, device=dev, dtype=torch.float32)
        align = torch.zeros(U, steps, N, device=dev, dtype=torch.float32) if return_alignments else None
        n_frames = torch.empty(U, device=dev, dtype=torch.int32)
        nbytes = lib.gvx_dec_infer_continuous_workspace_bytes(C.byref(dims), U, N, int(slots))
        if nbytes == 0:
            _native.check(1, "gvx_dec_infer_continuous_workspace_bytes")
        work = _buffer(nbytes, dev)
        ran = C.c_longlong(0)
        _native.check(lib.gvx_dec_infer_continuous(C.byref(dims), C.byref(weights), _ptr(packed), _ptr(memory), _ptr(lengths), U, N,
                                                   int(slots), steps, _ptr(caps), float(self.gate_threshold), int(bool(ignore_gate)),
                                                   self._next_seed(), self.dropout_row_offset, _ptr(mel), _ptr(gate), _ptr(align),
                                                   _ptr(n_frames), C.byref(ran), _ptr(work), _stream()),
                      "gvx_dec_infer_continuous")
        self.last_n_frames = n_frames
        self.last_steps_run = int(ran.value)
        tmax = int(n_frames.max().item())
        # as in inference(): an utterance that reached the last allowed step warns unless its gate fired there
        if not ignore_gate and tmax >= steps and not self._last_step_gate_fired(gate, n_frames, steps):
            print("Warning! Reached max decoder steps")      # tacotron2.py:408
        return mel[:, :, :tmax], gate[:, :tmax], (align[:, :tmax] if align is not None else None)

    def session(self, N, slots=64, capacity=1024, max_decoder_steps=None, ignore_gate=False, return_alignments=True):
        """A decoder session (genvox_b200.session.DecoderSession): `slots` decoder rows kept alive between calls, utterances
        of up to N tokens submitted at any time between calls and decoded through those rows, frames returned per step call.
        Up to `capacity` utterances may wait in its queue.  Utterance `id` decodes bit-identically to row r of a static
        `inference` call with the same slots rows, N, seed and precision, id in row r and dropout_row_offset =
        id + dropout_row_offset - r.  Eval mode only; the parameters must not change while the session runs."""
        from .session import DecoderSession
        return DecoderSession(self, N, slots=slots, capacity=capacity, max_decoder_steps=max_decoder_steps,
                              ignore_gate=ignore_gate, return_alignments=return_alignments)


def decoder_kwargs_from(ref_decoder):
    """Constructor arguments recovered from a reference Decoder instance (tacotron2.py:274-300)."""
    att = ref_decoder.attention_layer
    conv = att.location_layer.location_conv.conv
    return dict(
        n_mels=ref_decoder.n_mel_channels, encoder_embedding_dim=ref_decoder.encoder_embedding_dim,
        decoder_rnn_dim=ref_decoder.decoder_rnn_dim, prenet_dim=ref_decoder.prenet_dim,
        max_decoder_steps=ref_decoder.max_decoder_steps, gate_threshold=ref_decoder.gate_threshold,
        p_attention_dropout=ref_decoder.p_attention_dropout, p_decoder_dropout=ref_decoder.p_decoder_dropout,
        attention_rnn_dim=ref_decoder.attention_rnn_dim,
        attention_dim=att.query_layer.linear_layer.out_features,
        attention_location_n_filters=conv.out_channels, attention_location_kernel_size=conv.kernel_size[0])


def install(model, precision="fp32"):
    """Swap `model.decoder` (a reference Tacotron2, tacotron2.py:416-448) for the B200-native Decoder,
    keeping its parameters.  Tacotron2.forward/inference, the Trainer and the Synthesizer are untouched."""
    ref = model.decoder
    new = Decoder(**decoder_kwargs_from(ref))
    new.precision = precision
    new.load_state_dict(ref.state_dict(), strict=True)
    p = next(ref.parameters())
    new.to(device=p.device, dtype=p.dtype)
    new.train(ref.training)
    model.decoder = new
    return model
