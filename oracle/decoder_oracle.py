"""TEST INFRASTRUCTURE — CPU oracle of the GenVox Tacotron2 decoder recurrence.

A functional torch-CPU restatement (fp32 or fp64) of
/root/reference/models/tts/tacotron2.py:17-144 and :258-414.  It is *not* the product
and is never on the product path: only tests/, __graft_entry__.smoke() and bench.py's
cpu_baseline / --impl reference legs import it.

Why torch and not numpy: the path is floating point and the reference's arithmetic
*is* torch's (SURVEY.md §8c); staying on torch CPU ops keeps the oracle's rounding
identical to the reference's own CPU path and gives the BPTT reference for free
(torch.autograd over this graph == `loss.backward()` at tacotron2.py:520).

Pin: tests/golden/*.npz hold outputs of the UNMODIFIED reference modules (run by
oracle/make_golden.py in the build container) on the same weights, inputs and dropout
masks; tests/test_oracle_golden.py checks this file against them.

Dropout: masks come from oracle/philox.py (see its header) instead of torch's RNG.
"""
from typing import Dict, Optional

import numpy as np
import torch
import torch.nn.functional as F

from . import philox


# ---- optional bf16 semantics of the product's bf16 mode (gate / query / projection GEMM operands rounded to
# bf16, gradients of those GEMM outputs rounded to bf16 in backward; everything else in the working dtype)
_BF16 = False
_BF16_MEMORY = False


class bf16_semantics:
    """with O.bf16_semantics(): ...  — the oracle then mirrors genvox_b200's bf16 mode rounding points.
    round_memory=True adds the one extra rounding point of the fused persistent attention chain
    (genvox_b200/csrc/gvx_fused_fwd.cuh): the context bmm (tacotron2.py:127) reads a bf16 copy of the encoder memory."""

    def __init__(self, round_memory: bool = False):
        self.round_memory = round_memory

    def __enter__(self):
        global _BF16, _BF16_MEMORY
        self.prev, _BF16 = (_BF16, _BF16_MEMORY), True
        _BF16_MEMORY = self.round_memory

    def __exit__(self, *exc):
        global _BF16, _BF16_MEMORY
        _BF16, _BF16_MEMORY = self.prev


class _RoundFwd(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x):
        return x.to(torch.bfloat16).to(x.dtype)

    @staticmethod
    def backward(ctx, g):
        return g


class _RoundBwd(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x):
        return x.view_as(x)

    @staticmethod
    def backward(ctx, g):
        return g.to(torch.bfloat16).to(g.dtype)


def _rf(x):
    return _RoundFwd.apply(x) if _BF16 else x


def _rb(x):
    return _RoundBwd.apply(x) if (_BF16 and x.requires_grad) else x


def _t(x, dtype):
    if isinstance(x, torch.Tensor):
        return x.to(dtype) if x.is_floating_point() else x
    return torch.as_tensor(np.asarray(x)).to(dtype)


def as_params(weights: Dict[str, np.ndarray], dtype=torch.float32, requires_grad=False) -> Dict[str, torch.Tensor]:
    out = {}
    for k, v in weights.items():
        t = _t(v, dtype).clone()
        t.requires_grad_(requires_grad)
        out[k] = t
    return out


def get_mask_from_lengths(lengths: torch.Tensor, max_len: Optional[int] = None) -> torch.Tensor:
    """True = padded position.  tacotron2.py:17-21."""
    if max_len is None:
        max_len = int(lengths.max())
    ids = torch.arange(max_len, dtype=lengths.dtype)
    return ids[None, :] >= lengths[:, None]


def philox_dropout(x: torch.Tensor, p: float, on: bool, seed: int, site: int, t: int, row_offset: int = 0):
    """F.dropout(x, p, training=on) with the mask taken from the shared Philox stream.
    x: [rows, width].  tacotron2.py:143 (prenet, always on), :341, :358."""
    if not on or p == 0.0:
        return x
    keep = philox.keep_mask(seed, site, t, x.shape[0], x.shape[1], p, row_offset)
    m = torch.from_numpy(keep).to(x.dtype) * float(philox.dropout_scale(p))
    return x * m


def prenet(P, frames: torch.Tensor, seed: int, t0: int = 0, row_offset: int = 0) -> torch.Tensor:
    """Prenet.forward, tacotron2.py:140-144.  frames: [F, B, n_mels] -> [F, B, prenet_dim].
    Frame f uses stream index t = t0 + f; dropout p = 0.5 is on in every mode."""
    outs = []
    for f in range(frames.shape[0]):
        x = frames[f]
        for layer, site in ((0, philox.SITE_PRENET0), (1, philox.SITE_PRENET1)):
            w = P[f"prenet.layers.{layer}.linear_layer.weight"]
            x = philox_dropout(F.relu(F.linear(x, w)), 0.5, True, seed, site, t0 + f, row_offset)
        outs.append(x)
    return torch.stack(outs)


def lstm_cell(x, h, c, w_ih, w_hh, b_ih, b_hh):
    """nn.LSTMCell (tacotron2.py:286,294,340,357): gate row order i, f, g, o."""
    gates = _rb(F.linear(_rf(x), _rf(w_ih), b_ih) + F.linear(_rf(h), _rf(w_hh), b_hh))
    i, f, g, o = gates.chunk(4, dim=1)
    i, f, g, o = torch.sigmoid(i), torch.sigmoid(f), torch.tanh(g), torch.sigmoid(o)
    c_new = f * c + i * g
    return o * torch.tanh(c_new), c_new


def location_features(P, w_prev, w_cum):
    """LocationLayer.forward, tacotron2.py:48-53.  [B,N],[B,N] -> [B,N,att_dim]."""
    wc = P["attention_layer.location_layer.location_conv.conv.weight"]
    wd = P["attention_layer.location_layer.location_dense.linear_layer.weight"]
    cat = torch.stack((w_prev, w_cum), dim=1)                         # tacotron2.py:344
    conv = F.conv1d(cat, wc, padding=(wc.shape[2] - 1) // 2)          # tacotron2.py:31-39,50
    return F.linear(conv.transpose(1, 2), wd)                         # :51-52


def attention(P, h_att, memory, processed_memory, w_prev, w_cum, mask):
    """Attention.forward + get_alignment_energies, tacotron2.py:89-129."""
    q = _rb(F.linear(_rf(h_att), _rf(P["attention_layer.query_layer.linear_layer.weight"]))).unsqueeze(1)   # :98
    loc = location_features(P, w_prev, w_cum)                                                # :99
    e = F.linear(torch.tanh(q + loc + processed_memory),
                 P["attention_layer.v.linear_layer.weight"]).squeeze(-1)                     # :102-103
    if mask is not None:
        e = e.masked_fill(mask, float("-inf"))      # :125 (done on .data there: no grad through masked slots either way)
    w = F.softmax(e, dim=1)                          # :126
    ctx = torch.bmm(w.unsqueeze(1), _rf(memory) if _BF16_MEMORY else memory).squeeze(1)   # :127-128
    return ctx, w


class DecoderState:
    """initialize_decoder_states, tacotron2.py:303-315."""

    def __init__(self, P, memory, mask, dims):
        B, N = memory.shape[0], memory.shape[1]
        z = lambda n: memory.new_zeros(B, n)
        self.h_att, self.c_att = z(dims["attention_rnn_dim"]), z(dims["attention_rnn_dim"])
        self.h_dec, self.c_dec = z(dims["decoder_rnn_dim"]), z(dims["decoder_rnn_dim"])
        self.w, self.w_cum = z(N), z(N)
        self.ctx = z(memory.shape[2])
        self.memory = memory
        self.processed_memory = F.linear(memory, P["attention_layer.memory_layer.linear_layer.weight"])  # :314
        self.mask = mask


def decode_step(P, S: DecoderState, prenet_out, t: int, training: bool, p_att: float, p_dec: float,
                seed: int, row_offset: int = 0):
    """Decoder.decode, tacotron2.py:333-363.  Returns (mel_t [B,n_mels], gate_t [B], w_t [B,N])."""
    x = torch.cat((prenet_out, S.ctx), -1)                                                  # :338
    S.h_att, S.c_att = lstm_cell(x, S.h_att, S.c_att, P["attention_rnn.weight_ih"], P["attention_rnn.weight_hh"],
                                 P["attention_rnn.bias_ih"], P["attention_rnn.bias_hh"])    # :340
    S.h_att = philox_dropout(S.h_att, p_att, training, seed, philox.SITE_ATT, t, row_offset)  # :341 (carried)
    S.ctx, S.w = attention(P, S.h_att, S.memory, S.processed_memory, S.w, S.w_cum, S.mask)  # :344-352
    S.w_cum = S.w_cum + S.w                                                                 # :353
    x = torch.cat((S.h_att, S.ctx), -1)                                                     # :355
    S.h_dec, S.c_dec = lstm_cell(x, S.h_dec, S.c_dec, P["decoder_rnn.weight_ih"], P["decoder_rnn.weight_hh"],
                                 P["decoder_rnn.bias_ih"], P["decoder_rnn.bias_hh"])        # :357
    S.h_dec = philox_dropout(S.h_dec, p_dec, training, seed, philox.SITE_DEC, t, row_offset)  # :358 (carried)
    hc = torch.cat((S.h_dec, S.ctx), dim=1)                                                 # :360
    mel = F.linear(_rf(hc), _rf(P["linear_projection.linear_layer.weight"]), P["linear_projection.linear_layer.bias"])  # :361
    gate = F.linear(_rf(hc), _rf(P["gate_layer.linear_layer.weight"]), P["gate_layer.linear_layer.bias"])               # :362
    return mel, gate.squeeze(1), S.w


def _dims_of(P):
    return {
        "attention_rnn_dim": P["attention_rnn.weight_hh"].shape[1],
        "decoder_rnn_dim": P["decoder_rnn.weight_hh"].shape[1],
        "n_mels": P["linear_projection.linear_layer.weight"].shape[0],
    }


def forward_teacher(P, memory, mel_in, memory_lengths, seed: int, training: bool = True,
                    p_att: float = 0.1, p_dec: float = 0.1, row_offset: int = 0):
    """Decoder.forward, tacotron2.py:365-388.
    memory [B,N,E], mel_in [B,n_mels,T], memory_lengths [B] int64 ->
    mel [B,n_mels,T], gate [B,T], align [B,T,N]."""
    dims = _dims_of(P)
    B, T = mel_in.shape[0], mel_in.shape[2]
    go = memory.new_zeros(1, B, dims["n_mels"])                              # :370
    frames = torch.cat((go, mel_in.permute(2, 0, 1)), dim=0)                 # :317-320,:371-372  [T+1,B,M]
    pre = prenet(P, frames, seed, 0, row_offset)                             # :373 (all T+1 frames draw masks)
    mask = get_mask_from_lengths(torch.as_tensor(memory_lengths), memory.shape[1])
    S = DecoderState(P, memory, mask, dims)                                  # :375
    mels, gates, aligns = [], [], []
    for t in range(T):                                                        # :378-384
        m, g, w = decode_step(P, S, pre[t], t, training, p_att, p_dec, seed, row_offset)
        mels.append(m), gates.append(g), aligns.append(w)
    mel = torch.stack(mels).permute(1, 2, 0)                                  # :322-331
    gate = torch.stack(gates).transpose(0, 1)
    align = torch.stack(aligns).transpose(0, 1)
    return mel, gate, align


@torch.no_grad()
def inference(P, memory, memory_lengths=None, max_decoder_steps: int = 1000, gate_threshold: float = 0.5,
              ignore_gate: bool = False, seed: int = 0, training: bool = False,
              p_att: float = 0.1, p_dec: float = 0.1, row_offset: int = 0):
    """Decoder.inference, tacotron2.py:390-414, generalised to B >= 1 rows.

    The reference loop is B = 1 only (:405 raises for B > 1, SURVEY.md §3.2); per row the
    rule is the same: stop after the first frame whose sigmoid(gate) > threshold
    (strict, frame included, :405) or at max_decoder_steps (:407).  Rows that stopped keep
    being decoded until every row has stopped (their later frames are the continued
    recurrence); `n_frames[b]` is the per-row frame count the reference would return.
    Returns mel [B,n_mels,Tmax], gate [B,Tmax], align [B,Tmax,N], n_frames [B] int64."""
    dims = _dims_of(P)
    B = memory.shape[0]
    mask = None
    if memory_lengths is not None:
        mask = get_mask_from_lengths(torch.as_tensor(memory_lengths), memory.shape[1])
    S = DecoderState(P, memory, mask, dims)                                   # :394
    x = memory.new_zeros(B, dims["n_mels"])                                   # :392
    n_frames = torch.full([B], -1, dtype=torch.int64)
    mels, gates, aligns = [], [], []
    t = 0
    while True:
        pre = prenet(P, x[None], seed, t, row_offset)[0]                      # :398 (dropout on in eval too)
        m, g, w = decode_step(P, S, pre, t, training, p_att, p_dec, seed, row_offset)
        mels.append(m), gates.append(g), aligns.append(w)
        t += 1
        if not ignore_gate:
            fired = (torch.sigmoid(g) > gate_threshold) & (n_frames < 0)      # :405
            n_frames[fired] = t
        if t >= max_decoder_steps:                                            # :407
            n_frames[n_frames < 0] = t
        if bool((n_frames >= 0).all()):
            break
        x = m                                                                 # :410
    mel = torch.stack(mels).permute(1, 2, 0)
    gate = torch.stack(gates).transpose(0, 1)
    align = torch.stack(aligns).transpose(0, 1)
    return mel, gate, align, n_frames


def loss_and_grads(P, memory, mel_in, memory_lengths, r_mel, r_gate, seed, training=True,
                   p_att=0.1, p_dec=0.1, r_align=None, row_offset: int = 0):
    """BPTT reference (a13): L = <mel, r_mel> + <gate, r_gate> (+ <align, r_align>), gradients
    to every parameter and to `memory` by torch autograd — what loss.backward()
    (tacotron2.py:520) does to the decoder graph for upstream gradients r_*.
    row_offset: the rows' first index in the dropout stream (a data-parallel rank's share of the batch)."""
    P = {k: v.detach().clone().requires_grad_(True) for k, v in P.items()}
    memory = memory.detach().clone().requires_grad_(True)
    mel, gate, align = forward_teacher(P, memory, mel_in, memory_lengths, seed, training, p_att, p_dec, row_offset)
    loss = (mel * r_mel).sum() + (gate * r_gate).sum()
    if r_align is not None:
        loss = loss + (align * r_align).sum()
    loss.backward()
    grads = {k: v.grad if v.grad is not None else torch.zeros_like(v) for k, v in P.items()}
    return (mel.detach(), gate.detach(), align.detach()), grads, memory.grad
