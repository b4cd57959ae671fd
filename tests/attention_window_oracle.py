"""TEST INFRASTRUCTURE — the inference-time attention constraint (include/genvox_b200.h, gvx_dec_*_windowed) on top of the CPU
oracle (oracle/decoder_oracle.py), which it uses unmodified: `attention`, `decode_step` and `inference` below are that
file's functions with one step added, the window mask on the energies.  With window=None they compute exactly what the
oracle computes (tests/test_attention_window_host.py checks that bit for bit).

Rule: last = argmax_n w_prev[b, n] (lowest index on ties, as torch.argmax), or a forced peak; energies of tokens
n < last - backward or n >= last + forward become -inf, in addition to the memory-length mask.  A forced peak sequence
keeps a comparison with the GPU on the same windows where two tokens are near a tie.
"""
import torch
import torch.nn.functional as F

from oracle import decoder_oracle as O
from oracle import philox


def attention(P, h_att, memory, processed_memory, w_prev, w_cum, mask, window=None, peak=None):
    """O.attention (tacotron2.py:89-129) plus the window mask."""
    q = O._rb(F.linear(O._rf(h_att), O._rf(P["attention_layer.query_layer.linear_layer.weight"]))).unsqueeze(1)
    loc = O.location_features(P, w_prev, w_cum)
    e = F.linear(torch.tanh(q + loc + processed_memory), P["attention_layer.v.linear_layer.weight"]).squeeze(-1)
    if mask is not None:
        e = e.masked_fill(mask, float("-inf"))
    if window is not None:
        last = w_prev.argmax(dim=1) if peak is None else torch.as_tensor(peak, dtype=torch.int64).reshape(-1)
        n = torch.arange(e.shape[1])[None, :]
        e = e.masked_fill((n < last[:, None] - window[0]) | (n >= last[:, None] + window[1]), float("-inf"))
    w = F.softmax(e, dim=1)
    ctx = torch.bmm(w.unsqueeze(1), O._rf(memory) if O._BF16_MEMORY else memory).squeeze(1)
    return ctx, w


def decode_step(P, S, prenet_out, t, training, p_att, p_dec, seed, row_offset=0, window=None, peak=None):
    """O.decode_step (tacotron2.py:333-363) with the windowed attention."""
    x = torch.cat((prenet_out, S.ctx), -1)
    S.h_att, S.c_att = O.lstm_cell(x, S.h_att, S.c_att, P["attention_rnn.weight_ih"], P["attention_rnn.weight_hh"],
                                   P["attention_rnn.bias_ih"], P["attention_rnn.bias_hh"])
    S.h_att = O.philox_dropout(S.h_att, p_att, training, seed, philox.SITE_ATT, t, row_offset)
    S.ctx, S.w = attention(P, S.h_att, S.memory, S.processed_memory, S.w, S.w_cum, S.mask, window, peak)
    S.w_cum = S.w_cum + S.w
    x = torch.cat((S.h_att, S.ctx), -1)
    S.h_dec, S.c_dec = O.lstm_cell(x, S.h_dec, S.c_dec, P["decoder_rnn.weight_ih"], P["decoder_rnn.weight_hh"],
                                   P["decoder_rnn.bias_ih"], P["decoder_rnn.bias_hh"])
    S.h_dec = O.philox_dropout(S.h_dec, p_dec, training, seed, philox.SITE_DEC, t, row_offset)
    hc = torch.cat((S.h_dec, S.ctx), dim=1)
    mel = F.linear(O._rf(hc), O._rf(P["linear_projection.linear_layer.weight"]), P["linear_projection.linear_layer.bias"])
    gate = F.linear(O._rf(hc), O._rf(P["gate_layer.linear_layer.weight"]), P["gate_layer.linear_layer.bias"])
    return mel, gate.squeeze(1), S.w


@torch.no_grad()
def inference(P, memory, memory_lengths=None, max_decoder_steps=1000, gate_threshold=0.5, ignore_gate=False, seed=0,
              training=False, p_att=0.1, p_dec=0.1, row_offset=0, window=None, peaks=None):
    """O.inference (tacotron2.py:390-414, B >= 1 rows) with the window; peaks [T][B]: the `last` of step t is peaks[t]
    (None: the argmax of the previous step's weights).  Returns mel, gate, align, n_frames as O.inference does."""
    dims = O._dims_of(P)
    B = memory.shape[0]
    mask = None
    if memory_lengths is not None:
        mask = O.get_mask_from_lengths(torch.as_tensor(memory_lengths), memory.shape[1])
    S = O.DecoderState(P, memory, mask, dims)
    x = memory.new_zeros(B, dims["n_mels"])
    n_frames = torch.full([B], -1, dtype=torch.int64)
    mels, gates, aligns = [], [], []
    t = 0
    while True:
        pre = O.prenet(P, x[None], seed, t, row_offset)[0]
        m, g, w = decode_step(P, S, pre, t, training, p_att, p_dec, seed, row_offset, window,
                              peaks[t] if peaks is not None else None)
        mels.append(m), gates.append(g), aligns.append(w)
        t += 1
        if not ignore_gate:
            fired = (torch.sigmoid(g) > gate_threshold) & (n_frames < 0)
            n_frames[fired] = t
        if t >= max_decoder_steps:
            n_frames[n_frames < 0] = t
        if bool((n_frames >= 0).all()):
            break
        x = m
    return torch.stack(mels).permute(1, 2, 0), torch.stack(gates).transpose(0, 1), torch.stack(aligns).transpose(0, 1), n_frames
