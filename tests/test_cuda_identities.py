"""Exact identities of the decoder, checked at the benchmarked sizes on every training path.

The oracle tests (test_cuda_long.py, test_cuda_fused.py, test_cuda_bf16.py) bound bf16 mode at T = 800 by 3e-2 of max|ref|: rounding
flips compound over hundreds of recurrent steps.  A bound that loose cannot see a reduction that drops one K block or one frame, a
chain that leaks a little into a neighbouring row, or a prefetch that reads the wrong frame.  The decoder has structure that holds
exactly in floating point (or up to fp32 reassociation of a sum) at any length, and that needs no oracle:
  * batch rows never interact (forward: bit-exact; backward: exact zeros, and a row partition of the upstream gradient superposes);
  * teacher forcing is causal (a prefix run is a prefix; the gradient of a loss on the first t0 frames does not see later frames);
  * masked tokens carry exactly zero weight (padding content changes nothing);
  * alignments do not depend on the decoder LSTM;
  * bias gradients are column sums of the upstream gradient; the two LSTM bias gradients are one tensor;
  * the backward only reads the forward's stash: repeated backwards agree, a zero upstream gradient gives zero.

Paths (forced through gvx_debug_option):
  F  fused persistent chains, bf16, configs[2] shape (the benchmark)
  E  fused chains at their edge, bf16: odd batch, largest N of the fused forward
  O  per-step forward + persistent BPTT attention chain, bf16, configs[4] token count
  S  per-step chains, bf16
  P  fp32 mode, configs[0] shape
Only the alignment-gradient and row-offset tests call the CPU oracle, at T <= 12.
"""
import contextlib

import numpy as np
import pytest
import torch

from conftest import rel_err
from oracle import decoder_oracle as O
from oracle import synth
from test_cuda_parity import make_decoder

pytestmark = pytest.mark.gpu

SEED = 4242
# fp32 reassociation of the split-K weight-gradient GEMMs, column sums and post-pass reductions: per tensor, relative to max|g|
REASSOC_TOL = 1e-4
SAME_ROUNDING_FWD_TOL = 5e-3           # the bounds of test_cuda_bf16.py / test_cuda_fused.py
SAME_ROUNDING_GRAD_TOL = 3e-2


class Path:
    def __init__(self, pid, B, N, T, precision, fused):
        self.pid, self.B, self.N, self.T, self.precision, self.fused = pid, B, N, T, precision, fused
        # rows at the batch-half / CTA boundaries of the chains
        self.rows = sorted({0, B // 2 - 1, B // 2, B - 1})

    def __repr__(self):
        return self.pid


PATHS = {p.pid: p for p in (
    Path("F", 64, 150, 800, "bf16", 1),
    Path("E", 33, 160, 96, "bf16", 1),
    Path("O", 32, 300, 256, "bf16", 1),      # N > 160: the forward runs per step, the BPTT attention chain persistent
    Path("S", 64, 150, 200, "bf16", 0),
    Path("P", 16, 120, 600, "fp32", -1),
)}


@contextlib.contextmanager
def forced(path):
    """Force the path's chains for a forward or a backward (the backward re-derives the path: both must see the same)."""
    from genvox_b200 import _native
    lib = _native.load()
    try:
        if path.precision == "bf16":
            _native.check(lib.gvx_debug_option(b"fused", path.fused), "gvx_debug_option")
            _native.check(lib.gvx_debug_option(b"persistent", 1), "gvx_debug_option")
        yield
    finally:
        lib.gvx_debug_option(b"fused", -1)
        lib.gvx_debug_option(b"persistent", -1)


def _sync():
    import genvox_b200
    torch.cuda.synchronize()
    genvox_b200.check_device_errors()


class Fwd:
    """One teacher-forced forward; several backwards run on its graph, so every comparison sees the same forward."""

    def __init__(self, path, dec, memory, mel, lens):
        self.path, self.dec = path, dec
        self.memory = memory.detach().clone().requires_grad_(True)
        dec.set_dropout_seed(SEED)
        with forced(path):
            self.m, self.g, self.a = dec(self.memory, mel, lens)
        _sync()

    def grads(self, r_mel, r_gate, r_align=None):
        """Gradients of <mel, r_mel> + <gate, r_gate> (+ <align, r_align>) to every parameter and to `memory`."""
        outs = [(self.m, r_mel), (self.g, r_gate)] + ([(self.a, r_align)] if r_align is not None else [])
        named = list(self.dec.named_parameters())
        with forced(self.path):
            gr = torch.autograd.grad([o for o, _ in outs], [p for _, p in named] + [self.memory], [r for _, r in outs],
                                     retain_graph=True)
        _sync()
        return dict(zip([k for k, _ in named] + ["memory"], gr))


def _rel(x, ref):
    """max|x - ref| / max|ref| on the device (fp64)."""
    x, ref = x.double(), ref.double()
    return float((x - ref).abs().max() / ref.abs().max().clamp_min(1e-30))


def _rows(x, keep):
    return x[torch.as_tensor(keep, device=x.device)]


class Base:
    def __init__(self, path, dev):
        self.path, self.dev = path, dev
        self.dims = dims = synth.DecoderDims()
        self.dec = make_decoder(dims, synth.make_decoder_weights(31, dims), dev, True)
        self.dec.precision = path.precision
        mem, mel, lens = synth.make_inputs(89, path.B, path.N, path.T, dims, ragged=True)
        self.memory, self.mel, self.lens = (torch.from_numpy(x).to(dev) for x in (mem, mel, lens))
        g = torch.Generator(device=dev).manual_seed(89)
        u = lambda *shape: torch.rand(*shape, generator=g, device=dev) - 0.5
        B, N, T = path.B, path.N, path.T
        self.r_mel, self.r_gate, self.r_align = u(B, dims.n_mels, T), u(B, T), u(B, T, N)
        self.fwd = Fwd(path, self.dec, self.memory, self.mel, self.lens)
        self.full = self.fwd.grads(self.r_mel, self.r_gate)           # the benchmark's loss: d_align = NULL

    def gen(self, seed):
        return torch.Generator(device=self.dev).manual_seed(seed)


@pytest.fixture(scope="module", params=list(PATHS))
def base(request, cuda_device):
    b = Base(PATHS[request.param], cuda_device)
    yield b
    del b
    torch.cuda.empty_cache()


def _perturb_row(memory, mel, lens, r, gen):
    """Row r gets other memory, other mel frames and another length (max(lengths) stays N, as the collate guarantees)."""
    memory, mel, lens = (x.clone() if x is not None else None for x in (memory, mel, lens))
    N = memory.shape[1]
    memory[r] = 0.5 * torch.randn(memory[r].shape, generator=gen, device=memory.device)
    if mel is not None:
        mel[r] = torch.randn(mel[r].shape, generator=gen, device=mel.device)
    if lens is not None:
        if int(lens[r]) < N:
            lens[r] = N
        elif int((lens == N).sum()) > 1:
            lens[r] = N - 23
    return memory, mel, lens


def _padded(memory, lens, gen):
    """memory with the padded tokens (n >= len_b) replaced by other finite values, ~10x the normal scale."""
    out = memory.clone()
    N = memory.shape[1]
    for b, L in enumerate(lens.tolist()):
        if L < N:
            out[b, L:] = 5.0 * torch.randn(out[b, L:].shape, generator=gen, device=memory.device)
    return out


# --------------------------------------------------------------------------- 1. forward row isolation
def test_forward_rows_are_isolated(base):
    """Another memory / mel / length in row r leaves every other row's mel, gate and alignments bit-identical."""
    p = base.path
    ref = (base.fwd.m.detach(), base.fwd.g.detach(), base.fwd.a.detach())
    for r in p.rows:
        mem, mel, lens = _perturb_row(base.memory, base.mel, base.lens, r, base.gen(1000 + r))
        f = Fwd(p, base.dec, mem, mel, lens)
        keep = [b for b in range(p.B) if b != r]
        for name, x, y in zip(("mel", "gate", "align"), (f.m, f.g, f.a), ref):
            assert torch.equal(_rows(x.detach(), keep), _rows(y, keep)), (p.pid, r, name)
            assert not torch.equal(x[r].detach(), y[r]), (p.pid, r, name)       # the perturbation reached row r
        del f
    if p.pid != "F":
        return
    # memory_lengths=None: the same isolation, and the same results as lengths that are all N
    full_n = torch.full_like(base.lens, p.N)
    f0 = Fwd(p, base.dec, base.memory, base.mel, None)
    fn = Fwd(p, base.dec, base.memory, base.mel, full_n)
    for name, x, y in zip(("mel", "gate", "align"), (f0.m, f0.g, f0.a), (fn.m, fn.g, fn.a)):
        assert torch.equal(x, y), ("lengths=None vs all N", name)
    g0, gn = f0.grads(base.r_mel, base.r_gate), fn.grads(base.r_mel, base.r_gate)
    for k in g0:
        assert torch.equal(g0[k], gn[k]), ("lengths=None vs all N", k)
    del fn, g0, gn
    r = p.B // 2
    mem, mel, _ = _perturb_row(base.memory, base.mel, None, r, base.gen(2000))
    f1 = Fwd(p, base.dec, mem, mel, None)
    keep = [b for b in range(p.B) if b != r]
    for name, x, y in zip(("mel", "gate", "align"), (f1.m, f1.g, f1.a), (f0.m, f0.g, f0.a)):
        assert torch.equal(_rows(x, keep), _rows(y, keep)), ("lengths=None", r, name)


# --------------------------------------------------------------------------- 2. backward row isolation
def test_backward_rows_with_zero_upstream_get_zero_memory_gradient(base):
    p = base.path
    Z = sorted(set(p.rows) | {1, p.B // 3})
    keep = torch.ones(p.B, device=base.dev)
    keep[Z] = 0.0
    gr = base.fwd.grads(base.r_mel * keep[:, None, None], base.r_gate * keep[:, None], base.r_align * keep[:, None, None])
    dz = float(gr["memory"][Z].abs().max())
    assert dz == 0.0, (p.pid, Z, dz)
    others = [b for b in range(p.B) if b not in Z]
    assert float(_rows(gr["memory"], others).abs().amax(dim=(1, 2)).min()) > 0.0


# --------------------------------------------------------------------------- 3. row superposition
def test_row_partition_of_upstream_gradient_superposes(base):
    """grads(1_S r) + grads(1_S^c r) == grads(r): rows are computed independently, so what remains is fp32 reassociation of
    the reductions over rows and frames; d memory is a per-row computation and agrees bit for bit."""
    p = base.path
    S = (torch.arange(p.B, device=base.dev) % 3 == 1).float()
    C = 1.0 - S
    gs = base.fwd.grads(base.r_mel * S[:, None, None], base.r_gate * S[:, None])
    gc = base.fwd.grads(base.r_mel * C[:, None, None], base.r_gate * C[:, None])
    full = base.full
    rows_s, rows_c = S.bool(), C.bool()
    assert torch.equal(gs["memory"][rows_s], full["memory"][rows_s]), p.pid
    assert torch.equal(gc["memory"][rows_c], full["memory"][rows_c]), p.pid
    assert float(gs["memory"][rows_c].abs().max()) == 0.0 and float(gc["memory"][rows_s].abs().max()) == 0.0
    errs = {k: _rel(gs[k] + gc[k], full[k]) for k in full if k != "memory"}
    print(f"[{p.pid}] superposition floor (max|d| / max|g|):", {k: f"{v:.1e}" for k, v in errs.items()},
          "worst:", max(errs.items(), key=lambda kv: kv[1]))
    assert all(v < REASSOC_TOL for v in errs.values()), (p.pid, errs)


# --------------------------------------------------------------------------- 4. causality
def test_teacher_forcing_is_causal(base):
    """A T' = t0 run on the first t0 input frames is the prefix of the T run, bit for bit; the gradients of a loss on the first
    t0 frames agree up to reassociation (the weight-gradient GEMMs sum over T'*B instead of T*B frames)."""
    p = base.path
    t0 = p.T * 517 // 800
    short = Fwd(p, base.dec, base.memory, base.mel[:, :, :t0].contiguous(), base.lens)
    fw = {"mel": _rel(short.m.detach(), base.fwd.m.detach()[:, :, :t0]), "gate": _rel(short.g.detach(), base.fwd.g.detach()[:, :t0]),
          "align": _rel(short.a.detach(), base.fwd.a.detach()[:, :t0])}
    print(f"[{p.pid}] causality: forward prefix T'={t0} vs T={p.T}:", fw)
    assert all(v == 0.0 for v in fw.values()), (p.pid, fw)
    rm, rg, ra = base.r_mel[:, :, :t0].contiguous(), base.r_gate[:, :t0].contiguous(), base.r_align[:, :t0].contiguous()
    gs = short.grads(rm, rg, ra)
    cut = torch.zeros(p.T, device=base.dev)
    cut[:t0] = 1.0
    gl = base.fwd.grads(base.r_mel * cut, base.r_gate * cut, base.r_align * cut[:, None])
    errs = {k: _rel(gl[k], gs[k]) for k in gs}
    print(f"[{p.pid}] causality: gradients of the prefix loss:", {k: f"{v:.1e}" for k, v in errs.items()},
          "worst:", max(errs.items(), key=lambda kv: kv[1]))
    assert all(v < REASSOC_TOL for v in errs.values()), (p.pid, errs)


# --------------------------------------------------------------------------- 5. padding invariance
def test_padded_tokens_change_nothing(base):
    p = base.path
    mem = _padded(base.memory, base.lens, base.gen(3000))
    assert not torch.equal(mem, base.memory)
    f = Fwd(p, base.dec, mem, base.mel, base.lens)
    for name, x, y in zip(("mel", "gate", "align"), (f.m, f.g, f.a), (base.fwd.m, base.fwd.g, base.fwd.a)):
        assert torch.equal(x, y), (p.pid, name)
    gr = f.grads(base.r_mel, base.r_gate)
    for k, v in base.full.items():
        if k != "memory":
            assert torch.equal(gr[k], v), (p.pid, k)
    valid = torch.arange(p.N, device=base.dev)[None, :] < base.lens[:, None]
    assert float(gr["memory"][~valid].abs().max()) == 0.0, p.pid
    assert torch.equal(gr["memory"][valid], base.full["memory"][valid]), p.pid


# --------------------------------------------------------------------------- 6. bias identities
def test_bias_gradients_are_column_sums(base):
    p, full = base.path, base.full
    for key, r, dims in (("linear_projection.linear_layer.bias", base.r_mel, (0, 2)), ("gate_layer.linear_layer.bias", base.r_gate, None)):
        ref = r.double().sum(dims) if dims else r.double().sum().reshape(1)
        scale = r.double().abs().sum(dims) if dims else r.double().abs().sum().reshape(1)
        dev = (full[key].double() - ref).abs()
        print(f"[{p.pid}] {key}: max |g - sum| / sum|d| =", float((dev / scale).max()))
        assert bool((dev <= 1e-6 * scale).all()), (p.pid, key, float((dev / scale).max()))
    for lstm in ("attention_rnn", "decoder_rnn"):
        assert torch.equal(full[f"{lstm}.bias_ih"], full[f"{lstm}.bias_hh"]), (p.pid, lstm)


# --------------------------------------------------------------------------- 7. workspace and stash hygiene
def test_backward_reads_only_the_stash(base):
    """The backward takes the forward's stash as const: the same backward twice is bit-identical, and a zero upstream gradient
    right after a non-zero one gives exactly zero everywhere (nothing carried over in the workspace)."""
    p = base.path
    again = base.fwd.grads(base.r_mel, base.r_gate)
    for k, v in base.full.items():
        assert torch.equal(again[k], v), (p.pid, k)
    zero = base.fwd.grads(torch.zeros_like(base.r_mel), torch.zeros_like(base.r_gate), torch.zeros_like(base.r_align))
    for k, v in zero.items():
        assert float(v.abs().max()) == 0.0, (p.pid, k)


# --------------------------------------------------------------------------- 8a. alignment gradient: alignments do not see the decoder LSTM
def test_alignment_gradient_does_not_reach_decoder_lstm(base):
    p = base.path
    if p.pid not in ("F", "O", "S"):
        pytest.skip("run on the three bf16 chain layouts at their own shapes")
    gr = base.fwd.grads(torch.zeros_like(base.r_mel), torch.zeros_like(base.r_gate), base.r_align)
    for k, v in gr.items():
        if k.startswith(("decoder_rnn.", "linear_projection.", "gate_layer.")):
            assert float(v.abs().max()) == 0.0, (p.pid, k)
        elif k.startswith(("attention_rnn.", "attention_layer.", "memory")):
            assert float(v.abs().max()) > 0.0, (p.pid, k)


# --------------------------------------------------------------------------- inference: row isolation and padding invariance
@pytest.mark.parametrize("precision", ["bf16", "fp32"])
def test_inference_rows_and_padding(cuda_device, precision):
    dims = synth.DecoderDims()
    B, N, steps = 64, 150, 200
    dec = make_decoder(dims, synth.make_decoder_weights(31, dims), cuda_device, False)
    dec.precision = precision
    mem, _, lens = synth.make_inputs(91, B, N, 0, dims, ragged=True)
    memory, lens = torch.from_numpy(mem).to(cuda_device), torch.from_numpy(lens).to(cuda_device)

    def run(m, ln):
        dec.set_dropout_seed(SEED)
        out = dec.inference(m, memory_lengths=ln, ignore_gate=True, max_decoder_steps=steps)
        _sync()
        return out

    ref = run(memory, lens)
    for r in (0, 31, 32, 63):
        m, _, ln = _perturb_row(memory, None, lens, r, torch.Generator(device=cuda_device).manual_seed(4000 + r))
        out = run(m, ln)
        keep = [b for b in range(B) if b != r]
        for name, x, y in zip(("mel", "gate", "align"), out, ref):
            assert torch.equal(_rows(x, keep), _rows(y, keep)), (precision, r, name)
            assert not torch.equal(x[r], y[r]), (precision, r, name)
    out = run(_padded(memory, lens, torch.Generator(device=cuda_device).manual_seed(5000)), lens)
    for name, x, y in zip(("mel", "gate", "align"), out, ref):
        assert torch.equal(x, y), (precision, "padding", name)


# --------------------------------------------------------------------------- 8b. alignment gradient against the oracle
def _u(seed, stream, shape):
    return torch.from_numpy((synth.uniform01(seed, stream, int(np.prod(shape))) - 0.5).astype(np.float32).reshape(shape))


def _oracle_case(dev, B, N, T, fused, round_memory, row_offset, with_align, oracle=True):
    """GPU forward + backward (bf16, training) against the same-rounding oracle; returns (fwd errs, grad errs, gpu results)."""
    dims = synth.DecoderDims()
    W = synth.make_decoder_weights(23, dims)
    mem, mel, lens = synth.make_inputs(67, B, N, T, dims, ragged=True)
    r_mel, r_gate, r_align = _u(67, 20, (B, dims.n_mels, T)), _u(67, 21, (B, T)), _u(67, 22, (B, T, N))
    path = Path("oracle", B, N, T, "bf16", fused)
    dec = make_decoder(dims, W, dev, True)
    dec.precision = "bf16"
    dec.dropout_row_offset = row_offset
    d = lambda x: torch.from_numpy(x).to(dev)
    f = Fwd(path, dec, d(mem), d(mel), d(lens))
    gr = f.grads(r_mel.to(dev), r_gate.to(dev), r_align.to(dev) if with_align else None)
    got = (f.m.detach().cpu(), f.g.detach().cpu(), f.a.detach().cpu(), {k: v.cpu() for k, v in gr.items()})
    if not oracle:
        return None, None, got
    with O.bf16_semantics(round_memory=round_memory):
        (om, og, oa), ograds, omem = O.loss_and_grads(O.as_params(W), torch.from_numpy(mem), torch.from_numpy(mel), lens, r_mel, r_gate,
                                                      SEED, True, dims.p_attention_dropout, dims.p_decoder_dropout,
                                                      r_align=r_align if with_align else None, row_offset=row_offset)
    errs = {"mel": rel_err(got[0], om), "gate": rel_err(got[1], og), "align": rel_err(got[2], oa)}
    gerrs = {k: rel_err(got[3][k], ograds[k]) for k in ograds}
    gerrs["memory"] = rel_err(got[3]["memory"], omem)
    return errs, gerrs, got


@pytest.mark.parametrize("B,N,T,fused,round_memory", [(8, 50, 12, 1, True),      # fused chains
                                                      (16, 200, 9, 1, True),     # per-step forward + persistent BPTT chain
                                                      (8, 50, 12, 0, False)])    # per-step chains
def test_alignment_gradient_matches_same_rounding_oracle(cuda_device, B, N, T, fused, round_memory):
    errs, gerrs, _ = _oracle_case(cuda_device, B, N, T, fused, round_memory, 0, True)
    print("with d_align, vs same-rounding oracle:", errs, {k: f"{v:.1e}" for k, v in gerrs.items()})
    assert all(np.isfinite(v) and v < SAME_ROUNDING_FWD_TOL for v in errs.values()), errs
    assert all(np.isfinite(v) and v < SAME_ROUNDING_GRAD_TOL for v in gerrs.values()), gerrs


# --------------------------------------------------------------------------- 9. dropout row offset in the GPU kernels
@pytest.mark.parametrize("B,N,T,fused", [(16, 60, 12, 1), (16, 200, 12, 1)])
def test_dropout_row_offset_matches_oracle(cuda_device, B, N, T, fused):
    """Rows 48..63 of one dropout stream (a data-parallel rank's share of the batch) in the fused chains, the persistent LSTM
    chains and the all-frames prenet; the same call with offset 0 differs by O(1), so an ignored offset cannot pass."""
    errs, gerrs, got = _oracle_case(cuda_device, B, N, T, fused, True, 48, False)
    print("row offset 48 vs same-rounding oracle:", errs, {k: f"{v:.1e}" for k, v in gerrs.items()})
    assert all(np.isfinite(v) and v < SAME_ROUNDING_FWD_TOL for v in errs.values()), errs
    assert all(np.isfinite(v) and v < SAME_ROUNDING_GRAD_TOL for v in gerrs.values()), gerrs
    _, _, got0 = _oracle_case(cuda_device, B, N, T, fused, True, 0, False, oracle=False)
    d_mel = rel_err(got[0], got0[0])
    d_grad = rel_err(got[3]["attention_rnn.weight_hh"], got0[3]["attention_rnn.weight_hh"])
    print("offset 48 vs offset 0:", {"mel": d_mel, "d attention_rnn.weight_hh": d_grad})
    assert d_mel > 0.1 and d_grad > 0.1, (d_mel, d_grad)
