"""The attention constraint (Decoder.attention_window, gvx_dec_*_windowed) on the GPU, in each forward attention kernel
inference can select and in both precisions.

Rule (include/genvox_b200.h): at step t, last = argmax_n w_{t-1}[b, n] (lowest index on ties), and tokens outside
[last - backward, last + forward) get energy -inf.  The kernel is chosen by shape (launch_attention_fwd_best):
  * generic  k_attention_fwd       - shapes other than 32 filters / kernel 31 / attention_dim 128 (SMALL_DIMS);
  * c2       k_attention_fwd_c2    - the default shape with B <= 74 rows and N >= 32 tokens;
  * fast     k_attention_fwd_fast  - the default shape otherwise (here N < 32)."""
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from conftest import rel_err
from genvox_b200 import _native, install
from genvox_b200.decoder import _buffer, _ptr, _stream
import attention_window_oracle as WO
from oracle import decoder_oracle as O
from oracle import standin, synth
from test_cuda_bf16 import SAME_ROUNDING_FWD_TOL
from test_cuda_continuous import SEED, STEPS, _check_against_static, _continuous, _decoder, _queue, _sync
from test_cuda_parity import FWD_TOL, argmax_agrees
from test_cuda_session import _check_static, _drive, _session, _spread_caps, _staggered

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
WIN = (1, 3)
S = 4
ROUTES = {"generic": (synth.SMALL_DIMS, 24), "fast": (synth.DecoderDims(), 24), "c2": (synth.DecoderDims(), 64)}
CASES = [(r, p) for r in ROUTES for p in ("fp32", "bf16")]


def _route(dims, B, N):
    """the kernel launch_attention_fwd_best selects (attention_fast_ok, attention_fwd_uses_c2 in gvx_attention_*.cuh; the
    shared-memory limits are far off at these N)"""
    fast_ok = (dims.attention_location_n_filters, dims.attention_location_kernel_size, dims.attention_dim) == (32, 31, 128) \
        and dims.encoder_embedding_dim % 4 == 0
    if not fast_ok:
        return "generic"
    c2_on = not os.environ.get("GVX_ATT_C2", "").startswith("0")
    return "c2" if c2_on and B <= 74 and N >= 32 and dims.encoder_embedding_dim % 8 == 0 else "fast"


def _setup(dev, route, precision, gate_bias=-0.2):
    dims, N = ROUTES[route]
    assert _route(dims, S, N) == route
    dec, W = _decoder(dev, precision, dims, gate_bias=gate_bias)
    memory, lens = _queue(dev, 3 * S + 1, N, dims)          # _staggered needs at least 2 S + 4 utterances
    return dec, W, memory, lens, N


def _static(dec, memory, lens, window, ignore_gate=True, steps=STEPS):
    dec.set_dropout_seed(SEED)
    out = dec.inference(memory, memory_lengths=lens, ignore_gate=ignore_gate, max_decoder_steps=steps, attention_window=window)
    _sync()
    return [t.clone() for t in out], dec.last_n_frames.clone()


def _peaks(align):
    """the `last` of every step of a GPU decode: 0, then the argmax of the previous step's weights"""
    B, T, _ = align.shape
    p = align.argmax(-1).cpu()
    return [torch.zeros(B, dtype=torch.int64)] + [p[:, t - 1] for t in range(1, T)]


# --------------------------------------------------------------------------- 1. a window over everything changes nothing
@pytest.mark.parametrize("route,precision", CASES)
def test_window_over_every_token_is_bit_identical(cuda_device, route, precision):
    dec, _, memory, lens, N = _setup(cuda_device, route, precision)
    (m0, g0, a0), n0 = _static(dec, memory[:S], lens[:S], None)
    (m1, g1, a1), n1 = _static(dec, memory[:S], lens[:S], (N, N))
    assert torch.equal(m0, m1) and torch.equal(g0, g1) and torch.equal(a0, a1) and torch.equal(n0, n1)
    caps = _spread_caps(memory.shape[0], 7)
    (cm0, cg0, ca0), cn0 = _continuous(dec, memory, lens, S, caps)
    dec.attention_window = (N, N)
    (cm1, cg1, ca1), cn1 = _continuous(dec, memory, lens, S, caps)
    out1 = _drive(_session(dec, N, S), memory, lens, caps, _staggered(memory.shape[0], S, chunk=5))
    dec.attention_window = None
    assert torch.equal(cm0, cm1) and torch.equal(cg0, cg1) and torch.equal(ca0, ca1) and torch.equal(cn0, cn1)
    out0 = _drive(_session(dec, N, S), memory, lens, caps, _staggered(memory.shape[0], S, chunk=5))
    for u in out0:
        for x, y in zip(out0[u][:3], out1[u][:3]):
            assert torch.equal(x, y), u
        assert out0[u][3] == out1[u][3]


# --------------------------------------------------------------------------- 2. support and step bound, exact
@pytest.mark.parametrize("route,precision", CASES)
def test_support_and_step_bound(cuda_device, route, precision):
    dec, _, memory, lens, N = _setup(cuda_device, route, precision)
    (_, _, a), _ = _static(dec, memory[:S], lens[:S], WIN)
    (_, _, a0), _ = _static(dec, memory[:S], lens[:S], None)
    a, a0 = a.cpu(), a0.cpu()
    B, T, _ = a.shape
    p = a.argmax(-1)                                                        # torch.argmax: lowest index on ties
    prev = torch.cat([torch.zeros(B, 1, dtype=p.dtype), p[:, :-1]], dim=1)
    n = torch.arange(N)[None, None, :]
    outside = (n < prev[..., None] - WIN[0]) | (n >= prev[..., None] + WIN[1]) | (n >= lens[:S].cpu()[:, None, None])
    assert not bool(a[outside].any()), "weight outside the window"
    step = p - prev
    assert int(step.min()) >= -1 and int(step.max()) <= 2, (int(step.min()), int(step.max()))
    assert torch.allclose(a.double().sum(-1), torch.ones(B, T, dtype=torch.float64), atol=1e-5)
    assert not torch.equal(a, a0)


# --------------------------------------------------------------------------- 3. against the oracle
@pytest.mark.parametrize("route", list(ROUTES))
def test_fp32_matches_fp64_oracle(cuda_device, route):
    dec, W, memory, lens, N = _setup(cuda_device, route, "fp32")
    mem, ln = memory[:S], lens[:S]
    (m, g, a), nf = _static(dec, mem, ln, WIN, ignore_gate=False)
    T = m.shape[2]
    peaks = _peaks(a) + [None] * (STEPS - T)                                # past the GPU's last step: the oracle's own argmax
    rm, rg, ra, rn = WO.inference(O.as_params(W, torch.float64), mem.cpu().double(), ln.cpu(), STEPS, dec.gate_threshold, False,
                                 SEED, False, dec.p_attention_dropout, dec.p_decoder_dropout, window=WIN, peaks=peaks)
    assert nf.cpu().long().tolist() == rn.tolist()                          # stop steps exact
    assert ra.shape[1] == T
    for k, got, ref in (("mel", m, rm), ("gate", g, rg), ("align", a, ra)):
        e = rel_err(got.cpu(), ref)
        assert e <= FWD_TOL, (k, e)
    ok, _ = argmax_agrees(a.cpu().numpy(), ra.numpy())                      # its own argmax agrees where the margin is clear
    assert ok


@pytest.mark.parametrize("route", list(ROUTES))
def test_bf16_matches_same_rounding_oracle(cuda_device, route):
    dec, W, memory, lens, N = _setup(cuda_device, route, "bf16")
    mem, ln = memory[:S], lens[:S]
    (m, g, a), _ = _static(dec, mem, ln, WIN)
    assert m.shape[2] == STEPS <= 64
    with O.bf16_semantics():
        rm, rg, ra, _ = WO.inference(O.as_params(W), mem.cpu(), ln.cpu(), STEPS, dec.gate_threshold, True, SEED, False,
                                    dec.p_attention_dropout, dec.p_decoder_dropout, window=WIN, peaks=_peaks(a))
    errs = {k: rel_err(got.cpu(), ref) for k, got, ref in (("mel", m, rm), ("gate", g, rg), ("align", a, ra))}
    assert all(np.isfinite(v) and v < SAME_ROUNDING_FWD_TOL for v in errs.values()), errs


# --------------------------------------------------------------------------- 4. the continuous and session contracts
@pytest.mark.parametrize("route,precision", CASES)
def test_continuous_and_session_equal_static_with_the_window(cuda_device, route, precision):
    dec, _, memory, lens, N = _setup(cuda_device, route, precision)
    U = memory.shape[0]
    caps = _spread_caps(U, 31)
    dec.attention_window = WIN          # the helpers call inference / inference_continuous / session without a window
    try:
        nf = _check_against_static(dec, memory, lens, S, caps, row_offset=3)
        assert len(set(nf.tolist())) >= 3, nf                              # slots refill at different steps
        sess = _session(dec, N, S, row_offset=3)
        out = _drive(sess, memory, lens, caps, _staggered(U, S, chunk=5))
        _check_static(dec, memory, lens, S, out, caps, row_offset=3)
    finally:
        dec.attention_window = None
    # the window really applied: an unconstrained static call differs
    dec.dropout_row_offset = 3
    (_, _, a_free), _ = _static(dec, memory[:S], lens[:S], None)
    (_, _, a_win), _ = _static(dec, memory[:S], lens[:S], WIN)
    dec.dropout_row_offset = 0
    assert not torch.equal(a_free, a_win)


def test_session_fixes_its_window_at_creation(cuda_device):
    dec, _, memory, lens, N = _setup(cuda_device, "c2", "fp32")
    caps = _spread_caps(memory.shape[0], 31)
    dec.attention_window = WIN
    sess = _session(dec, N, S)
    dec.attention_window = None                                             # later edits do not reach a running session
    out = _drive(sess, memory, lens, caps, [("submit", 0, 6), ("step", 5), ("submit", 6, memory.shape[0]), ("drain", 7)])
    dec.attention_window = WIN
    try:
        _check_static(dec, memory, lens, S, out, caps)
    finally:
        dec.attention_window = None


# --------------------------------------------------------------------------- 5. launch count
@pytest.mark.parametrize("route,precision", [("c2", "fp32"), ("c2", "bf16"), ("generic", "fp32")])
def test_launch_count_does_not_change(cuda_device, route, precision):
    lib = _native.load()
    dec, _, memory, lens, N = _setup(cuda_device, route, precision, gate_bias=-30.0)     # the gate never fires

    def launches(fn):
        _sync()
        c0 = lib.gvx_launch_count()
        fn()
        _sync()
        return lib.gvx_launch_count() - c0

    caps = torch.full((memory.shape[0],), 8, dtype=torch.int32)
    dec.inference(memory[:S], memory_lengths=lens[:S], max_decoder_steps=2)                 # warm (weight packing)
    counts = {}
    for win in (None, WIN):
        dec.attention_window = win
        try:
            static = launches(lambda: dec.inference(memory[:S], memory_lengths=lens[:S], max_decoder_steps=12))
            cont = launches(lambda: dec.inference_continuous(memory, lens, slots=S, max_decoder_steps=STEPS, frame_caps=caps))
            sess = _session(dec, N, S)
            sess.submit(memory, lens)
            step = launches(lambda: sess.step(6))
        finally:
            dec.attention_window = None
        counts[win] = (static, cont, step, dec.last_steps_run)
    assert counts[None] == counts[WIN], counts


# --------------------------------------------------------------------------- 6. graph cache key
def _graph_cache_run():
    """Run in a child process with GVX_GRAPHS=1 (the switch is read once per process): fixed-step calls with window A on
    one set of buffers (eager, captured, replayed), then window B on the same buffers, then B eagerly on fresh buffers."""
    dev = torch.device("cuda:0")
    dec, _, memory, lens, N = _setup(dev, "c2", "fp32")
    lib = _native.load()
    mem, ln = memory[:S].contiguous(), lens[:S].contiguous()
    params = [p.detach() for p in dec._ordered_params()]
    dims, weights, packed = dec._native_state(params)

    def buffers():
        return dict(mel=torch.empty(S, dec.n_mel_channels, STEPS, device=dev), gate=torch.empty(S, STEPS, device=dev),
                    align=torch.empty(S, STEPS, N, device=dev), nf=torch.empty(S, dtype=torch.int32, device=dev),
                    work=_buffer(lib.gvx_dec_infer_workspace_bytes(C.byref(dims), S, N, STEPS), dev))

    def run(b, win):
        ran = C.c_int(0)
        _native.check(lib.gvx_dec_infer_windowed(C.byref(dims), C.byref(weights), _ptr(packed), _ptr(mem), _ptr(ln), S, N, STEPS,
                                                 0.5, 1, SEED, 0, 0, _ptr(b["mel"]), _ptr(b["gate"]), _ptr(b["align"]),
                                                 _ptr(b["nf"]), C.byref(ran), win[0], win[1], _ptr(b["work"]), _stream()),
                      "gvx_dec_infer_windowed")
        torch.cuda.synchronize()
        return b["mel"].clone(), b["align"].clone()

    def stats():
        s = (C.c_ulonglong * 4)()
        _native.check(lib.gvx_graph_stats(s), "gvx_graph_stats")
        return list(s)

    A, B = (1, 3), (0, 2)
    same = buffers()
    s0 = stats()
    outs_a = [run(same, A) for _ in range(3)]
    s1 = stats()
    out_b = run(same, B)
    s2 = stats()
    eager_b = run(buffers(), B)
    s3 = stats()
    res = {
        "a_captured_and_replayed": [s1[1] - s0[1], s1[2] - s0[2]],
        "a_runs_equal": all(torch.equal(x[0], outs_a[0][0]) and torch.equal(x[1], outs_a[0][1]) for x in outs_a),
        "b_not_replayed_from_a": s2[2] == s1[2],
        "b_eager": s3[0] - s2[0],
        "b_equals_eager_b": torch.equal(out_b[0], eager_b[0]) and torch.equal(out_b[1], eager_b[1]),
        "b_differs_from_a": not torch.equal(out_b[1], outs_a[0][1]),
    }
    print("GRAPH_RESULT " + json.dumps(res))


def test_graph_cache_keys_on_the_window(cuda_device):
    env = dict(os.environ, GVX_GRAPHS="1", PYTHONPATH=os.pathsep.join([ROOT, os.path.join(ROOT, "tests")]))
    code = "import test_cuda_attention_window as t; t._graph_cache_run()"
    py = [sys.executable] + (["-s"] if sys.flags.no_user_site else [])
    p = subprocess.run(py + ["-c", code], env=env, cwd=ROOT, capture_output=True, text=True, timeout=900)
    lines = [ln for ln in p.stdout.splitlines() if ln.startswith("GRAPH_RESULT ")]
    assert p.returncode == 0 and lines, p.stdout[-2000:] + p.stderr[-4000:]
    res = json.loads(lines[-1][len("GRAPH_RESULT "):])
    assert res["a_captured_and_replayed"] == [1, 1], res
    assert res["a_runs_equal"] and res["b_not_replayed_from_a"] and res["b_eager"] >= 1, res
    assert res["b_equals_eager_b"] and res["b_differs_from_a"], res


# --------------------------------------------------------------------------- 7. drop-in on an installed model
def test_attribute_on_an_installed_decoder(cuda_device):
    dims = synth.SMALL_DIMS
    model = standin.Tacotron2(dims, n_tokens=40).to(cuda_device).eval()
    install(model)
    model.decoder.gate_layer.linear_layer.bias.data.fill_(-0.15)
    model.decoder._next_seed = lambda: 1234
    tokens = torch.randint(0, 40, (1, 23), generator=torch.Generator().manual_seed(3)).to(cuda_device)
    free = model.inference({"tokens": tokens})
    model.decoder.attention_window = WIN
    got = model.inference({"tokens": tokens})
    model.decoder.attention_window = None
    enc = model.encoder.inference(model.embedding(tokens).transpose(1, 2))
    mel, gate, align = model.decoder.inference(enc, attention_window=WIN)
    _sync()
    assert torch.equal(got["mel_outputs"], mel) and torch.equal(got["gate_outputs"], gate) and torch.equal(got["alignments"], align)
    assert got["alignments"].shape != free["alignments"].shape or not torch.equal(got["alignments"], free["alignments"])
