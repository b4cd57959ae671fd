"""CPU-side checks of decoder sessions: argument validation of Decoder.session and of the C ABI (gvx_dec_session_*), and the
session workspace size.  Every refusal here happens before the library touches a device."""
import ctypes as C

import pytest
import torch

READY = 0x53455353          # gvx_session.ready as gvx_dec_session_init leaves it (csrc/gvx_session.cuh)
E, D = 512, 128


def _decoder(precision="fp32"):
    import genvox_b200
    dec = genvox_b200.Decoder(80, 512, 1024, 256, 1000, 0.5, 0.1, 0.1, 1024, 128, 32, 31).eval()
    dec.precision = precision
    return dec


def _session(**kw):
    from genvox_b200 import _native
    s = _native.GvxSession()
    s.N, s.slots, s.capacity, s.max_steps, s.with_alignments, s.gate_threshold = 50, 8, 64, 100, 1, 0.5
    for k, v in kw.items():
        setattr(s, k, v)
    return s


def _refused(rc, match):
    from genvox_b200 import _native
    assert rc != 0
    with pytest.raises(RuntimeError, match=match):
        _native.check(rc, "session")


def test_session_rejects_bad_arguments():
    dec = _decoder("bf16")
    for slots in (0, -1, 129):
        with pytest.raises(ValueError, match="slots"):
            dec.session(50, slots=slots)
    dec.precision = "fp32"
    for kw in ({"capacity": 0}, {"max_decoder_steps": 0}):
        with pytest.raises(ValueError, match="positive"):
            dec.session(50, slots=4, **kw)
    with pytest.raises(ValueError, match="positive"):
        dec.session(0, slots=4)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        dec.session(50, slots=4)
    dec.train()
    with pytest.raises(RuntimeError, match="eval mode"):
        dec.session(50, slots=4)


def test_c_abi_refusals():
    from genvox_b200 import _native
    lib = _native.load()
    d = _decoder()._dims()
    w = _native.GvxWeights()
    dummy = C.c_void_p(16)          # never dereferenced: every call below is refused first
    ran = C.c_int(-1)

    def submit(s, k=1, memory=dummy, dims=d):
        return lib.gvx_dec_session_submit(C.byref(dims), C.byref(w), dummy, C.byref(s), memory, None, None, k, dummy, None)

    def step(s, k=16, frames=dummy, dims=d):
        return lib.gvx_dec_session_step(C.byref(dims), C.byref(w), dummy, C.byref(s), k, frames, dummy, dummy, dummy, dummy,
                                        C.byref(ran), dummy, None)

    # init: bad fields, bf16 with more than 128 slots, null workspace
    for kw in ({"N": 0}, {"slots": 0}, {"capacity": 0}, {"max_steps": 0}):
        _refused(lib.gvx_dec_session_init(C.byref(d), C.byref(_session(**kw)), dummy, None), "positive")
    _refused(lib.gvx_dec_session_init(C.byref(d), C.byref(_session(row_offset=-1)), dummy, None), "row_offset")
    _refused(lib.gvx_dec_session_init(C.byref(d), C.byref(_session()), None, None), "null")
    bf = _decoder("bf16")._dims()
    _refused(lib.gvx_dec_session_init(C.byref(bf), C.byref(_session(slots=129)), dummy, None), "128")
    bad = _native.GvxDims(80, 512, 1024, 1024, 256, 128, 32, 30, 0.1, 0.1)       # even conv kernel
    _refused(lib.gvx_dec_session_init(C.byref(bad), C.byref(_session()), dummy, None), "odd")
    # a submit or a step before init
    _refused(submit(_session()), "init")
    _refused(step(_session()), "init")
    # the ring: submitted + k - admitted > capacity
    _refused(submit(_session(ready=READY), k=65), "ring is full")
    _refused(submit(_session(ready=READY, submitted=100, admitted=40), k=5), "ring is full")
    # ids: id + row_offset past 2^31 - 1
    _refused(submit(_session(ready=READY, row_offset=2 ** 31 - 10, capacity=64), k=11), "2\\^31")
    _refused(submit(_session(ready=READY, submitted=2 ** 31 - 1, admitted=2 ** 31 - 1), k=2), "2\\^31")
    # null and out-of-range arguments
    _refused(submit(_session(ready=READY), memory=None), "null")
    _refused(submit(_session(ready=READY), k=0), "k must be positive")
    _refused(step(_session(ready=READY), frames=None), "null")
    _refused(step(_session(ready=READY), k=0), "positive")
    # a step with nothing queued and nothing running does nothing and launches nothing
    c0 = lib.gvx_launch_count()
    assert step(_session(ready=READY)) == 0 and ran.value == 0
    assert lib.gvx_launch_count() == c0


def test_session_workspace_size():
    from genvox_b200 import _native
    lib = _native.load()
    dec = _decoder()
    d = dec._dims()
    size = lambda cap, N=150, S=64: lib.gvx_dec_session_workspace_bytes(C.byref(d), N, S, cap)
    assert 0 < size(64) < size(1024) < size(4096)
    # the queue ring: memory [N, E] and processed memory [N, D] floats, an int64 length and an int32 frame cap per entry
    assert size(4096) - size(64) == (4096 - 64) * (150 * (E + D) * 4 + 8 + 4)
    assert size(1024) - size(960) == 64 * (150 * (E + D) * 4 + 8 + 4)
    assert size(0) == 0 and size(-1) == 0 and size(64, N=0) == 0 and size(64, S=0) == 0
    bad = _native.GvxDims(80, 512, 1024, 1024, 256, 128, 32, 30, 0.1, 0.1)
    assert lib.gvx_dec_session_workspace_bytes(C.byref(bad), 150, 64, 64) == 0
    dec.precision = "bf16"
    d = dec._dims()
    assert size(64, S=128) > 0 and size(64, S=129) == 0
