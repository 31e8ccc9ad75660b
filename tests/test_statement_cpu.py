"""Proof and statement in one call (sipp_prove_native_statement and its batched, ragged and device forms) without a GPU: every argument
error with the code and order of the sibling prover (all of them before the device is touched), the loud failure of a valid call
without a device, sentinel-filled outputs left untouched on every error, and the Python wrappers' ValueErrors."""
import ctypes

import pytest

SENT = b"\x5a"


@pytest.fixture(scope="module")
def lib():
    from sipp_b200 import _lib
    return _lib.load()


def _offs(*o):
    return (ctypes.c_size_t * len(o))(*o)


def _bufs(count, np):
    return [ctypes.create_string_buffer(SENT * k, k) for k in (384 * np, 64 * count, 128 * count, 384 * count)]


def _untouched(bufs):
    return all(b.raw == SENT * len(b.raw) for b in bufs)


def single(lib, a=bytes(64 * 4), a_len=4, b=bytes(128 * 4), b_len=4, proof=True, finals=(True, True, True)):
    bufs = _bufs(1, 5)
    fin = [f if on else None for f, on in zip(bufs[1:], finals)]
    rc = lib.sipp_prove_native_statement(a, a_len, b, b_len, bufs[0] if proof else None, *fin)
    return rc, bufs


def batch(lib, device=False, a=True, b=True, n=4, count=2, proofs=True):
    bufs = _bufs(count, 5)
    if device:  # never dereferenced: every case below fails before the device is touched, or without one
        ptr = [ctypes.addressof(x) for x in bufs]
        rc = lib.sipp_prove_native_batch_statement_device(0x1000 if a else None, 0x2000 if b else None, n, count, ptr[0] if proofs else None,
                                                          *ptr[1:])
    else:
        rc = lib.sipp_prove_native_batch_statement(bytes(64 * n * max(1, count)) if a else None, bytes(128 * n * max(1, count)) if b else None,
                                                   n, count, bufs[0] if proofs else None, *bufs[1:])
    return rc, bufs


RA, RB = bytes(64 * 6), bytes(128 * 6)


def ragged(lib, device=False, a=RA, a_len=6, b=RB, b_len=6, offs=(0, 2, 6), count=2, proofs=True):
    bufs = _bufs(max(1, count), 8)
    o = None if offs is None else _offs(*offs)
    if device:
        ptr = [ctypes.addressof(x) for x in bufs]
        rc = lib.sipp_prove_native_batch_ragged_statement_device(0x1000 if a is not None else None, 0x2000 if b is not None else None, a_len, o,
                                                                 count, ptr[0] if proofs else None, *ptr[1:])
    else:
        rc = lib.sipp_prove_native_batch_ragged_statement(a, a_len, b, b_len, o, count, bufs[0] if proofs else None, *bufs[1:])
    return rc, bufs


def test_single_argument_errors(lib):
    """the checks of sipp_prove_native, in its order: lengths, then a power of two, then the pointers"""
    from sipp_b200 import _lib
    cases = [({"b_len": 2}, _lib.ERR_LENGTH),
             ({"b_len": 2, "a": None}, _lib.ERR_LENGTH),           # the length check comes first
             ({"a_len": 3, "b_len": 3}, _lib.ERR_ARG),
             ({"a_len": 0, "b_len": 0}, _lib.ERR_ARG),
             ({"a_len": 3, "b_len": 3, "proof": False}, _lib.ERR_ARG),
             ({"a": None}, _lib.ERR_ARG),
             ({"b": None}, _lib.ERR_ARG),
             ({"proof": False}, _lib.ERR_ARG)]
    for kw, want in cases:
        rc, bufs = single(lib, **kw)
        assert rc == want, kw
        assert _untouched(bufs), kw
        assert rc == lib.sipp_prove_native(kw.get("a", bytes(256)), kw.get("a_len", 4), kw.get("b", bytes(512)), kw.get("b_len", 4),
                                           None if kw.get("proof") is False else ctypes.create_string_buffer(384 * 5)), kw


def test_batch_argument_errors(lib):
    """the checks of sipp_prove_native_batch (pointers and count, then n) for the host and the device form"""
    from sipp_b200 import _lib
    for device in (False, True):
        for kw in ({"a": False}, {"b": False}, {"proofs": False}, {"count": 0}, {"n": 3}, {"n": 0}, {"n": 3, "a": False}):
            rc, bufs = batch(lib, device=device, **kw)
            assert rc == _lib.ERR_ARG, (device, kw)
            assert _untouched(bufs), (device, kw)


def test_ragged_argument_errors(lib):
    """the checks of sipp_prove_native_batch_ragged, in its order, for the host and the device form"""
    from sipp_b200 import _lib
    for device in (False, True):
        big = 1 << 32                                                                    # more than 2^32 - 1 pairs (never read)
        cases = [({"b_len": 5}, _lib.ERR_LENGTH),
                 ({"b_len": 5, "a": None}, _lib.ERR_LENGTH),
                 ({"a": None}, _lib.ERR_ARG),
                 ({"b": None}, _lib.ERR_ARG),
                 ({"offs": None}, _lib.ERR_ARG),
                 ({"proofs": False}, _lib.ERR_ARG),
                 ({"count": 0}, _lib.ERR_ARG),
                 ({"offs": (1, 2, 6)}, _lib.ERR_ARG),                                  # offsets[0] != 0
                 ({"offs": (0, 4, 2, 6), "count": 3}, _lib.ERR_ARG),                   # decreasing
                 ({"offs": (0, 2, 4)}, _lib.ERR_ARG),                                  # offsets[count] != a_len
                 ({"offs": (0, 0, 2, 6), "count": 3}, _lib.ERR_ARG),                   # an empty instance
                 ({"offs": (0, 3, 6)}, _lib.ERR_ARG),                                  # not a power of two
                 ({"a_len": big, "b_len": big, "offs": (0, big), "count": 1}, _lib.ERR_ARG)]
        for kw, want in cases:
            if device and kw.get("b_len") == 5:
                continue                                                                 # the device form has one n
            rc, bufs = ragged(lib, device=device, **kw)
            assert rc == want, (device, kw)
            assert _untouched(bufs), (device, kw)
            if not device:
                o = kw.get("offs", (0, 2, 6))
                assert rc == lib.sipp_prove_native_batch_ragged(kw.get("a", RA), kw.get("a_len", 6), kw.get("b", RB), kw.get("b_len", 6),
                                                                None if o is None else _offs(*o), kw.get("count", 2),
                                                                None if kw.get("proofs") is False else ctypes.create_string_buffer(384 * 8)), kw


def test_no_gpu_fails_loudly(lib):
    """valid arguments without a device: SIPP_ERR_CUDA from all five calls, NULL finals included, and nothing written"""
    import sipp_b200
    from sipp_b200 import _lib
    if lib.sipp_device_count() > 0:
        pytest.skip("a GPU is present")
    for finals in ((True, True, True), (False, True, True), (True, False, True), (True, True, False), (False, False, False)):
        rc, bufs = single(lib, finals=finals)
        assert rc == _lib.ERR_CUDA and _untouched(bufs), finals
    for device in (False, True):
        rc, bufs = batch(lib, device=device)
        assert rc == _lib.ERR_CUDA and _untouched(bufs), device
        rc, bufs = ragged(lib, device=device)
        assert rc == _lib.ERR_CUDA and _untouched(bufs), device
    rc, bufs = single(lib, a_len=1, b_len=1, a=bytes(64), b=bytes(128))
    assert rc == _lib.ERR_CUDA and _untouched(bufs)
    calls = [lambda: sipp_b200.sipp_prove_native_statement(bytes(64 * 4), bytes(128 * 4)),
             lambda: sipp_b200.sipp_prove_native_batch_statement(bytes(64 * 8), bytes(128 * 8), 4),
             lambda: sipp_b200.sipp_prove_native_batch_ragged_statement(RA, RB, [2, 4]),
             lambda: sipp_b200.sipp_prove_native_batch_statement_device(0x1000, 0x2000, 4, 2, 0x3000, 0, 0, 0),
             lambda: sipp_b200.sipp_prove_native_batch_ragged_statement_device(0x1000, 0x2000, 6, [2, 4], 0x3000, 0, 0, 0)]
    for call in calls:
        with pytest.raises(sipp_b200.SippError) as ei:
            call()
        assert ei.value.code == _lib.ERR_CUDA


def test_python_argument_errors():
    import sipp_b200
    with pytest.raises(AssertionError):
        sipp_b200.sipp_prove_native_statement(bytes(64 * 4), bytes(128 * 2))
    with pytest.raises(ValueError):
        sipp_b200.sipp_prove_native_statement(bytes(63), bytes(128))                     # not whole points
    for A, B, n in ((bytes(64 * 6), bytes(128 * 6), 4), (bytes(64 * 4), bytes(128 * 4), 0), (b"", b"", 4)):
        with pytest.raises(ValueError):
            sipp_b200.sipp_prove_native_batch_statement(A, B, n)
    with pytest.raises(AssertionError):
        sipp_b200.sipp_prove_native_batch_statement(bytes(64 * 4), bytes(128 * 8), 4)
    for lengths in ([3, 3], [6], [0, 2, 4], [-2, 8], [2, 2]):                      # as sipp_prove_native_batch_ragged
        with pytest.raises(ValueError):
            sipp_b200.sipp_prove_native_batch_ragged_statement(RA, RB, lengths)
        with pytest.raises(ValueError):
            sipp_b200.sipp_prove_native_batch_ragged_statement_device(0x1000, 0x2000, 6, lengths, 0x3000, 0, 0, 0)
    with pytest.raises(ValueError):
        sipp_b200.sipp_prove_native_batch_ragged_statement(b"", b"", [])
    with pytest.raises(AssertionError):
        sipp_b200.sipp_prove_native_batch_ragged_statement(RA, bytes(128 * 4), [2, 4])
