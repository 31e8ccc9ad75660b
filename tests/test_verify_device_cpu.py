"""Batched verification on device buffers (sipp_verify_native_batch_device, sipp_verify_native_batch_ragged_device) without a GPU:
every argument error and its code, in the order the header gives (all of them come before the device is touched), the loud failure
of a valid call without a device, and the Python wrappers' ValueErrors.  The device pointers here are never dereferenced."""
import ctypes

import pytest

FAKE = 0x7f0000001000          # a device address that is never read: every call below stops before the device is touched
N_POFFS = (0, 3, 8)            # n = 2, 4: proofs of 3 and 5 elements
N_OFFS = (0, 2, 6)


@pytest.fixture(scope="module")
def lib():
    from sipp_b200 import _lib
    return _lib.load()


def _szt(*o):
    return (ctypes.c_size_t * len(o))(*o)


def batch(lib, dA=FAKE, dB=FAKE, n=4, count=2, proofs=FAKE, proof_len=5, results=FAKE, fins=(FAKE, FAKE, FAKE)):
    return lib.sipp_verify_native_batch_device(dA, dB, n, count, proofs, proof_len, results, *fins)


def ragged(lib, dA=FAKE, dB=FAKE, n=6, offs=N_OFFS, count=2, proofs=FAKE, poffs=N_POFFS, results=FAKE, fins=(FAKE, FAKE, FAKE)):
    return lib.sipp_verify_native_batch_ragged_device(dA, dB, n, None if offs is None else _szt(*offs), count, proofs,
                                                      None if poffs is None else _szt(*poffs), results, *fins)


def test_batch_argument_errors(lib):
    """batch_args' checks, then a NULL d_results, then the proof length"""
    from sipp_b200 import _lib
    assert batch(lib, dA=None) == _lib.ERR_ARG
    assert batch(lib, dB=None) == _lib.ERR_ARG
    assert batch(lib, proofs=None) == _lib.ERR_ARG
    assert batch(lib, count=0) == _lib.ERR_ARG
    for n in (0, 3, 6, 12):
        assert batch(lib, n=n) == _lib.ERR_ARG
    assert batch(lib, results=None) == _lib.ERR_ARG
    assert batch(lib, proof_len=4) == _lib.ERR_SHORT_PROOF                  # 4 < sipp_proof_len(4) = 5
    assert batch(lib, n=1, proof_len=0) == _lib.ERR_SHORT_PROOF
    # the order: batch_args before the NULL results, both before the proof length
    assert batch(lib, dA=None, results=None, proof_len=0) == _lib.ERR_ARG
    assert batch(lib, n=3, proof_len=0) == _lib.ERR_ARG
    assert batch(lib, results=None, proof_len=0) == _lib.ERR_ARG
    assert "results" in lib.sipp_last_error().decode()


def test_ragged_argument_errors(lib):
    """ragged_args, then ragged_verify_args, unchanged from the host form"""
    from sipp_b200 import _lib
    assert ragged(lib, dA=None) == _lib.ERR_ARG
    assert ragged(lib, dB=None) == _lib.ERR_ARG
    assert ragged(lib, offs=None) == _lib.ERR_ARG
    assert ragged(lib, proofs=None) == _lib.ERR_ARG
    assert ragged(lib, count=0) == _lib.ERR_ARG
    assert ragged(lib, offs=(1, 2, 6)) == _lib.ERR_ARG                          # offsets[0] != 0
    assert ragged(lib, offs=(0, 4, 2, 6), count=3, poffs=(0, 5, 8, 11)) == _lib.ERR_ARG   # decreasing
    assert ragged(lib, offs=(0, 2, 4)) == _lib.ERR_ARG                          # offsets[count] != n
    assert ragged(lib, offs=(0, 0, 2, 6), count=3, poffs=(0, 1, 4, 9)) == _lib.ERR_ARG   # an empty instance
    assert ragged(lib, offs=(0, 3, 6)) == _lib.ERR_ARG                          # not a power of two
    big = 1 << 32                                                                # more than 2^32 - 1 pairs (never read)
    assert ragged(lib, n=big, offs=(0, big), count=1, poffs=(0, 65)) == _lib.ERR_ARG
    assert ragged(lib, results=None) == _lib.ERR_ARG
    assert ragged(lib, poffs=None) == _lib.ERR_ARG
    assert ragged(lib, poffs=(1, 3, 8)) == _lib.ERR_ARG                         # proof_offsets[0] != 0
    assert ragged(lib, poffs=(0, 9, 8)) == _lib.ERR_ARG                         # decreasing
    assert ragged(lib, poffs=(0, 2, 8)) == _lib.ERR_SHORT_PROOF                 # proof 0: 2 < 3 elements
    assert ragged(lib, poffs=(0, 3, 7)) == _lib.ERR_SHORT_PROOF                 # proof 1: 4 < 5 elements
    assert ragged(lib, n=2, offs=(0, 1, 2), poffs=(0, 0, 1)) == _lib.ERR_SHORT_PROOF   # n = 1 reads one element
    # the order: the offsets before the proof offsets and results, the proof-offset order before any length
    assert ragged(lib, offs=(0, 3, 6), poffs=(0, 0, 0), results=None) == _lib.ERR_ARG
    assert "prove_native_batch_ragged" in lib.sipp_last_error().decode()
    assert ragged(lib, poffs=(0, 2, 1)) == _lib.ERR_ARG


def test_no_gpu_fails_loudly(lib):
    """valid calls without a device return SIPP_ERR_CUDA (longer proofs and NULL finals are valid arguments)"""
    import sipp_b200
    from sipp_b200 import _lib
    if lib.sipp_device_count() > 0:
        pytest.skip("a GPU is present")
    assert batch(lib) == _lib.ERR_CUDA
    assert batch(lib, proof_len=9, fins=(None, None, None)) == _lib.ERR_CUDA
    assert ragged(lib) == _lib.ERR_CUDA
    assert ragged(lib, poffs=(0, 4, 12), fins=(None, FAKE, None)) == _lib.ERR_CUDA
    with pytest.raises(sipp_b200.SippError) as ei:
        sipp_b200.sipp_verify_native_batch_device(FAKE, FAKE, 4, 2, FAKE, 5, FAKE)
    assert ei.value.code == _lib.ERR_CUDA
    with pytest.raises(sipp_b200.SippError) as ei:
        sipp_b200.sipp_verify_native_batch_ragged_device(FAKE, FAKE, 6, [2, 4], FAKE, [3, 5], FAKE)
    assert ei.value.code == _lib.ERR_CUDA


def test_python_argument_errors():
    import sipp_b200
    f = sipp_b200.sipp_verify_native_batch_ragged_device
    for lengths in ([3, 3], [6], [0, 2, 4], [-2, 8], [2, 2]):                    # as sipp_verify_native_batch_ragged
        with pytest.raises(ValueError):
            f(FAKE, FAKE, 6, lengths, FAKE, [3, 5], FAKE)
    with pytest.raises(ValueError):
        f(FAKE, FAKE, 0, [], FAKE, [], FAKE)                                      # no instances
    for plens in ([3], [3, 5, 1]):                                                # one proof length per instance
        with pytest.raises(ValueError):
            f(FAKE, FAKE, 6, [2, 4], FAKE, plens, FAKE)
    with pytest.raises(ValueError):
        f(FAKE, FAKE, 6, [2, 4], FAKE, [-3, 11], FAKE)                            # a negative proof length
