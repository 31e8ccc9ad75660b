"""Proof and statement in one call: sipp_prove_native_statement, sipp_prove_native_batch_statement(_device) and
sipp_prove_native_batch_ragged_statement(_device).  Every proof must equal the sibling prover's, and every (final_A, final_B, final_Z)
must equal what sipp_verify_native writes for that proof, under the option values that change the single prover's code path, the
oracle's under all four H1 / H2 conventions, and the batched verifiers'.  NULL finals, bad points and the stats are covered too."""
import ctypes
import os
import random

import pytest

pytestmark = pytest.mark.gpu
THREADS = os.cpu_count() or 1
P = 0x30644E72E131A029B85045B68181585D97816A916871CA8D3C208C16D87CFD47

# every option of include/sipp_b200.h with its default
DEFAULTS = {1: 0, 2: 0, 3: 0, 4: 1, 5: 8192, 6: 1, 7: 256, 8: 1536, 9: 32, 10: 1, 11: 0, 12: 1, 13: 1, 14: 32, 15: 256, 16: 8, 17: 1, 18: 0}
MIXED = [1 << k for k in range(11)]   # 1, 2, 4, ..., 1024
SIZES = [1 << k for k in range(13)]   # 1 .. 4096
# the option values that change which code the single prover runs at the end of a proof (SIPP_OPT_MATRIX_TAIL 14,
# SIPP_OPT_MATRIX_FIRST 17, SIPP_OPT_MATRIX_BLOCK_N 15, SIPP_OPT_PIPELINE 4, SIPP_OPT_FE_ENGINE 6, SIPP_OPT_VALIDATE_POINTS 13)
SINGLE_OPTS = [("defaults", {}), ("tail_0", {14: 0}), ("tail_2", {14: 2}), ("tail_4", {14: 4}), ("tail_64", {14: 64}), ("first_0", {17: 0}),
               ("block_n_0", {15: 0}), ("pipeline_0", {4: 0}), ("fe_engine_0", {6: 0}), ("validate_0", {13: 0})]
UNTOUCHED = b"\xa5"


@pytest.fixture(scope="module")
def sipp():
    import sipp_b200
    from sipp_b200 import _lib
    _lib.require_gpu_once()
    return sipp_b200


@pytest.fixture(scope="module")
def lib(sipp):
    from sipp_b200 import _lib
    return _lib.load()


@pytest.fixture(autouse=True)
def options(lib):
    """every test starts from the defaults, whatever earlier tests left, and leaves the options as it found them"""
    from sipp_b200 import _lib
    saved = {o: lib.sipp_get_option(o) for o in DEFAULTS}
    try:
        for o, v in DEFAULTS.items():
            _lib.check(lib.sipp_set_option(o, v))
        yield
    finally:
        for o, v in saved.items():
            _lib.check(lib.sipp_set_option(o, v))


@pytest.fixture(scope="module")
def inputs(sipp):
    return sipp.seeded_inputs(300, 4096)


def offsets(lengths):
    o = [0]
    for length in lengths:
        o.append(o[-1] + length)
    return o


def split(A, B, lengths):
    o = offsets(lengths)
    return [(A[64 * o[j]:64 * o[j + 1]], B[128 * o[j]:128 * o[j + 1]]) for j in range(len(lengths))]


def proof_len(n):
    return 2 * (n.bit_length() - 1) + 1


def sentinel(k):
    return ctypes.create_string_buffer(UNTOUCHED * k, k)


def single(lib, a, b, finals=(1, 1, 1)):
    """sipp_prove_native_statement: (return value, proof bytes, (final_A, final_B, final_Z)) with sentinel-filled outputs"""
    n = len(a) // 64
    pf = sentinel(384 * proof_len(n))
    fins = [sentinel(k) for k in (64, 128, 384)]
    rc = lib.sipp_prove_native_statement(a, n, b, n, pf, *[f if on else None for f, on in zip(fins, finals)])
    return rc, pf.raw, tuple(f.raw for f in fins)


def native_verify(lib, a, b, proof):
    fa, fb, fz = (ctypes.create_string_buffer(k) for k in (64, 128, 384))
    rc = lib.sipp_verify_native(a, len(a) // 64, b, len(b) // 128, proof, len(proof) // 384, fa, fb, fz)
    return rc, (fa.raw, fb.raw, fz.raw)


def batch(lib, A, B, n, finals=(1, 1, 1)):
    count = len(A) // (64 * n)
    pf = sentinel(384 * proof_len(n) * count)
    fins = [sentinel(k * count) for k in (64, 128, 384)]
    rc = lib.sipp_prove_native_batch_statement(A, B, n, count, pf, *[f if on else None for f, on in zip(fins, finals)])
    return rc, pf.raw, [tuple(f.raw[k * j:k * (j + 1)] for f, k in zip(fins, (64, 128, 384))) for j in range(count)]


def ragged(lib, A, B, lengths, finals=(1, 1, 1)):
    count, n = len(lengths), len(A) // 64
    pf = sentinel(384 * sum(proof_len(x) for x in lengths))
    fins = [sentinel(k * count) for k in (64, 128, 384)]
    rc = lib.sipp_prove_native_batch_ragged_statement(A, n, B, n, (ctypes.c_size_t * (count + 1))(*offsets(lengths)), count, pf,
                                                      *[f if on else None for f, on in zip(fins, finals)])
    return rc, pf.raw, [tuple(f.raw[k * j:k * (j + 1)] for f, k in zip(fins, (64, 128, 384))) for j in range(count)]


def ragged_verify_finals(sipp, A, B, lengths, proofs):
    sts = sipp.sipp_verify_native_batch_ragged(A, B, lengths, proofs)
    assert all(isinstance(s, sipp.SIPPStatement) for s in sts)
    return [(s.final_A, s.final_B, s.final_Z) for s in sts]


@pytest.mark.parametrize("name,opts", SINGLE_OPTS, ids=[o[0] for o in SINGLE_OPTS])
def test_single_matches_prover_and_verifier(sipp, lib, inputs, name, opts):
    """n = 1 .. 2^12: the proof is sipp_prove_native's and the finals are sipp_verify_native's on it"""
    for o, v in opts.items():
        sipp.set_option(o, v)
    A, B = inputs
    for n in SIZES:
        a, b = A[:64 * n], B[:128 * n]
        rc, pf, fins = single(lib, a, b)
        assert rc == 0, (name, n)
        assert pf == b"".join(sipp.sipp_prove_native(a, b)), (name, n)
        vrc, want = native_verify(lib, a, b, pf)
        assert vrc == 0 and fins == want, (name, n)


def test_single_large(sipp, lib):
    A, B = sipp.seeded_inputs(301, 1 << 16)
    rc, pf, fins = single(lib, A, B)
    assert rc == 0
    assert pf == b"".join(sipp.sipp_prove_native(A, B))
    assert native_verify(lib, A, B, pf) == (0, fins)


@pytest.mark.parametrize("conv", [0, 1, 2, 3], ids=["default", "ark-normalisation", "nested-order", "ark-nested"])
def test_conventions_against_oracle(sipp, lib, oracle, conv):
    """n <= 64 under each H1 / H2 convention: the proof is the oracle's and the finals are pyoracle.sipp_verify's"""
    sipp.set_option(1, conv & 1)
    sipp.set_option(2, conv >> 1)
    A, B = oracle.seeded_inputs(302 + conv, 95, threads=THREADS)
    for n in (1, 2, 4, 8, 16, 32, 64):
        a, b = A[:64 * n], B[:128 * n]
        rc, pf, fins = single(lib, a, b)
        assert rc == 0
        assert pf == oracle.sipp_prove(a, b, opts=conv, threads=THREADS), (conv, n)
        ok, fin = oracle.sipp_verify(a, b, pf, opts=conv, threads=THREADS)
        assert ok and fins == (fin["final_A"], fin["final_B"], fin["final_Z"]), (conv, n)
    lengths = [16, 1, 4, 64, 2, 8]
    rc, pf, fins = ragged(lib, A, B, lengths)
    assert rc == 0
    for j, (a, b) in enumerate(split(A, B, lengths)):
        ok, fin = oracle.sipp_verify(a, b, oracle.sipp_prove(a, b, opts=conv, threads=THREADS), opts=conv, threads=THREADS)
        assert ok and fins[j] == (fin["final_A"], fin["final_B"], fin["final_Z"]), (conv, j)


@pytest.mark.parametrize("n", [1, 2, 128])
@pytest.mark.parametrize("count", [1, 3, 64])
def test_uniform_batch(sipp, lib, n, count):
    A, B = sipp.seeded_inputs(303 + n + count, n * count)
    rc, pf, fins = batch(lib, A, B, n)
    assert rc == 0
    proofs = sipp.sipp_prove_native_batch(A, B, n)
    assert pf == b"".join(b"".join(p) for p in proofs)
    sts = sipp.sipp_verify_native_batch(A, B, n, proofs)
    assert fins == [(s.final_A, s.final_B, s.final_Z) for s in sts]
    for j, (a, b) in enumerate(split(A, B, [n] * count)):
        assert native_verify(lib, a, b, b"".join(proofs[j])) == (0, fins[j]), j


def test_uniform_batch_sub_streams(sipp, lib):
    """SIPP_OPT_BATCH_STREAMS 4: the finals are read after every sub-batch stream has joined"""
    n, count = 16, 256
    A, B = sipp.seeded_inputs(304, n * count)
    want = batch(lib, A, B, n)
    sipp.set_option(11, 4)
    assert batch(lib, A, B, n) == want
    sts = sipp.sipp_verify_native_batch(A, B, n, sipp.sipp_prove_native_batch(A, B, n))
    assert want[2] == [(s.final_A, s.final_B, s.final_Z) for s in sts]


def test_ragged_mixed_shuffled(sipp, lib):
    lengths = MIXED + MIXED[::2]
    random.Random(305).shuffle(lengths)
    A, B = sipp.seeded_inputs(305, sum(lengths))
    rc, pf, fins = ragged(lib, A, B, lengths)
    assert rc == 0
    proofs = sipp.sipp_prove_native_batch_ragged(A, B, lengths)
    assert pf == b"".join(b"".join(p) for p in proofs)
    assert fins == ragged_verify_finals(sipp, A, B, lengths, proofs)
    for j in random.Random(306).sample(range(len(lengths)), 5):
        a, b = split(A, B, lengths)[j]
        assert native_verify(lib, a, b, b"".join(proofs[j])) == (0, fins[j]), j


def test_ragged_big_among_small(sipp, lib):
    lengths = [16] * 60 + [4096] + [16] * 67
    A, B = sipp.seeded_inputs(307, sum(lengths))
    rc, pf, fins = ragged(lib, A, B, lengths)
    assert rc == 0
    proofs = sipp.sipp_prove_native_batch_ragged(A, B, lengths)
    assert pf == b"".join(b"".join(p) for p in proofs)
    assert fins == ragged_verify_finals(sipp, A, B, lengths, proofs)


def test_device_forms_match_host_forms(sipp, lib):
    import torch
    dev = torch.device("cuda", 0)

    def to_dev(x):
        return torch.frombuffer(bytearray(x), dtype=torch.uint8).to(dev)

    def run_dev(call, np, count):
        out = [torch.full((k,), 0xa5, dtype=torch.uint8, device=dev) for k in (384 * np, 64 * count, 128 * count, 384 * count)]
        call(*[t.data_ptr() for t in out])
        torch.cuda.synchronize()
        return [bytes(t.cpu().numpy()) for t in out]

    n, count = 8, 5
    A, B = sipp.seeded_inputs(308, n * count)
    dA, dB = to_dev(A), to_dev(B)
    rc, pf, fins = batch(lib, A, B, n)
    assert rc == 0
    got = run_dev(lambda p, fa, fb, fz: sipp.sipp_prove_native_batch_statement_device(dA.data_ptr(), dB.data_ptr(), n, count, p, fa, fb, fz),
                  proof_len(n) * count, count)
    assert got == [pf, b"".join(f[0] for f in fins), b"".join(f[1] for f in fins), b"".join(f[2] for f in fins)]
    lengths = [4, 1, 32, 2, 8]
    A, B = sipp.seeded_inputs(309, sum(lengths))
    dA, dB = to_dev(A), to_dev(B)
    rc, pf, fins = ragged(lib, A, B, lengths)
    assert rc == 0
    got = run_dev(lambda p, fa, fb, fz: sipp.sipp_prove_native_batch_ragged_statement_device(dA.data_ptr(), dB.data_ptr(), sum(lengths), lengths,
                                                                                            p, fa, fb, fz),
                  sum(proof_len(x) for x in lengths), len(lengths))
    assert got == [pf, b"".join(f[0] for f in fins), b"".join(f[1] for f in fins), b"".join(f[2] for f in fins)]
    # a final not wanted (NULL) stays untouched
    got = run_dev(lambda p, fa, fb, fz: sipp.sipp_prove_native_batch_ragged_statement_device(dA.data_ptr(), dB.data_ptr(), sum(lengths), lengths,
                                                                                            p, fa, 0, fz),
                  sum(proof_len(x) for x in lengths), len(lengths))
    assert got[0] == pf and got[2] == UNTOUCHED * 128 * len(lengths) and got[3] == b"".join(f[2] for f in fins)


@pytest.mark.parametrize("opts", [{}, {14: 0}], ids=["tail", "no_tail"])
def test_null_finals(sipp, lib, inputs, opts):
    """one NULL final at a time: the others are unchanged and the NULL one is not written"""
    for o, v in opts.items():
        sipp.set_option(o, v)
    A, B = inputs
    a, b = A[:64 * 256], B[:128 * 256]
    lengths = [8, 1, 64, 2]
    full = (single(lib, a, b), batch(lib, A[:64 * 96], B[:128 * 96], 32), ragged(lib, A[:64 * 75], B[:128 * 75], lengths))
    for k in range(3):
        finals = tuple(int(i != k) for i in range(3))
        got = (single(lib, a, b, finals), batch(lib, A[:64 * 96], B[:128 * 96], 32, finals), ragged(lib, A[:64 * 75], B[:128 * 75], lengths, finals))
        for (rc, pf, fins), (wrc, wpf, wfins) in zip(got, full):
            assert rc == wrc == 0 and pf == wpf
            fl = fins if isinstance(fins, list) else [fins]
            wfl = wfins if isinstance(wfins, list) else [wfins]
            for f, w in zip(fl, wfl):
                for i in range(3):
                    assert f[i] == (UNTOUCHED * len(w[i]) if i == k else w[i]), (k, i)


def test_bad_point_writes_nothing(sipp, lib, inputs):
    """a point off the curve or a coordinate >= p fails every call with SIPP_ERR_ENCODING; proofs and finals keep their sentinels"""
    from sipp_b200 import _lib
    A, B = inputs
    for where in ("off_curve", "coordinate"):
        a, b = bytearray(A[:64 * 64]), bytearray(B[:128 * 64])
        if where == "off_curve":
            a[64 * 9 + 32] ^= 1                          # y of A_9
        else:
            b[128 * 9:128 * 9 + 32] = P.to_bytes(32, "little")   # x.c0 of B_9 == p
        a, b = bytes(a), bytes(b)
        for n in (64, 16):  # a first stage, then a tail stage; a whole-proof matrix of the inputs
            rc, pf, fins = single(lib, a[:64 * n], b[:128 * n])
            assert rc == _lib.ERR_ENCODING, (where, n)
            assert pf == UNTOUCHED * len(pf) and fins == (UNTOUCHED * 64, UNTOUCHED * 128, UNTOUCHED * 384), (where, n)
        rc, pf, fins = batch(lib, a, b, 16)
        assert rc == _lib.ERR_ENCODING and pf == UNTOUCHED * len(pf)
        assert fins == [(UNTOUCHED * 64, UNTOUCHED * 128, UNTOUCHED * 384)] * 4
        rc, pf, fins = ragged(lib, a, b, [32, 1, 16, 8, 4, 2, 1])
        assert rc == _lib.ERR_ENCODING and pf == UNTOUCHED * len(pf)
        assert fins == [(UNTOUCHED * 64, UNTOUCHED * 128, UNTOUCHED * 384)] * 7
    assert single(lib, A[:64 * 64], B[:128 * 64])[0] == 0   # a good call follows


def test_python_statements(sipp, inputs):
    """the wrappers' statements equal sipp_verify_native's field for field, to_vec() included"""
    A, B = inputs
    for n in (1, 32, 512):
        a, b = A[:64 * n], B[:128 * n]
        proof, st = sipp.sipp_prove_native_statement(a, b)
        assert proof == sipp.sipp_prove_native(a, b)
        want = sipp.sipp_verify_native(a, b, proof)
        assert st == want and st.to_vec() == want.to_vec(), n
    for (proof, st), (a, b) in zip(sipp.sipp_prove_native_batch_statement(A[:64 * 48], B[:128 * 48], 16), split(A[:64 * 48], B[:128 * 48], [16] * 3)):
        want = sipp.sipp_verify_native(a, b, proof)
        assert st == want and st.to_vec() == want.to_vec()
    lengths = [4, 64, 1, 16]
    pairs = sipp.sipp_prove_native_batch_ragged_statement(A[:64 * 85], B[:128 * 85], lengths)
    for (proof, st), (a, b) in zip(pairs, split(A[:64 * 85], B[:128 * 85], lengths)):
        want = sipp.sipp_verify_native(a, b, proof)
        assert st == want and st.to_vec() == want.to_vec()


@pytest.mark.parametrize("opts,extra", [({}, 0), ({14: 0}, 1)], ids=["tail", "no_tail"])
def test_stats(sipp, lib, inputs, opts, extra):
    """miller_pairs: as the sibling prover, plus count on the batched paths and 1 on the single path without a tail stage;
    fold_points: as the sibling prover"""
    for o, v in opts.items():
        sipp.set_option(o, v)
    A, B = inputs

    def counts(call):
        sipp.stats(reset=True)
        call()
        st = sipp.stats(reset=True)
        return st["miller_pairs"], st["fold_points"]

    def check(got, want, extra_pairs):
        assert got == (want[0] + extra_pairs, want[1])

    a, b = A[:64 * 128], B[:128 * 128]
    plain = counts(lambda: sipp.sipp_prove_native(a, b))
    check(counts(lambda: single(lib, a, b)), plain, extra)
    check(counts(lambda: single(lib, a, b, (1, 1, 0))), plain, 0)
    A2, B2 = A[:64 * 96], B[:128 * 96]
    check(counts(lambda: batch(lib, A2, B2, 32)), counts(lambda: sipp.sipp_prove_native_batch(A2, B2, 32)), 3)
    lengths = [8, 1, 64, 2]
    A3, B3 = A[:64 * 75], B[:128 * 75]
    check(counts(lambda: ragged(lib, A3, B3, lengths)), counts(lambda: sipp.sipp_prove_native_batch_ragged(A3, B3, lengths)), 4)
