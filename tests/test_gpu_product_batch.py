"""Batched independent products on the GPU (sipp_inner_product_batch, sipp_inner_product_batch_device, sipp_pairing_batch): every
output against the oracle and against the one-product calls, at scale against the Z of the batched prover, under each option that
changes which kernels run, and the error behaviour of the whole call."""
import ctypes
import os
import random

import pytest

pytestmark = pytest.mark.gpu
H = bytes.fromhex
P = 0x30644E72E131A029B85045B68181585D97816A916871CA8D3C208C16D87CFD47
R = 0x30644E72E131A029B85045B68181585D2833E84879B9709143E1F593F0000001
ONE12 = (1).to_bytes(32, "little") + bytes(352)
THREADS = os.cpu_count() or 1

# every option of include/sipp_b200.h with its default
DEFAULTS = {1: 0, 2: 0, 3: 0, 4: 1, 5: 8192, 6: 1, 7: 256, 8: 1536, 9: 32, 10: 1, 11: 0, 12: 1, 13: 1, 14: 32, 15: 256, 16: 8, 17: 1, 18: 0}
RAGGED = [0, 1, 2, 3, 5, 7, 8, 31, 64, 100, 129, 0, 1500]
# a twist point (on y^2 = x^3 + 3/xi) outside the order-r subgroup (tests/test_gpu_parity.py)
TWIST_NOT_G2 = H("fbee9e35ab3c0ac619c62937bfe3caf537f37ffb5991752a801d56df83aea70a5de70f4aba744b50f26b23f62869ea32968c0a8a8e5449e0444c86ada8f60b28"
                 "b220740d239210aa74480d7e4ebe546a6b9f5fa2f8cf8c0a0a4580f18c2e612775f82b46ee8dc7599bf9c136ec784e777e061d68a3c8d110c06b2a0e0d572002")


def le(v): return v.to_bytes(32, "little")


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
    """every test starts from the defaults and leaves the options as it found them"""
    from sipp_b200 import _lib
    saved = {o: lib.sipp_get_option(o) for o in DEFAULTS}
    try:
        for o, v in DEFAULTS.items():
            _lib.check(lib.sipp_set_option(o, v))
        yield
    finally:
        for o, v in saved.items():
            _lib.check(lib.sipp_set_option(o, v))


def segments(A, B, lengths):
    out, pos = [], 0
    for length in lengths:
        out.append((A[64 * pos:64 * (pos + length)], B[128 * pos:128 * (pos + length)]))
        pos += length
    return out


def offsets(lengths):
    o = [0]
    for length in lengths:
        o.append(o[-1] + length)
    return o


def ragged_inputs(sipp):
    """seeded points for RAGGED with identity points planted inside segments: an A, a B, and both halves of a one-pair segment"""
    o = offsets(RAGGED)
    A, B = sipp.seeded_inputs(61, o[-1])
    A, B = bytearray(A), bytearray(B)
    A[64 * (o[4] + 2):64 * (o[4] + 3)] = bytes(64)          # A inside the 5-pair segment
    B[128 * (o[9] + 50):128 * (o[9] + 51)] = bytes(128)     # B inside the 100-pair segment
    A[64 * o[1]:64 * (o[1] + 1)] = bytes(64)                # the whole 1-pair segment: e(O, O)
    B[128 * o[1]:128 * (o[1] + 1)] = bytes(128)
    B[128 * (o[12] + 700):128 * (o[12] + 701)] = bytes(128)  # and one in the long segment
    return bytes(A), bytes(B)


@pytest.mark.parametrize("fe_norm", [0, 1], ids=["exact", "ark"])
def test_ragged_matches_oracle_and_single(sipp, oracle, fe_norm):
    """every output == oracle.inner_product of its segment == sipp.inner_product on it, under both FE normalisations (H1)"""
    from sipp_b200 import _lib
    sipp.set_option(_lib.OPT_FE_NORMALISATION, fe_norm)
    A, B = ragged_inputs(sipp)
    out = sipp.inner_product_batch(A, B, RAGGED)
    assert len(out) == len(RAGGED)
    for j, (a, b) in enumerate(segments(A, B, RAGGED)):
        assert out[j] == sipp.inner_product(a, b), j
        assert out[j] == oracle.inner_product(a, b, opts=oracle.FE_ARK if fe_norm else 0, threads=THREADS), j
    assert out[0] == out[1] == out[11] == ONE12


def test_pairing_batch_golden(sipp, oracle, golden):
    """pairing_batch == the committed pairings (both normalisations) and the oracle"""
    from sipp_b200 import _lib
    g, rs = golden["pairing_gen"], golden["pairing_random"]
    a = [H(g["a"])] + [H(c["a"]) for c in rs]
    b = [H(g["b"])] + [H(c["b"]) for c in rs]
    assert sipp.pairing_batch(a, b) == [H(g["exact"])] + [H(c["exact"]) for c in rs]
    sipp.set_option(_lib.OPT_FE_NORMALISATION, 1)
    assert sipp.pairing_batch(a[:1], b[:1]) == [H(g["ark"])]
    sipp.set_option(_lib.OPT_FE_NORMALISATION, 0)
    A, B = sipp.seeded_inputs(62, 300)
    out = sipp.pairing_batch(A, B)
    for j in range(0, 300, 23):
        a1, b1 = A[64 * j:64 * (j + 1)], B[128 * j:128 * (j + 1)]
        assert out[j] == oracle.pairing(a1, b1) == sipp.pairing(a1, b1), j


def test_aggregate_scale_equals_batched_z(sipp):
    """4,096 products of 128 pairs (the aggregate-check shape): each == Z (proof[-1]) of the batched prover on the same pairs"""
    n, count = 128, 4096
    A, B = sipp.seeded_inputs(71, n * count)
    out = sipp.inner_product_batch(A, B, [n] * count)
    proofs = sipp.sipp_prove_native_batch(A, B, n)
    bad = [j for j in range(count) if out[j] != proofs[j][-1]]
    assert not bad, bad[:10]


def _plan_chunks(lib, lengths, chunk_pairs):
    o = offsets(lengths)
    arr = (ctypes.c_size_t * len(o))(*o)
    g = lib.sipp_test_product_plan(arr, len(lengths), 32, chunk_pairs, None, 0, None)
    out = (ctypes.c_size_t * (4 * g))()
    assert lib.sipp_test_product_plan(arr, len(lengths), 32, chunk_pairs, out, 4 * g, None) == g
    return [tuple(out[4 * i:4 * i + 4]) for i in range(g)]


@pytest.mark.parametrize("chunk_pairs", [37, 100])
def test_forced_chunks(sipp, lib, chunk_pairs):
    """SIPP_OPT_PRODUCT_CHUNK_PAIRS: segments straddling chunks (groups cut at the boundaries) give the default's bytes"""
    from sipp_b200 import _lib
    lengths = [0, 5, 40, 1, 100, 0, 77, 3, 64, 250]
    A, B = sipp.seeded_inputs(63, sum(lengths))
    want = sipp.inner_product_batch(A, B, lengths)
    groups = _plan_chunks(lib, lengths, chunk_pairs)
    chunks_of_seg = {}
    for _, _, seg, chunk in groups:
        chunks_of_seg.setdefault(seg, set()).add(chunk)
    assert max(len(c) for c in chunks_of_seg.values()) >= 3 and max(g[3] for g in groups) >= 5
    sipp.set_option(_lib.OPT_PRODUCT_CHUNK_PAIRS, chunk_pairs)
    sipp.stats(reset=True)
    assert sipp.inner_product_batch(A, B, lengths) == want
    assert sipp.stats()["miller_launches"] == max(g[3] for g in groups) + 1
    assert want[9] == sipp.inner_product(*segments(A, B, lengths)[9])


@pytest.mark.parametrize("option,value", [(6, 0), (6, 1), (5, 0), (5, 8192), (9, 1), (9, 32)],
                         ids=["fe-engine-0", "fe-engine-1", "wide-lines-0", "wide-lines-default", "kpg-max-1", "kpg-max-32"])
def test_option_variants(sipp, option, value):
    """SIPP_OPT_FE_ENGINE, SIPP_OPT_WIDE_LINES_MAX and SIPP_OPT_BATCH_KPG_MAX change kernels, not bytes; SIPP_OPT_PIPELINE is not read"""
    A, B = ragged_inputs(sipp)
    want = sipp.inner_product_batch(A, B, RAGGED)
    sipp.set_option(option, value)
    assert sipp.inner_product_batch(A, B, RAGGED) == want
    sipp.set_option(4, 0)
    assert sipp.inner_product_batch(A, B, RAGGED) == want


def test_skewed(sipp):
    """one 2^14 segment (several passes of the segmented product) among many short ones == sipp.inner_product per segment"""
    rng = random.Random(64)
    lengths = [rng.randrange(0, 65) for _ in range(200)]
    lengths.insert(77, 1 << 14)
    A, B = sipp.seeded_inputs(64, sum(lengths))
    out = sipp.inner_product_batch(A, B, lengths)
    for j, (a, b) in enumerate(segments(A, B, lengths)):
        assert out[j] == sipp.inner_product(a, b), j


def test_device_form_equals_host_form(sipp):
    import torch
    A, B = ragged_inputs(sipp)
    n = sum(RAGGED)
    dA = torch.frombuffer(bytearray(A), dtype=torch.uint8).cuda()
    dB = torch.frombuffer(bytearray(B), dtype=torch.uint8).cuda()
    dO = torch.zeros(len(RAGGED) * 384, dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()
    sipp.inner_product_batch_device(dA.data_ptr(), dB.data_ptr(), n, RAGGED, dO.data_ptr())
    torch.cuda.synchronize()
    assert dO.cpu().numpy().tobytes() == b"".join(sipp.inner_product_batch(A, B, RAGGED))


def test_bad_points_and_empty_batches(sipp, lib):
    """a bad point fails the whole call (SIPP_ERR_ENCODING, nothing written); trusted inputs pass; count == 0 and all-empty batches"""
    from sipp_b200 import _lib
    lengths = [5, 0, 15]
    A, B = sipp.seeded_inputs(65, 20)

    def refused(a, b, what):
        out = ctypes.create_string_buffer(3 * 384)
        o = (ctypes.c_size_t * 4)(*offsets(lengths))
        assert lib.sipp_inner_product_batch(a, 20, b, 20, o, 3, out) == _lib.ERR_ENCODING
        assert what in lib.sipp_last_error().decode() and out.raw == bytes(3 * 384)
    bad = bytearray(A); bad[64 * 3 + 32] ^= 1                 # y of A_3: off the curve
    refused(bytes(bad), B, "not on the curve")
    bad = bytearray(A); bad[64 * 7:64 * 7 + 32] = le(P)       # x == p: not canonical
    refused(bytes(bad), B, "coordinate >= p")
    badB = bytearray(B); badB[128 * 12:128 * 13] = TWIST_NOT_G2
    refused(A, bytes(badB), "subgroup")
    sipp.set_option(_lib.OPT_VALIDATE_POINTS, 0)
    out = sipp.inner_product_batch(A, bytes(badB), lengths)   # trusted inputs: no check, same kernels as the one-product call
    assert out[2] == sipp.inner_product(A[64 * 5:], bytes(badB)[128 * 5:]) and out[1] == ONE12
    sipp.set_option(_lib.OPT_VALIDATE_POINTS, 1)
    assert sipp.inner_product_batch(b"", b"", []) == []
    o = (ctypes.c_size_t * 1)(0)
    assert lib.sipp_inner_product_batch(None, 0, None, 0, o, 0, None) == _lib.OK
    assert sipp.inner_product_batch(b"", b"", [0, 0, 0]) == [ONE12] * 3
    assert sipp.inner_product_batch(A[:64], B[:128], [0, 1, 0]) == [ONE12, sipp.pairing(A[:64], B[:128]), ONE12]


def test_bls_aggregate_checks_as_segments(sipp, golden):
    """the BLS-demo instance of tests/test_gpu_parity.py::test_bls_aggregation_demo and its forged variant as two segments of one
    call: inner_product(pk || -G1, m || sigma) == 1 for the honest aggregate only"""
    n = 128
    rng = random.Random(24)
    g2 = H(golden["pairing_gen"]["b"])
    sks = [le(rng.randrange(1, R)) for _ in range(n - 1)]
    pks = sipp.g1_generator_mul_batch(sks)
    ms = sipp.g2_mul_batch(g2, [le(rng.randrange(1, R)) for _ in range(n - 1)])
    sigs = sipp.g2_mul_batch(ms, sks)
    A2 = b"".join(pks) + sipp.g1_neg_generator()
    B2 = b"".join(ms) + sipp.g2_sum(sigs)
    forged = b"".join(ms) + sipp.g2_sum(sigs[1:])
    out = sipp.inner_product_batch(A2 + A2, B2 + forged, [n, n])
    assert out[0] == ONE12 and out[1] != ONE12
    assert out[1] == sipp.inner_product(A2, forged)


def test_stats_and_profile(sipp):
    """miller_pairs grows by the pair count; SIPP_OPT_PROFILE times lines + accumulation and reduction + final exponentiation"""
    from sipp_b200 import _lib
    A, B = ragged_inputs(sipp)
    sipp.stats(reset=True)
    sipp.inner_product_batch(A, B, RAGGED)
    assert sipp.stats()["miller_pairs"] == sum(RAGGED)
    sipp.set_option(_lib.OPT_PROFILE, 1)
    sipp.stats(reset=True)
    sipp.pairing_batch(A[:64 * 10], B[:128 * 10])
    st = sipp.stats(reset=True)
    assert st["miller_pairs"] == 10 and st["miller_ms"] > 0 and st["reduce_fe_ms"] > 0
