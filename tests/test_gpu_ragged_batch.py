"""Ragged batched proving (sipp_prove_native_batch_ragged): independent instances of different sizes in lock-step, byte for byte
against sipp_prove_native on each instance, the uniform batched prover, the CPU oracle (both H1 / H2 alternatives) and the golden
proofs.  The schedule hook (sipp_test_ragged_schedule) asserts which fold kernel every shape reaches, so that a later change of a
threshold cannot turn a test into a no-op."""
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


def offsets(lengths):
    o = [0]
    for length in lengths:
        o.append(o[-1] + length)
    return o


def split(A, B, lengths):
    o = offsets(lengths)
    return [(A[64 * o[j]:64 * o[j + 1]], B[128 * o[j]:128 * o[j + 1]]) for j in range(len(lengths))]


def schedule(lib, lengths):
    o = offsets(lengths)
    arr = (ctypes.c_size_t * len(o))(*o)
    rounds = lib.sipp_test_ragged_schedule(arr, len(lengths), None, 0)
    assert rounds > 0
    out = (ctypes.c_longlong * (5 * rounds))()
    assert lib.sipp_test_ragged_schedule(arr, len(lengths), out, 5 * rounds) == rounds
    return [tuple(out[5 * r:5 * r + 5]) for r in range(rounds)]


def kernels(lib, lengths):
    return {r[3] for r in schedule(lib, lengths)[1:]}


def by_size(sipp, A, B, lengths):
    """the reference: one uniform batched call per distinct size, proofs back in the instances' order"""
    inst = split(A, B, lengths)
    out = [None] * len(lengths)
    for n in sorted(set(lengths)):
        js = [j for j in range(len(lengths)) if lengths[j] == n]
        proofs = sipp.sipp_prove_native_batch(b"".join(inst[j][0] for j in js), b"".join(inst[j][1] for j in js), n)
        for j, p in zip(js, proofs):
            out[j] = p
    return out


@pytest.fixture(scope="module")
def pool(sipp):
    """the instances of MIXED (and a duplicate of each) with their single-proof references"""
    lengths = MIXED + MIXED
    A, B = sipp.seeded_inputs(90, sum(lengths))
    inst = split(A, B, lengths)
    return [(a, b, sipp.sipp_prove_native(a, b)) for a, b in inst]


@pytest.mark.parametrize("order", ["ascending", "descending", "shuffled", "duplicates"])
def test_mixed_sizes_match_single_proofs(sipp, pool, order):
    """every proof == sipp_prove_native on its pairs, whatever the order; a permuted batch gives every instance the same proof"""
    idx = list(range(len(MIXED)))
    if order == "descending":
        idx = idx[::-1]
    elif order == "shuffled":
        random.Random(91).shuffle(idx)
    elif order == "duplicates":
        idx = list(range(2 * len(MIXED)))
        random.Random(92).shuffle(idx)
        idx += idx[:5]
    A = b"".join(pool[i][0] for i in idx)
    B = b"".join(pool[i][1] for i in idx)
    proofs = sipp.sipp_prove_native_batch_ragged(A, B, [len(pool[i][0]) // 64 for i in idx])
    assert len(proofs) == len(idx)
    for j, i in enumerate(idx):
        assert proofs[j] == pool[i][2], (order, j, len(pool[i][0]) // 64)


def test_small_sizes_against_oracle_and_golden(sipp, oracle, golden):
    rng = random.Random(93)
    lengths = [rng.choice([1, 2, 4, 8, 16, 32, 64]) for _ in range(12)]
    A, B = oracle.seeded_inputs(94, sum(lengths), threads=THREADS)
    proofs = sipp.sipp_prove_native_batch_ragged(A, B, lengths)
    for j, (a, b) in enumerate(split(A, B, lengths)):
        assert b"".join(proofs[j]) == oracle.sipp_prove(a, b, threads=THREADS), j
    H = bytes.fromhex
    cases = golden["prove"]
    A = b"".join(H(c["A"]) for c in cases)
    B = b"".join(H(c["B"]) for c in cases)
    proofs = sipp.sipp_prove_native_batch_ragged(A, B, [c["n"] for c in cases])
    for c, p in zip(cases, proofs):
        assert b"".join(p).hex() == c["proof"], c["name"]


@pytest.mark.parametrize("n,count", [(2, 5), (16, 33), (128, 4), (128, 4096)])
def test_equal_sizes_match_uniform_batch(sipp, n, count):
    A, B = sipp.seeded_inputs(95 + n, n * count)
    want = sipp.sipp_prove_native_batch(A, B, n)
    assert sipp.sipp_prove_native_batch_ragged(A, B, [n] * count) == want


def test_unit_and_single_large_instances(sipp, lib):
    """n = 1 only == sipp_pairing_batch; one 2^12 instance alone and among 255 instances of n = 16"""
    A, B = sipp.seeded_inputs(96, 300)
    proofs = sipp.sipp_prove_native_batch_ragged(A, B, [1] * 300)
    assert [p for (p,) in proofs] == sipp.pairing_batch(A, B)
    assert schedule(lib, [1] * 300) == [(300, 300, 0, -1, 1)]
    A, B = sipp.seeded_inputs(97, 4096)
    big = sipp.sipp_prove_native(A, B)
    assert sipp.sipp_prove_native_batch_ragged(A, B, [4096]) == [big]
    A2, B2 = sipp.seeded_inputs(98, 16 * 255)
    lengths = [16] * 100 + [4096] + [16] * 155
    A3 = A2[:64 * 1600] + A + A2[64 * 1600:]
    B3 = B2[:128 * 1600] + B + B2[128 * 1600:]
    proofs = sipp.sipp_prove_native_batch_ragged(A3, B3, lengths)
    assert proofs[100] == big
    small = sipp.sipp_prove_native_batch(A2, B2, 16)
    assert proofs[:100] + proofs[101:] == small


# (name, options, lengths, the fold kernels the rounds must reach)
FOLD_CASES = [
    ("default", {}, [256] * 64 + [128] * 130 + [4, 2, 1], {0, 1, 2}),
    ("no_straus", {10: 0}, [256] * 64 + [128] * 130 + [4, 2, 1], {0, 1}),
    ("wide_fold_max_0", {7: 0}, [64] * 30 + [8] * 5 + [2] * 3, {0, 1}),
    ("wide_fold_max_large", {7: 1 << 20, 10: 0}, [256] * 40 + [16] * 9 + [2] * 7 + [1], {1}),
    # k_fold_batch: one warp holds the end of an h = 2 instance and a run of h = 1 instances
    ("lane_split_mixed_warp", {7: 0}, [1024, 4] + [2] * 40, {0, 1}),
    # k_fold_wide_batch: h = 1 instances right after large ones in the same small round
    ("wide_mixed_h1", {}, [128, 2, 64, 2, 2, 32, 2], {1}),
]


@pytest.mark.parametrize("name,opts,lengths,want", FOLD_CASES, ids=[c[0] for c in FOLD_CASES])
def test_fold_kernels(sipp, lib, name, opts, lengths, want):
    for o, v in opts.items():
        sipp.set_option(o, v)
    assert kernels(lib, lengths) == want
    if name == "lane_split_mixed_warp":
        assert schedule(lib, lengths)[1][2:4] == (512 + 2 + 40, 0)   # elements 512, 513 (h = 2) share a warp with h = 1 ones
    rng = random.Random(hash(name) & 0xffff)
    order = list(range(len(lengths)))
    rng.shuffle(order)
    lengths = [lengths[i] for i in order]
    A, B = sipp.seeded_inputs(99, sum(lengths))
    assert sipp.sipp_prove_native_batch_ragged(A, B, lengths) == by_size(sipp, A, B, lengths)


@pytest.mark.parametrize("opts", [{18: 37}, {18: 100}, {5: 0}, {6: 0}, {9: 1}],
                         ids=["chunk37", "chunk100", "wide_lines_0", "fe_engine_0", "kpg_1"])
def test_product_options(sipp, lib, opts):
    """forced line-table chunks cut through instances; the kernel-selecting options do not change a bit"""
    lengths = [64, 1, 8, 256, 2, 32, 4, 16, 128, 2, 1]
    A, B = sipp.seeded_inputs(100, sum(lengths))
    want = sipp.sipp_prove_native_batch_ragged(A, B, lengths)
    assert want == by_size(sipp, A, B, lengths)
    for o, v in opts.items():
        sipp.set_option(o, v)
    if 18 in opts:
        sch = schedule(lib, lengths)
        assert sch[0][4] == (sum(lengths) + opts[18] - 1) // opts[18] and sch[1][4] > 1
    assert sipp.sipp_prove_native_batch_ragged(A, B, lengths) == want


@pytest.mark.parametrize("conv", [1, 2, 3], ids=["ark-normalisation", "nested-order", "ark-nested"])
def test_conventions_against_oracle(sipp, oracle, conv):
    sipp.set_option(1, conv & 1)
    sipp.set_option(2, conv >> 1)
    lengths = [16, 1, 4, 8, 2, 4]
    A, B = oracle.seeded_inputs(101, sum(lengths), threads=THREADS)
    proofs = sipp.sipp_prove_native_batch_ragged(A, B, lengths)
    for j, (a, b) in enumerate(split(A, B, lengths)):
        assert b"".join(proofs[j]) == oracle.sipp_prove(a, b, opts=conv, threads=THREADS), (conv, j)


def test_identity_and_equal_points(sipp):
    lengths = [32, 4, 1, 8, 2]
    A, B = sipp.seeded_inputs(102, sum(lengths))
    A, B = bytearray(A), bytearray(B)
    A[64 * 3:64 * 4] = bytes(64)                         # identity in G1 (instance 0)
    B[128 * 33:128 * 34] = bytes(128)                    # identity in G2 (instance 1)
    A[64 * 36:64 * 37] = bytes(64)                       # instance 2: e(O, O)
    B[128 * 36:128 * 37] = bytes(128)
    A[64 * 40:64 * 41] = A[64 * 37:64 * 38]              # instance 3: equal points, so folds double
    B[128 * 40:128 * 41] = B[128 * 37:128 * 38]
    A[64 * 45:64 * 46] = A[64 * 44:64 * 45]              # instance 4: both pairs equal
    B[128 * 45:128 * 46] = B[128 * 44:128 * 45]
    A, B = bytes(A), bytes(B)
    proofs = sipp.sipp_prove_native_batch_ragged(A, B, lengths)
    for j, (a, b) in enumerate(split(A, B, lengths)):
        assert proofs[j] == sipp.sipp_prove_native(a, b), j


def test_bad_point_writes_nothing(sipp, lib):
    """one bad point in one instance fails the whole call in host and device form; the sentinel stays; a good call follows"""
    import torch
    from sipp_b200 import _lib
    lengths = [8, 2, 16, 1, 4]
    n, np_total = sum(lengths), sum(2 * (x.bit_length() - 1) + 1 for x in lengths)
    A, B = sipp.seeded_inputs(103, n)
    o = (ctypes.c_size_t * (len(lengths) + 1))(*offsets(lengths))
    for bad_A in (True, False):
        a, b = bytearray(A), bytearray(B)
        if bad_A:
            a[64 * 12 + 32] ^= 1                         # y of a point of instance 2: off the curve
        else:
            b[128 * 27:128 * 27 + 32] = P.to_bytes(32, "little")   # x.c0 == p in instance 3: not canonical
        out = ctypes.create_string_buffer(b"\xa5" * (384 * np_total), 384 * np_total)
        assert lib.sipp_prove_native_batch_ragged(bytes(a), n, bytes(b), n, o, len(lengths), out) == _lib.ERR_ENCODING
        assert out.raw == b"\xa5" * (384 * np_total)
        dA = torch.frombuffer(bytearray(a), dtype=torch.uint8).cuda()
        dB = torch.frombuffer(bytearray(b), dtype=torch.uint8).cuda()
        dO = torch.full((384 * np_total,), 0xa5, dtype=torch.uint8, device="cuda")
        torch.cuda.synchronize()
        rc = lib.sipp_prove_native_batch_ragged_device(dA.data_ptr(), dB.data_ptr(), n, o, len(lengths), dO.data_ptr())
        assert rc == _lib.ERR_ENCODING
        torch.cuda.synchronize()
        assert bool((dO == 0xa5).all())
    proofs = sipp.sipp_prove_native_batch_ragged(A, B, lengths)
    assert proofs == by_size(sipp, A, B, lengths)


def test_device_form_equals_host_form(sipp):
    import torch
    lengths = [64, 1, 8, 256, 2, 32, 4, 16]
    n, np_total = sum(lengths), sum(2 * (x.bit_length() - 1) + 1 for x in lengths)
    A, B = sipp.seeded_inputs(104, n)
    dA = torch.frombuffer(bytearray(A), dtype=torch.uint8).cuda()
    dB = torch.frombuffer(bytearray(B), dtype=torch.uint8).cuda()
    dO = torch.zeros(384 * np_total, dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()
    sipp.sipp_prove_native_batch_ragged_device(dA.data_ptr(), dB.data_ptr(), n, lengths, dO.data_ptr())
    torch.cuda.synchronize()
    assert dO.cpu().numpy().tobytes() == b"".join(b"".join(p) for p in sipp.sipp_prove_native_batch_ragged(A, B, lengths))


def test_stats(sipp):
    lengths = [64, 1, 8, 256, 2, 32, 4, 16, 1]
    A, B = sipp.seeded_inputs(105, sum(lengths))
    sipp.stats(reset=True)
    sipp.sipp_prove_native_batch_ragged(A, B, lengths)
    st = sipp.stats(reset=True)
    assert st["miller_pairs"] == sum(3 * n - 2 for n in lengths)
    assert st["fold_points"] == sum(n - 1 for n in lengths)


def test_proofs_verify_per_size(sipp):
    """the ragged proofs pass sipp_verify_native_batch run once per size; one tampered proof is rejected alone"""
    lengths = [16, 4, 16, 1, 64, 4, 16, 2]
    A, B = sipp.seeded_inputs(106, sum(lengths))
    proofs = sipp.sipp_prove_native_batch_ragged(A, B, lengths)
    proofs[2] = list(proofs[2])
    proofs[2][3] = proofs[0][3]                          # a Z_L / Z_R of another instance
    inst = split(A, B, lengths)
    for n in sorted(set(lengths)):
        js = [j for j in range(len(lengths)) if lengths[j] == n]
        sts = sipp.sipp_verify_native_batch(b"".join(inst[j][0] for j in js), b"".join(inst[j][1] for j in js), n, [proofs[j] for j in js])
        for j, st in zip(js, sts):
            assert isinstance(st, sipp.VerificationError) == (j == 2), (n, j)
