"""Ragged batched verification (sipp_verify_native_batch_ragged): independent verifications of instances of different sizes in one
call, against sipp_verify_native on every instance (its return value and, for Ok and Err, its final_A, final_B, final_Z byte for
byte), the uniform batched verifier, the CPU oracle under all four H1 / H2 conventions and the golden proofs.  The schedule hook
(sipp_test_ragged_schedule) asserts which fold kernel every shape reaches."""
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


def flat(proof):
    return proof if isinstance(proof, (bytes, bytearray)) else b"".join(proof)


def ragged(lib, A, B, lengths, proofs, sentinel=0):
    """the C call: (return value, results, [(final_A, final_B, final_Z) per instance]); sentinel-filled outputs beforehand"""
    count = len(lengths)
    n = sum(lengths)
    ps = [flat(p) for p in proofs]
    po = offsets([len(p) // 384 for p in ps])
    res = (ctypes.c_int * count)(*([sentinel] * count))
    fa, fb, fz = (ctypes.create_string_buffer(b"\xa5" * (k * count), k * count) for k in (64, 128, 384))
    rc = lib.sipp_verify_native_batch_ragged(A, n, B, n, (ctypes.c_size_t * (count + 1))(*offsets(lengths)), count, b"".join(ps),
                                             (ctypes.c_size_t * (count + 1))(*po), res, fa, fb, fz)
    fins = [(fa.raw[64 * j:64 * j + 64], fb.raw[128 * j:128 * j + 128], fz.raw[384 * j:384 * j + 384]) for j in range(count)]
    return rc, list(res), fins


def native(lib, a, b, proof):
    """sipp_verify_native: (return value, (final_A, final_B, final_Z))"""
    p = flat(proof)
    fa, fb, fz = (ctypes.create_string_buffer(k) for k in (64, 128, 384))
    rc = lib.sipp_verify_native(a, len(a) // 64, b, len(b) // 128, p, len(p) // 384, fa, fb, fz)
    return rc, (fa.raw, fb.raw, fz.raw)


def check_against_native(lib, A, B, lengths, proofs, want_codes=None):
    """the contract: results[j] == sipp_verify_native on instance j, finals byte-equal for Ok and Err"""
    from sipp_b200 import _lib
    rc, res, fins = ragged(lib, A, B, lengths, proofs)
    assert rc == _lib.OK
    for j, (a, b) in enumerate(split(A, B, lengths)):
        nrc, nfin = native(lib, a, b, proofs[j])
        assert res[j] == nrc, (j, lengths[j])
        if want_codes is not None:
            assert res[j] == want_codes[j], (j, lengths[j])
        if nrc in (_lib.OK, _lib.ERR_VERIFY):
            assert fins[j] == nfin, (j, lengths[j])
        else:
            assert fins[j] == (b"\xa5" * 64, b"\xa5" * 128, b"\xa5" * 384), j
    return res, fins


@pytest.fixture(scope="module")
def pool(sipp, lib):
    """the instances of MIXED and a duplicate of each, proved in one ragged call, with sipp_verify_native's finals"""
    lengths = MIXED + MIXED
    A, B = sipp.seeded_inputs(190, sum(lengths))
    proofs = sipp.sipp_prove_native_batch_ragged(A, B, lengths)
    out = []
    for (a, b), p in zip(split(A, B, lengths), proofs):
        rc, fin = native(lib, a, b, p)
        assert rc == 0
        out.append((a, b, p, fin))
    return out


@pytest.mark.parametrize("order", ["ascending", "descending", "shuffled", "duplicates"])
def test_mixed_sizes_match_single_verifications(sipp, lib, pool, order):
    idx = list(range(len(MIXED)))
    if order == "descending":
        idx = idx[::-1]
    elif order == "shuffled":
        random.Random(191).shuffle(idx)
    elif order == "duplicates":
        idx = list(range(2 * len(MIXED)))
        random.Random(192).shuffle(idx)
        idx += idx[:5]
    A = b"".join(pool[i][0] for i in idx)
    B = b"".join(pool[i][1] for i in idx)
    lengths = [len(pool[i][0]) // 64 for i in idx]
    rc, res, fins = ragged(lib, A, B, lengths, [pool[i][2] for i in idx])
    assert rc == 0 and res == [0] * len(idx)
    for j, i in enumerate(idx):
        assert fins[j] == pool[i][3], (order, j, lengths[j])
    sts = sipp.sipp_verify_native_batch_ragged(A, B, lengths, [pool[i][2] for i in idx])
    for j, i in enumerate(idx):
        st = sts[j]
        assert isinstance(st, sipp.SIPPStatement)
        assert (st.final_A, st.final_B, st.final_Z) == pool[i][3] and st.Z == pool[i][2][-1]
        assert b"".join(st.A) == pool[i][0] and b"".join(st.B) == pool[i][1]


@pytest.mark.parametrize("n,count", [(16, 33), (128, 4096)])
def test_equal_sizes_match_uniform_batch(sipp, n, count):
    A, B = sipp.seeded_inputs(193 + n, n * count)
    proofs = sipp.sipp_prove_native_batch(A, B, n)
    proofs[count // 2] = list(proofs[count // 2])
    proofs[count // 2][1] = proofs[0][1]                 # one Err among them
    want = sipp.sipp_verify_native_batch(A, B, n, proofs)
    got = sipp.sipp_verify_native_batch_ragged(A, B, [n] * count, proofs)
    for j, (w, g) in enumerate(zip(want, got)):
        assert type(w) is type(g), j
        if isinstance(w, sipp.SIPPStatement):
            assert (g.final_A, g.final_B, g.final_Z, g.Z) == (w.final_A, w.final_B, w.final_Z, w.Z), j
    assert isinstance(got[count // 2], sipp.VerificationError)
    assert sum(isinstance(g, sipp.VerificationError) for g in got) == 1


def test_tampering_fails_alone(sipp, lib):
    """a changed Z, round-1 Z_L, last-round Z_R or A point fails its instance only; every other instance keeps its result and finals"""
    from sipp_b200 import _lib
    lengths = [16, 4, 64, 1, 8, 32, 2, 128, 1]
    A, B = sipp.seeded_inputs(194, sum(lengths))
    proofs = sipp.sipp_prove_native_batch_ragged(A, B, lengths)
    rc, res, clean = ragged(lib, A, B, lengths, proofs)
    assert rc == 0 and res == [0] * len(lengths)
    t = [list(p) for p in proofs]
    t[2][-1] = proofs[0][-1]                             # instance 2: Z of another instance
    t[5][-2] = proofs[7][-2]                             # instance 5: round-1 Z_L (slot np - 2)
    t[7][0] = proofs[5][0]                               # instance 7: last-round Z_R (slot 0)
    t[8][0] = proofs[3][0]                               # instance 8 (n = 1): another Z
    o = offsets(lengths)
    a = bytearray(A)
    a[64 * o[1] + 64:64 * o[1] + 128] = A[64 * o[4]:64 * o[4] + 64]   # instance 1: an A point swapped for another valid point
    a = bytes(a)
    bad = {1, 2, 5, 7, 8}
    res, fins = check_against_native(lib, a, B, lengths, t, [_lib.ERR_VERIFY if j in bad else _lib.OK for j in range(len(lengths))])
    for j in range(len(lengths)):
        if j not in bad:
            assert fins[j] == clean[j], j
    sts = sipp.sipp_verify_native_batch_ragged(a, B, lengths, t)
    assert [isinstance(s, sipp.VerificationError) for s in sts] == [j in bad for j in range(len(lengths))]


def test_non_canonical_proof_element(sipp, lib):
    """a coordinate >= p among the elements read gives SIPP_ERR_ENCODING for that instance alone; the wrapper returns a SippError"""
    from sipp_b200 import _lib
    lengths = [8, 2, 32, 1, 4]
    A, B = sipp.seeded_inputs(195, sum(lengths))
    proofs = [list(p) for p in sipp.sipp_prove_native_batch_ragged(A, B, lengths)]
    _, _, clean = ragged(lib, A, B, lengths, proofs)
    z = bytearray(proofs[2][3])
    z[32 * 7:32 * 8] = P.to_bytes(32, "little")          # one Fq coordinate == p
    proofs[2][3] = bytes(z)
    z = bytearray(proofs[3][0])
    z[0:32] = (P + 5).to_bytes(32, "little")             # n = 1: Z itself
    proofs[3][0] = bytes(z)
    want = [_lib.OK, _lib.OK, _lib.ERR_ENCODING, _lib.ERR_ENCODING, _lib.OK]
    res, fins = check_against_native(lib, A, B, lengths, proofs, want)
    for j in (0, 1, 4):
        assert fins[j] == clean[j]
    sts = sipp.sipp_verify_native_batch_ragged(A, B, lengths, proofs)
    for j in (2, 3):
        assert isinstance(sts[j], sipp.SippError) and sts[j].code == _lib.ERR_ENCODING
        assert not isinstance(sts[j], sipp.SIPPStatement)
    assert all(isinstance(sts[j], sipp.SIPPStatement) for j in (0, 1, 4))


def test_longer_proofs_verify_like_their_suffix(sipp, lib):
    """extra leading elements are never read, not even for the canonicality check"""
    lengths = [4, 16, 1, 2, 64]
    A, B = sipp.seeded_inputs(196, sum(lengths))
    proofs = sipp.sipp_prove_native_batch_ragged(A, B, lengths)
    _, _, clean = ragged(lib, A, B, lengths, proofs)
    junk = b"\xff" * 384                                 # not canonical
    longer = [[junk] * (j % 3) + [proofs[(j + 1) % 5][0]] * (j % 2) + list(p) for j, p in enumerate(proofs)]
    res, fins = check_against_native(lib, A, B, lengths, longer, [0] * len(lengths))
    assert fins == clean
    longer[1][-2], longer[1][-3] = longer[1][-3], longer[1][-2]   # the suffix itself changed (round-1 Z_L and Z_R swapped): Err
    res, _ = check_against_native(lib, A, B, lengths, longer)
    assert res == [0, -7, 0, 0, 0]


def test_whole_call_errors_write_nothing(sipp, lib):
    """a short proof and a bad input point fail the whole call; results and finals keep their sentinels; a good call follows"""
    from sipp_b200 import _lib
    lengths = [8, 2, 16, 1, 4]
    A, B = sipp.seeded_inputs(197, sum(lengths))
    proofs = sipp.sipp_prove_native_batch_ragged(A, B, lengths)
    untouched = [(b"\xa5" * 64, b"\xa5" * 128, b"\xa5" * 384)] * len(lengths)
    short = list(proofs)
    short[2] = proofs[2][1:]
    rc, res, fins = ragged(lib, A, B, lengths, short, sentinel=77)
    assert rc == _lib.ERR_SHORT_PROOF and res == [77] * len(lengths) and fins == untouched
    for bad_A in (True, False):
        a, b = bytearray(A), bytearray(B)
        if bad_A:
            a[64 * 12 + 32] ^= 1                         # y of a point of instance 2: off the curve
        else:
            b[128 * 27:128 * 27 + 32] = P.to_bytes(32, "little")   # x.c0 == p in instance 3
        rc, res, fins = ragged(lib, bytes(a), bytes(b), lengths, proofs, sentinel=77)
        assert rc == _lib.ERR_ENCODING and res == [77] * len(lengths) and fins == untouched
    with pytest.raises(sipp.SippError):
        sipp.sipp_verify_native_batch_ragged(A, B, lengths, short)
    check_against_native(lib, A, B, lengths, proofs, [0] * len(lengths))


@pytest.mark.parametrize("conv", [0, 1, 2, 3], ids=["default", "ark-normalisation", "nested-order", "ark-nested"])
def test_conventions_against_oracle(sipp, lib, oracle, conv):
    """oracle proofs made under one H1 / H2 convention verify under that convention's options only (n >= 4; n <= 2 under its
    normalisation), as pyoracle.sipp_verify says"""
    lengths = [16, 1, 4, 8, 2, 4]
    A, B = oracle.seeded_inputs(198 + conv, sum(lengths), threads=THREADS)
    inst = split(A, B, lengths)
    proofs = [oracle.sipp_prove(a, b, opts=conv, threads=THREADS) for a, b in inst]
    for opts in range(4):
        sipp.set_option(1, opts & 1)
        sipp.set_option(2, opts >> 1)
        rc, res, fins = ragged(lib, A, B, lengths, proofs)
        assert rc == 0
        for j, (a, b) in enumerate(inst):
            ok, fin = oracle.sipp_verify(a, b, proofs[j], opts=opts, threads=THREADS)
            assert (res[j] == 0) == ok, (conv, opts, j)
            assert fins[j] == (fin["final_A"], fin["final_B"], fin["final_Z"]), (conv, opts, j)
            # with one round (n <= 2) Z_L and Z_R are products of the unfolded inputs, so an honest proof holds for any challenge
            # and only the normalisation must match; from n = 4 the transcript order must match too
            assert ok == ((opts == conv) if lengths[j] >= 4 else (opts & 1) == (conv & 1)), (conv, opts, j)
        check_against_native(lib, A, B, lengths, proofs)


def test_golden_proofs(sipp, lib, golden):
    H = bytes.fromhex
    cases = golden["prove"]
    A = b"".join(H(c["A"]) for c in cases)
    B = b"".join(H(c["B"]) for c in cases)
    proofs = [H(c["proof"]) for c in cases]
    rc, res, fins = ragged(lib, A, B, [c["n"] for c in cases], proofs)
    assert rc == 0 and res == [0] * len(cases)
    for c, f in zip(cases, fins):
        assert f == (H(c["final_A"]), H(c["final_B"]), H(c["final_Z"])), c["name"]


# (name, options, lengths, the fold kernels the rounds must reach) -- the shapes of the ragged prover's tests
FOLD_CASES = [
    ("default", {}, [256] * 64 + [128] * 130 + [4, 2, 1], {0, 1, 2}),
    ("no_straus", {10: 0}, [256] * 64 + [128] * 130 + [4, 2, 1], {0, 1}),
    ("wide_fold_max_0", {7: 0}, [64] * 30 + [8] * 5 + [2] * 3, {0, 1}),
    ("wide_fold_max_large", {7: 1 << 20, 10: 0}, [256] * 40 + [16] * 9 + [2] * 7 + [1], {1}),
    ("lane_split_mixed_warp", {7: 0}, [1024, 4] + [2] * 40, {0, 1}),
    ("wide_mixed_h1", {}, [128, 2, 64, 2, 2, 32, 2], {1}),
]


@pytest.mark.parametrize("name,opts,lengths,want", FOLD_CASES, ids=[c[0] for c in FOLD_CASES])
def test_fold_kernels(sipp, lib, name, opts, lengths, want):
    """every ragged fold kernel, checked against the uniform batched verifier once per size"""
    rng = random.Random(hash(name) & 0xffff)
    order = list(range(len(lengths)))
    rng.shuffle(order)
    lengths = [lengths[i] for i in order]
    A, B = sipp.seeded_inputs(199, sum(lengths))
    proofs = sipp.sipp_prove_native_batch_ragged(A, B, lengths)
    for o, v in opts.items():
        sipp.set_option(o, v)
    assert {r[3] for r in schedule(lib, lengths)[1:]} == want
    proofs[len(proofs) // 2] = list(proofs[len(proofs) // 2])
    proofs[len(proofs) // 2][-1] = proofs[0][-1] if len(proofs) // 2 else proofs[1][-1]   # one Err
    got = sipp.sipp_verify_native_batch_ragged(A, B, lengths, proofs)
    inst = split(A, B, lengths)
    for n in sorted(set(lengths)):
        js = [j for j in range(len(lengths)) if lengths[j] == n]
        want_sts = sipp.sipp_verify_native_batch(b"".join(inst[j][0] for j in js), b"".join(inst[j][1] for j in js), n, [proofs[j] for j in js])
        for j, w in zip(js, want_sts):
            assert type(got[j]) is type(w), (name, j)
            if isinstance(w, sipp.SIPPStatement):
                assert (got[j].final_A, got[j].final_B, got[j].final_Z) == (w.final_A, w.final_B, w.final_Z), (name, j)
    assert sum(isinstance(g, sipp.VerificationError) for g in got) == 1


@pytest.mark.parametrize("opts", [{18: 1}, {6: 0}, {5: 0}], ids=["chunk_pairs_1", "fe_engine_0", "wide_lines_0"])
def test_final_pairing_options(sipp, lib, opts):
    """the options of the final pairings change no bit"""
    lengths = [64, 1, 8, 256, 2, 32, 4, 16, 128, 2, 1]
    A, B = sipp.seeded_inputs(200, sum(lengths))
    proofs = [list(p) for p in sipp.sipp_prove_native_batch_ragged(A, B, lengths)]
    proofs[4][-1] = proofs[1][-1]
    want = ragged(lib, A, B, lengths, proofs)
    assert want[0] == 0 and want[1] == [0, 0, 0, 0, -7, 0, 0, 0, 0, 0, 0]
    for o, v in opts.items():
        sipp.set_option(o, v)
    assert ragged(lib, A, B, lengths, proofs) == want
    check_against_native(lib, A, B, lengths, proofs)


def test_unit_single_and_big_among_small(sipp, lib):
    """n = 1 only: Ok exactly when pairing(A_i, B_i) == Z; one 2^12 instance alone and among 255 instances of n = 16"""
    from sipp_b200 import _lib
    A, B = sipp.seeded_inputs(201, 300)
    zs = sipp.pairing_batch(A, B)
    proofs = [[z] for z in zs]
    proofs[17] = [zs[18]]
    rc, res, fins = ragged(lib, A, B, [1] * 300, proofs)
    assert rc == 0 and res == [_lib.ERR_VERIFY if j == 17 else 0 for j in range(300)]
    for j in range(300):
        assert fins[j] == (A[64 * j:64 * j + 64], B[128 * j:128 * j + 128], proofs[j][0])
    A, B = sipp.seeded_inputs(202, 4096)
    big = sipp.sipp_prove_native(A, B)
    nrc, nfin = native(lib, A, B, big)
    assert nrc == 0
    rc, res, fins = ragged(lib, A, B, [4096], [big])
    assert (rc, res, fins) == (0, [0], [nfin])
    A2, B2 = sipp.seeded_inputs(203, 16 * 255)
    lengths = [16] * 100 + [4096] + [16] * 155
    A3 = A2[:64 * 1600] + A + A2[64 * 1600:]
    B3 = B2[:128 * 1600] + B + B2[128 * 1600:]
    small = sipp.sipp_prove_native_batch(A2, B2, 16)
    rc, res, fins = ragged(lib, A3, B3, lengths, small[:100] + [big] + small[100:])
    assert rc == 0 and res == [0] * 256
    assert fins[100] == nfin
    want = sipp.sipp_verify_native_batch(A2, B2, 16, small)
    assert [f for j, f in enumerate(fins) if j != 100] == [(w.final_A, w.final_B, w.final_Z) for w in want]


def test_stats(sipp, lib):
    lengths = [64, 1, 8, 256, 2, 32, 4, 16, 1]
    A, B = sipp.seeded_inputs(204, sum(lengths))
    proofs = sipp.sipp_prove_native_batch_ragged(A, B, lengths)
    sipp.stats(reset=True)
    rc, res, _ = ragged(lib, A, B, lengths, proofs)
    st = sipp.stats(reset=True)
    assert rc == 0 and res == [0] * len(lengths)
    assert st["fold_points"] == sum(n - 1 for n in lengths)
    assert st["miller_pairs"] == len(lengths)
