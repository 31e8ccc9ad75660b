"""Batched verification on device buffers: sipp_verify_native_batch_device and sipp_verify_native_batch_ragged_device.  Inputs are
torch CUDA uint8 tensors made by sipp_seeded_inputs_device and proved by the device provers.  Every result and every final must be
byte-identical to the host form's on the same bytes and options, in buffers pre-filled with a sentinel.  Also covered: tampering in
place in HBM, longer proofs, whole-call errors, NULL finals, the H1 / H2 conventions, the order after torch's default stream and the
stats.  A, B and the proofs must be unchanged after every call."""
import ctypes
import itertools
import random

import pytest

pytestmark = pytest.mark.gpu
P = 0x30644E72E131A029B85045B68181585D97816A916871CA8D3C208C16D87CFD47
SENT = 0x5a
RES_SENT = 0x5a5a5a5a

# every option of include/sipp_b200.h with its default
DEFAULTS = {1: 0, 2: 0, 3: 0, 4: 1, 5: 8192, 6: 1, 7: 256, 8: 1536, 9: 32, 10: 1, 11: 0, 12: 1, 13: 1, 14: 32, 15: 256, 16: 8, 17: 1, 18: 0}
MIXED = [1 << k for k in range(11)]   # 1, 2, 4, ..., 1024
# a twist point (on y^2 = x^3 + 3/xi) outside the order-r subgroup (tests/test_gpu_parity.py)
TWIST_NOT_G2 = bytes.fromhex("fbee9e35ab3c0ac619c62937bfe3caf537f37ffb5991752a801d56df83aea70a5de70f4aba744b50f26b23f62869ea32968c0a8a8e5449e0444c86ada8f60b28"
                             "b220740d239210aa74480d7e4ebe546a6b9f5fa2f8cf8c0a0a4580f18c2e612775f82b46ee8dc7599bf9c136ec784e777e061d68a3c8d110c06b2a0e0d572002")


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


@pytest.fixture(scope="module")
def torch(sipp):
    import torch
    return torch


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


def proof_len(n):
    return 2 * (n.bit_length() - 1) + 1


def offsets(lengths):
    o = [0]
    for length in lengths:
        o.append(o[-1] + length)
    return o


def host(t):
    return t.cpu().numpy().tobytes()


def seeded(torch, lib, seed, n):
    """device A, B (torch uint8) from sipp_seeded_inputs_device"""
    from sipp_b200 import _lib
    dA = torch.empty(64 * n, dtype=torch.uint8, device="cuda")
    dB = torch.empty(128 * n, dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()
    _lib.check(lib.sipp_seeded_inputs_device(seed, n, dA.data_ptr(), dB.data_ptr()))
    return dA, dB


def prove_batch(torch, lib, dA, dB, n, count):
    from sipp_b200 import _lib
    dP = torch.zeros(count * proof_len(n) * 384, dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()
    _lib.check(lib.sipp_prove_native_batch_device(dA.data_ptr(), dB.data_ptr(), n, count, dP.data_ptr()))
    return dP


def prove_ragged(torch, lib, dA, dB, lengths):
    from sipp_b200 import _lib
    dP = torch.zeros(sum(proof_len(x) for x in lengths) * 384, dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()
    o = offsets(lengths)
    _lib.check(lib.sipp_prove_native_batch_ragged_device(dA.data_ptr(), dB.data_ptr(), sum(lengths), (ctypes.c_size_t * len(o))(*o),
                                                         len(lengths), dP.data_ptr()))
    return dP


def outputs(torch, count, null=()):
    """sentinel-filled d_results and finals (None where NULL is passed)"""
    res = torch.full((count,), RES_SENT, dtype=torch.int32, device="cuda")
    fins = [None if k in null else torch.full((s * count,), SENT, dtype=torch.uint8, device="cuda") for k, s in enumerate((64, 128, 384))]
    return res, fins


def gather(rc, res, fins, count):
    """(return value, results, [(final_A, final_B, final_Z) per instance]), None for a NULL final"""
    fb = [None if f is None else host(f) for f in fins]
    return rc, res.cpu().tolist(), [tuple(None if f is None else f[s * j:s * (j + 1)] for f, s in zip(fb, (64, 128, 384))) for j in range(count)]


def unchanged(torch, *tensors):
    """snapshot of the inputs; calling the result asserts that none changed"""
    before = [t.clone() for t in tensors]
    return lambda: all(torch.equal(a, b) for a, b in zip(before, tensors))


def dev_batch(torch, lib, dA, dB, n, count, dP, plen, null=()):
    res, fins = outputs(torch, count, null)
    same = unchanged(torch, dA, dB, dP)
    rc = lib.sipp_verify_native_batch_device(dA.data_ptr(), dB.data_ptr(), n, count, dP.data_ptr(), plen, res.data_ptr(),
                                             *[None if f is None else f.data_ptr() for f in fins])
    assert same(), "an input changed"
    return gather(rc, res, fins, count)


def host_batch(lib, A, B, n, count, P_, plen):
    res = (ctypes.c_int * count)(*([RES_SENT] * count))
    fins = [ctypes.create_string_buffer(bytes([SENT]) * (s * count), s * count) for s in (64, 128, 384)]
    rc = lib.sipp_verify_native_batch(A, B, n, count, P_, plen, res, *fins)
    return rc, list(res), [tuple(f.raw[s * j:s * (j + 1)] for f, s in zip(fins, (64, 128, 384))) for j in range(count)]


def dev_ragged(torch, lib, dA, dB, lengths, dP, plens, null=()):
    count = len(lengths)
    res, fins = outputs(torch, count, null)
    o, po = offsets(lengths), offsets(plens)
    same = unchanged(torch, dA, dB, dP)
    rc = lib.sipp_verify_native_batch_ragged_device(dA.data_ptr(), dB.data_ptr(), sum(lengths), (ctypes.c_size_t * len(o))(*o), count, dP.data_ptr(),
                                                    (ctypes.c_size_t * len(po))(*po), res.data_ptr(),
                                                    *[None if f is None else f.data_ptr() for f in fins])
    assert same(), "an input changed"
    return gather(rc, res, fins, count)


def host_ragged(lib, A, B, lengths, P_, plens):
    count, n = len(lengths), sum(lengths)
    o, po = offsets(lengths), offsets(plens)
    res = (ctypes.c_int * count)(*([RES_SENT] * count))
    fins = [ctypes.create_string_buffer(bytes([SENT]) * (s * count), s * count) for s in (64, 128, 384)]
    rc = lib.sipp_verify_native_batch_ragged(A, n, B, n, (ctypes.c_size_t * len(o))(*o), count, P_, (ctypes.c_size_t * len(po))(*po), res, *fins)
    return rc, list(res), [tuple(f.raw[s * j:s * (j + 1)] for f, s in zip(fins, (64, 128, 384))) for j in range(count)]


def both_batch(torch, lib, dA, dB, n, count, dP, plen):
    """the device form == the host form on the downloaded bytes; returns the device form's outcome"""
    got = dev_batch(torch, lib, dA, dB, n, count, dP, plen)
    assert got == host_batch(lib, host(dA), host(dB), n, count, host(dP), plen)
    return got


def both_ragged(torch, lib, dA, dB, lengths, dP, plens):
    got = dev_ragged(torch, lib, dA, dB, lengths, dP, plens)
    assert got == host_ragged(lib, host(dA), host(dB), lengths, host(dP), plens)
    return got


def set_bytes(t, pos, value):
    t[pos:pos + len(value)] = t.new_tensor(list(value))


@pytest.mark.parametrize("n,count", [(16, 33), (128, 4096)])
def test_batch_equals_host_form(sipp, lib, torch, n, count):
    """device prover -> device verifier: all Ok, results and finals == the host form's and == the statement prover's finals; the
    stats grow as for the host form"""
    dA, dB = seeded(torch, lib, 400 + n, n * count)
    dP = prove_batch(torch, lib, dA, dB, n, count)
    plen = proof_len(n)
    sipp.stats(reset=True)
    got = dev_batch(torch, lib, dA, dB, n, count, dP, plen)
    st_dev = sipp.stats(reset=True)
    want = host_batch(lib, host(dA), host(dB), n, count, host(dP), plen)
    st_host = sipp.stats(reset=True)
    assert got[0] == 0 and got[1] == [0] * count
    assert got == want
    for k in ("fold_points", "miller_pairs"):
        assert st_dev[k] == st_host[k], k
    assert st_dev["fold_points"] == count * (n - 1)
    stmts = sipp.sipp_prove_native_batch_statement(host(dA), host(dB), n)
    assert b"".join(b"".join(p) for p, _ in stmts) == host(dP)
    assert [(s.final_A, s.final_B, s.final_Z) for _, s in stmts] == got[2]


@pytest.fixture(scope="module")
def pool(sipp, lib, torch):
    """the instances of MIXED and a duplicate of each (host bytes), proved in one ragged device call"""
    lengths = MIXED + MIXED
    dA, dB = seeded(torch, lib, 410, sum(lengths))
    dP = prove_ragged(torch, lib, dA, dB, lengths)
    A, B, Pb = host(dA), host(dB), host(dP)
    o, po = offsets(lengths), offsets([proof_len(x) for x in lengths])
    return [(A[64 * o[j]:64 * o[j + 1]], B[128 * o[j]:128 * o[j + 1]], Pb[384 * po[j]:384 * po[j + 1]]) for j in range(len(lengths))]


def to_dev(torch, b):
    return torch.frombuffer(bytearray(b), dtype=torch.uint8).cuda()


@pytest.mark.parametrize("order", ["ascending", "descending", "shuffled", "duplicates"])
def test_ragged_mixes_equal_host_form(sipp, lib, torch, pool, order):
    idx = list(range(len(MIXED)))
    if order == "descending":
        idx = idx[::-1]
    elif order == "shuffled":
        random.Random(411).shuffle(idx)
    elif order == "duplicates":
        idx = list(range(2 * len(MIXED)))
        random.Random(412).shuffle(idx)
        idx += idx[:5]
    lengths = [len(pool[i][0]) // 64 for i in idx]
    dA, dB, dP = (to_dev(torch, b"".join(pool[i][k] for i in idx)) for k in range(3))
    torch.cuda.synchronize()
    rc, res, _ = both_ragged(torch, lib, dA, dB, lengths, dP, [proof_len(x) for x in lengths])
    assert rc == 0 and res == [0] * len(idx)


def test_ragged_units_and_big_among_small(sipp, lib, torch):
    """n_j = 1 only (one Z swapped: Err), and one 2^10 instance among small ones; the stats grow as for the host form"""
    from sipp_b200 import _lib
    dA, dB = seeded(torch, lib, 413, 300)
    dP = prove_ragged(torch, lib, dA, dB, [1] * 300)
    dP[384 * 17:384 * 18] = dP[384 * 18:384 * 19].clone()
    rc, res, fins = both_ragged(torch, lib, dA, dB, [1] * 300, dP, [1] * 300)
    assert rc == 0 and res == [_lib.ERR_VERIFY if j == 17 else 0 for j in range(300)]
    A = host(dA)
    assert all(fins[j][0] == A[64 * j:64 * j + 64] for j in range(300))
    lengths = [8] * 40 + [1024] + [2] * 60 + [1] * 7 + [16] * 20
    random.Random(414).shuffle(lengths)
    dA, dB = seeded(torch, lib, 415, sum(lengths))
    dP = prove_ragged(torch, lib, dA, dB, lengths)
    plens = [proof_len(x) for x in lengths]
    sipp.stats(reset=True)
    got = dev_ragged(torch, lib, dA, dB, lengths, dP, plens)
    st_dev = sipp.stats(reset=True)
    want = host_ragged(lib, host(dA), host(dB), lengths, host(dP), plens)
    st_host = sipp.stats(reset=True)
    assert got == want and got[1] == [0] * len(lengths)
    for k in ("fold_points", "miller_pairs"):
        assert st_dev[k] == st_host[k], k
    assert st_dev["fold_points"] == sum(x - 1 for x in lengths) and st_dev["miller_pairs"] == len(lengths)


def test_batch_tampering_in_place(sipp, lib, torch):
    """in HBM: a flipped byte of a Z_L fails its instance alone (Err); a read coordinate == p or == 2^256 - 1 gives SIPP_ERR_ENCODING
    for its instance, whose finals still match the host form's; longer proofs with a non-canonical unread prefix verify like their
    suffix"""
    from sipp_b200 import _lib
    n, count = 16, 24
    np_ = proof_len(n)
    dA, dB = seeded(torch, lib, 420, n * count)
    dP = prove_batch(torch, lib, dA, dB, n, count)
    clean = both_batch(torch, lib, dA, dB, n, count, dP, np_)
    assert clean[1] == [0] * count
    t = dP.clone()
    t[384 * (3 * np_ + np_ - 2) + 5] ^= 1                                   # instance 3: round-1 Z_L
    set_bytes(t, 384 * (7 * np_ + 2) + 32 * 5, P.to_bytes(32, "little"))   # instance 7: a coordinate of the last-round Z_L == p
    set_bytes(t, 384 * (11 * np_ + np_ - 1), b"\xff" * 32)                 # instance 11: a coordinate of Z == 2^256 - 1
    torch.cuda.synchronize()
    rc, res, fins = both_batch(torch, lib, dA, dB, n, count, t, np_)
    assert rc == 0
    assert res == [_lib.ERR_VERIFY if j == 3 else _lib.ERR_ENCODING if j in (7, 11) else 0 for j in range(count)]
    assert all(fins[j] == clean[2][j] for j in range(count) if j not in (3, 7, 11))
    extra = 3
    junk = torch.full((count, 384 * extra), 0xff, dtype=torch.uint8, device="cuda")
    longer = torch.cat([junk, dP.view(count, -1)], dim=1).reshape(-1).contiguous()
    torch.cuda.synchronize()
    assert both_batch(torch, lib, dA, dB, n, count, longer, np_ + extra) == clean


def test_ragged_tampering_in_place(sipp, lib, torch):
    """the same for the ragged form, whose SIPP_ERR_ENCODING instances keep the sentinel in their final slots"""
    from sipp_b200 import _lib
    lengths = [16, 4, 64, 1, 8, 32, 2, 128, 1]
    plens = [proof_len(x) for x in lengths]
    po = offsets(plens)
    dA, dB = seeded(torch, lib, 421, sum(lengths))
    dP = prove_ragged(torch, lib, dA, dB, lengths)
    clean = both_ragged(torch, lib, dA, dB, lengths, dP, plens)
    assert clean[1] == [0] * len(lengths)
    t = dP.clone()
    t[384 * (po[2] + plens[2] - 2) + 100] ^= 0x10                          # instance 2: round-1 Z_L
    set_bytes(t, 384 * (po[5] + 3) + 32 * 11, P.to_bytes(32, "little"))   # instance 5: a coordinate == p
    set_bytes(t, 384 * po[8] + 32 * 4, b"\xff" * 32)                       # instance 8 (n = 1): a coordinate of Z == 2^256 - 1
    torch.cuda.synchronize()
    rc, res, fins = both_ragged(torch, lib, dA, dB, lengths, t, plens)
    assert rc == 0
    assert res == [_lib.ERR_VERIFY if j == 2 else _lib.ERR_ENCODING if j in (5, 8) else 0 for j in range(len(lengths))]
    untouched = (bytes([SENT]) * 64, bytes([SENT]) * 128, bytes([SENT]) * 384)
    assert fins[5] == untouched and fins[8] == untouched
    assert all(fins[j] == clean[2][j] for j in range(len(lengths)) if j not in (2, 5, 8))
    # longer proofs: j % 3 leading non-canonical elements that are never read
    parts = []
    for j in range(len(lengths)):
        parts.append(torch.full((384 * (j % 3),), 0xff, dtype=torch.uint8, device="cuda"))
        parts.append(dP[384 * po[j]:384 * po[j + 1]])
    longer = torch.cat(parts).contiguous()
    torch.cuda.synchronize()
    assert both_ragged(torch, lib, dA, dB, lengths, longer, [p + j % 3 for j, p in enumerate(plens)]) == clean


@pytest.mark.parametrize("what", ["coordinate_p", "g2_not_in_subgroup"])
def test_whole_call_errors_write_nothing(sipp, lib, torch, what):
    """a coordinate >= p in dA, or (SIPP_OPT_VALIDATE_POINTS on) a G2 point outside the subgroup in dB, fails the whole call with
    SIPP_ERR_ENCODING for both forms; d_results and the finals keep their sentinels, the inputs are unchanged"""
    from sipp_b200 import _lib
    sipp.set_option(_lib.OPT_VALIDATE_POINTS, 1)
    n, count = 8, 6
    dA, dB = seeded(torch, lib, 430, n * count)
    dP = prove_batch(torch, lib, dA, dB, n, count)
    if what == "coordinate_p":
        set_bytes(dA, 64 * 13, P.to_bytes(32, "little"))                    # x of A_13 (instance 1)
    else:
        set_bytes(dB, 128 * 29, TWIST_NOT_G2)                               # B_29 (instance 3)
    torch.cuda.synchronize()
    sent = (bytes([SENT]) * 64, bytes([SENT]) * 128, bytes([SENT]) * 384)
    assert dev_batch(torch, lib, dA, dB, n, count, dP, proof_len(n)) == (_lib.ERR_ENCODING, [RES_SENT] * count, [sent] * count)
    lengths = [8, 16, 4, 2, 1, 1, 16]
    assert dev_ragged(torch, lib, dA, dB, lengths, dP, [proof_len(x) for x in lengths]) \
        == (_lib.ERR_ENCODING, [RES_SENT] * len(lengths), [sent] * len(lengths))
    # the same call with the point restored runs
    dA2, dB2 = seeded(torch, lib, 430, n * count)
    assert dev_batch(torch, lib, dA2, dB2, n, count, dP, proof_len(n))[1] == [0] * count


def test_null_finals(sipp, lib, torch):
    """any subset of NULL finals gives the same results, and the other finals are unchanged"""
    from sipp_b200 import _lib
    n, count = 8, 10
    dA, dB = seeded(torch, lib, 440, n * count)
    dP = prove_batch(torch, lib, dA, dB, n, count)
    np_ = proof_len(n)
    dP[384 * (2 * np_ + 1) + 7] ^= 1                                       # instance 2: Err
    set_bytes(dP, 384 * (5 * np_), b"\xff" * 32)                           # instance 5: SIPP_ERR_ENCODING
    lengths = [8, 2, 32, 1, 4, 1, 16, 8]
    plens = [proof_len(x) for x in lengths]
    po = offsets(plens)
    rA, rB = seeded(torch, lib, 441, sum(lengths))
    rP = prove_ragged(torch, lib, rA, rB, lengths)
    rP[384 * po[1] + 40] ^= 1                                              # instance 1: Err
    set_bytes(rP, 384 * (po[6] + 2), P.to_bytes(32, "little"))             # instance 6: SIPP_ERR_ENCODING
    torch.cuda.synchronize()
    full_b = both_batch(torch, lib, dA, dB, n, count, dP, np_)
    full_r = both_ragged(torch, lib, rA, rB, lengths, rP, plens)
    assert full_b[1] == [_lib.ERR_VERIFY if j == 2 else _lib.ERR_ENCODING if j == 5 else 0 for j in range(count)]
    assert full_r[1] == [_lib.ERR_VERIFY if j == 1 else _lib.ERR_ENCODING if j == 6 else 0 for j in range(len(lengths))]
    for k in range(1, 4):
        for null in itertools.combinations(range(3), k):
            for got, full in ((dev_batch(torch, lib, dA, dB, n, count, dP, np_, null), full_b),
                              (dev_ragged(torch, lib, rA, rB, lengths, rP, plens, null), full_r)):
                assert got[:2] == full[:2], null
                assert got[2] == [tuple(None if i in null else f[i] for i in range(3)) for f in full[2]], null


def test_conventions(sipp, lib, torch):
    """SIPP_OPT_FE_NORMALISATION = 1 and SIPP_OPT_FQ12_ORDER = 1: the same bytes as the host form under the same options"""
    from sipp_b200 import _lib
    sipp.set_option(_lib.OPT_FE_NORMALISATION, 1)
    sipp.set_option(_lib.OPT_FQ12_ORDER, 1)
    n, count = 16, 12
    dA, dB = seeded(torch, lib, 450, n * count)
    dP = prove_batch(torch, lib, dA, dB, n, count)
    dP[384 * (4 * proof_len(n)) + 3] ^= 2                                  # one Err
    torch.cuda.synchronize()
    rc, res, _ = both_batch(torch, lib, dA, dB, n, count, dP, proof_len(n))
    assert rc == 0 and res == [_lib.ERR_VERIFY if j == 4 else 0 for j in range(count)]
    lengths = [4, 32, 1, 8, 2, 16]
    rA, rB = seeded(torch, lib, 451, sum(lengths))
    rP = prove_ragged(torch, lib, rA, rB, lengths)
    rc, res, _ = both_ragged(torch, lib, rA, rB, lengths, rP, [proof_len(x) for x in lengths])
    assert rc == 0 and res == [0] * len(lengths)


def test_stream_order_after_torch(sipp, lib, torch):
    """a tamper enqueued by torch on its default stream behind a long kernel, then the device verifier called right away without a
    synchronisation: the verifier sees the tampered proof"""
    from sipp_b200 import _lib
    assert torch.cuda.current_stream().cuda_stream == 0                    # the legacy default stream
    n, count = 16, 8
    np_ = proof_len(n)
    dA, dB = seeded(torch, lib, 460, n * count)
    dP = prove_batch(torch, lib, dA, dB, n, count)
    torch.cuda.synchronize()
    torch.cuda._sleep(200_000_000)                                         # ~0.1 s on torch's stream
    dP[384 * (6 * np_ + np_ - 1) + 9] ^= 4                                 # instance 6: Z
    res, fins = outputs(torch, count)
    _lib.check(lib.sipp_verify_native_batch_device(dA.data_ptr(), dB.data_ptr(), n, count, dP.data_ptr(), np_, res.data_ptr(),
                                                   *[f.data_ptr() for f in fins]))
    assert res.cpu().tolist() == [_lib.ERR_VERIFY if j == 6 else 0 for j in range(count)]
    lengths = [16, 2, 8, 1, 4]
    plens = [proof_len(x) for x in lengths]
    rA, rB = seeded(torch, lib, 461, sum(lengths))
    rP = prove_ragged(torch, lib, rA, rB, lengths)
    torch.cuda.synchronize()
    torch.cuda._sleep(200_000_000)
    rP[384 * offsets(plens)[2] + 9] ^= 4                                   # instance 2: last-round Z_R
    res, fins = outputs(torch, len(lengths))
    sipp.sipp_verify_native_batch_ragged_device(rA.data_ptr(), rB.data_ptr(), sum(lengths), lengths, rP.data_ptr(), plens, res.data_ptr(),
                                               *[f.data_ptr() for f in fins])
    assert res.cpu().tolist() == [_lib.ERR_VERIFY if j == 2 else 0 for j in range(len(lengths))]


def test_python_wrappers(sipp, lib, torch):
    """the wrappers give the C calls' bytes; a whole-call error raises SippError"""
    from sipp_b200 import _lib
    n, count = 8, 5
    dA, dB = seeded(torch, lib, 470, n * count)
    dP = prove_batch(torch, lib, dA, dB, n, count)
    want = dev_batch(torch, lib, dA, dB, n, count, dP, proof_len(n))
    res, fins = outputs(torch, count, null=(1,))
    sipp.sipp_verify_native_batch_device(dA.data_ptr(), dB.data_ptr(), n, count, dP.data_ptr(), proof_len(n), res.data_ptr(),
                                         d_final_A=fins[0].data_ptr(), d_final_Z=fins[2].data_ptr())
    assert gather(0, res, fins, count) == (0, want[1], [(f[0], None, f[2]) for f in want[2]])
    lengths = [4, 1, 2, 1, 32]
    plens = [proof_len(x) for x in lengths]
    rA, rB = seeded(torch, lib, 471, sum(lengths))
    rP = prove_ragged(torch, lib, rA, rB, lengths)
    want = dev_ragged(torch, lib, rA, rB, lengths, rP, plens)
    res, fins = outputs(torch, len(lengths))
    sipp.sipp_verify_native_batch_ragged_device(rA.data_ptr(), rB.data_ptr(), sum(lengths), lengths, rP.data_ptr(), plens, res.data_ptr(),
                                               *[f.data_ptr() for f in fins])
    assert gather(0, res, fins, len(lengths)) == want
    with pytest.raises(sipp.SippError) as ei:
        sipp.sipp_verify_native_batch_ragged_device(rA.data_ptr(), rB.data_ptr(), sum(lengths), lengths, rP.data_ptr(),
                                                   [p - 1 for p in plens], res.data_ptr())
    assert ei.value.code == _lib.ERR_SHORT_PROOF
