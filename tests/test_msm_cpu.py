"""Batched multi-scalar multiplications (sipp_g1_msm_batch, sipp_g2_msm_batch and their _device forms) without a GPU: every
argument error of the four entry points and its code, the host forms' encoding refusals before the device is touched, the loud
failure of a valid call without a device, the Python wrappers' ValueErrors, the per-segment plan at its thresholds, and the kernels'
recoding and bucket code (sipp_b200/csrc/msm.cuh, compiled for the host by tests/msmcheck) against the oracle."""
import ctypes
import os
import random
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
P = 0x30644E72E131A029B85045B68181585D97816A916871CA8D3C208C16D87CFD47
R = 0x30644E72E131A029B85045B68181585D2833E84879B9709143E1F593F0000001
LAMBDA_G1 = 0xb3c4d79d41a917585bfc41088d8daaa78b17ea66b99c90dd   # phi(x, y) = (beta x, y) acts as [LAMBDA_G1] on G1
LAMBDA_G2 = 0x6f4d8248eeb859fbf83e9682e87cfd46                   # psi acts as [6 x^2] on G2
FAKE = 0x7f0000001000          # a device address that is never read: every call below stops before the device is touched
STRAUS_BELOW = {1: 13, 2: 8}   # segments shorter than this take the Straus path (include/sipp_b200.h)


def le(v): return v.to_bytes(32, "little")


@pytest.fixture(scope="module")
def lib():
    from sipp_b200 import _lib
    return _lib.load()


def _szt(*o):
    return (ctypes.c_size_t * len(o))(*o)


ENTRIES = ("sipp_g1_msm_batch", "sipp_g2_msm_batch", "sipp_g1_msm_batch_device", "sipp_g2_msm_batch_device")


def call(lib, name, points=FAKE, scalars=FAKE, n=5, offs=(0, 2, 5), count=2, out=FAKE):
    host = not name.endswith("_device")
    size = 64 if name.startswith("sipp_g1") else 128
    if host:  # valid host buffers unless the test passes None: the encoding checks read them
        points = bytes(size * n) if points == FAKE else points
        scalars = bytes(32 * n) if scalars == FAKE else scalars
        out = ctypes.create_string_buffer(max(1, size * count)) if out == FAKE else out
    return getattr(lib, name)(points, scalars, n, None if offs is None else _szt(*offs), count, out)


@pytest.mark.parametrize("name", ENTRIES)
def test_argument_errors(lib, name):
    """the offsets rules of sipp_inner_product_batch, NULL pointers, more than 2^32 - 1 points: SIPP_ERR_ARG"""
    from sipp_b200 import _lib
    assert call(lib, name, points=None) == _lib.ERR_ARG
    assert call(lib, name, scalars=None) == _lib.ERR_ARG
    assert call(lib, name, out=None) == _lib.ERR_ARG
    assert call(lib, name, offs=None) == _lib.ERR_ARG
    assert call(lib, name, offs=(1, 2, 5)) == _lib.ERR_ARG                     # offsets[0] != 0
    assert call(lib, name, offs=(0, 4, 2, 5), count=3) == _lib.ERR_ARG         # decreasing
    assert call(lib, name, offs=(0, 2, 4)) == _lib.ERR_ARG                     # offsets[count] != n
    assert call(lib, name, n=3, offs=(0,), count=0) == _lib.ERR_ARG            # count == 0 with points
    if name.endswith("_device"):                                               # more than 2^32 - 1 points (never read)
        big = 1 << 32
        assert call(lib, name, n=big, offs=(0, big), count=1) == _lib.ERR_ARG
        assert "2^32" in lib.sipp_last_error().decode()
    # the order: the NULL pointers before the offsets
    assert call(lib, name, points=None, offs=(1, 2, 5)) == _lib.ERR_ARG
    assert "null" in lib.sipp_last_error().decode()


@pytest.mark.parametrize("group", (1, 2))
def test_host_encoding_refused_before_the_device(lib, group):
    """host forms: a scalar >= r, then a coordinate >= p, give SIPP_ERR_ENCODING without a device (valid arguments give SIPP_ERR_CUDA)"""
    from sipp_b200 import _lib
    name = ENTRIES[group - 1]
    size = 64 if group == 1 else 128
    good_k = le(1) * 5
    for k in (R, R + 1, 2**256 - 1):
        assert call(lib, name, scalars=le(3) * 4 + le(k)) == _lib.ERR_ENCODING
        assert "r" in lib.sipp_last_error().decode()
    pts = bytearray(size * 5)
    pts[size * 2:size * 2 + 32] = le(P)
    assert call(lib, name, points=bytes(pts), scalars=good_k) == _lib.ERR_ENCODING
    assert "p" in lib.sipp_last_error().decode()
    # the scalar check comes first
    assert call(lib, name, points=bytes(pts), scalars=le(R) * 5) == _lib.ERR_ENCODING
    assert "scalar" in lib.sipp_last_error().decode()


def test_no_gpu_fails_loudly(lib):
    """valid calls without a device return SIPP_ERR_CUDA, count == 0 included (as sipp_inner_product_batch)"""
    import sipp_b200
    from sipp_b200 import _lib
    if lib.sipp_device_count() > 0:
        pytest.skip("a GPU is present")
    for name in ENTRIES:
        assert call(lib, name) == _lib.ERR_CUDA
        assert call(lib, name, n=0, offs=(0,), count=0) == _lib.ERR_CUDA
        assert call(lib, name, n=5, offs=(0, 0, 5, 5), count=3) == _lib.ERR_CUDA   # empty segments are valid
    for fn in (sipp_b200.g1_msm_batch_device, sipp_b200.g2_msm_batch_device):
        with pytest.raises(sipp_b200.SippError) as ei:
            fn(FAKE, FAKE, 5, [2, 3], FAKE)
        assert ei.value.code == _lib.ERR_CUDA


def test_python_argument_errors():
    import sipp_b200
    for fn, size in ((sipp_b200.g1_msm_batch, 64), (sipp_b200.g2_msm_batch, 128)):
        with pytest.raises(ValueError):
            fn(bytes(size * 3), bytes(32 * 2), [3])            # points / scalars
        with pytest.raises(ValueError):
            fn(bytes(size * 3), bytes(32 * 3), [1, 1])         # lengths
        with pytest.raises(ValueError):
            fn(bytes(size * 3), bytes(32 * 3), [4, -1])        # negative length
        with pytest.raises(ValueError):
            fn(bytes(size * 3 + 1), bytes(32 * 3), [3])        # not whole points
    for fn in (sipp_b200.g1_msm_batch_device, sipp_b200.g2_msm_batch_device):
        with pytest.raises(ValueError):
            fn(FAKE, FAKE, 5, [2, 2], FAKE)


def _window_bits(group, length):
    """the cost model of msm.cu: the c in 5..16 minimising W (NC len + 3 2^(c-1)), W = bits // c + 1 (smallest c on ties)"""
    nc, bits = (2, 128) if group == 1 else (4, 66)
    costs = [((bits // c + 1) * (nc * length + 3 * 2 ** (c - 1)), c) for c in range(5, 17)]
    return min(costs)[1]


def test_plan_thresholds(lib):
    """Straus below STRAUS_BELOW points (and for empty segments), Pippenger from there on, with the window size of the cost model"""
    from sipp_b200 import _lib
    T1, T2 = STRAUS_BELOW[1], STRAUS_BELOW[2]
    lengths = [0, 1, 2, 3, T1 - 1, T1, T1 + 1, T2 - 1, T2, T2 + 1, 0, 64, 128, 1000, 4096, 1 << 12, 1 << 16, 1 << 20, 0]
    offs = [0]
    for length in lengths:
        offs.append(offs[-1] + length)
    out = (ctypes.c_int * (4 * len(lengths)))()
    assert lib.sipp_test_msm_plan(_szt(*offs), len(lengths), out, 4 * len(lengths)) == len(lengths)
    for j, length in enumerate(lengths):
        for g in (1, 2):
            path, c = out[4 * j + 2 * (g - 1)], out[4 * j + 2 * (g - 1) + 1]
            if length < STRAUS_BELOW[g]:
                assert (path, c) == (0, 0), (length, g)
            else:
                assert path == 1 and c == _window_bits(g, length), (length, g, c)
    # pinned points of the model: c grows with the length
    assert [_window_bits(2, n) for n in (32, 128, 1 << 12, 1 << 16, 1 << 20)] == [5, 7, 10, 14, 14]
    assert [_window_bits(1, n) for n in (32, 128, 1 << 12, 1 << 16, 1 << 20)] == [5, 6, 10, 13, 15]
    # the entry points' offsets checks
    assert lib.sipp_test_msm_plan(_szt(1, 2), 1, out, 4) == _lib.ERR_ARG
    assert lib.sipp_test_msm_plan(_szt(0, 2, 1), 2, out, 8) == _lib.ERR_ARG
    assert lib.sipp_test_msm_plan(None, 1, out, 4) == _lib.ERR_ARG
    assert lib.sipp_test_msm_plan(_szt(0), 0, out, 0) == 0


# ---- the kernels' recoding and bucket code on the host ---------------------------------------------------------------------------
@pytest.fixture(scope="module")
def mc(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("msmcheck") / "msmcheck.so")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-x", "c++", "-o", so,
                           os.path.join(ROOT, "tests", "msmcheck", "msmcheck.cpp")])
    return ctypes.CDLL(so)


def _recode(mc, group, k, c):
    nc = 2 if group == 1 else 4
    negs, mags, digits = (ctypes.c_int * nc)(), ctypes.create_string_buffer(24 * nc), (ctypes.c_int * (nc * 40))()
    w = mc.hc_msm_recode(group, le(k), c, negs, mags, digits)
    assert w > 0, (group, hex(k), w)
    subs = [(-1 if negs[j] else 1, int.from_bytes(mags.raw[24 * j:24 * j + 24], "little")) for j in range(nc)]
    return w, subs, [[digits[j * w + i] for i in range(w)] for j in range(nc)]


def _crafted_scalars():
    rng = random.Random(7)
    ks = [0, 1, 2, R - 1, R - 2, 2**127, 2**128, 2**128 - 1, 2**66, LAMBDA_G1, LAMBDA_G2, (R - 1) // 2, R // LAMBDA_G2, R - LAMBDA_G1,
          LAMBDA_G2**2 % R, LAMBDA_G2**3 % R]
    # lattice edges: scalars that round to the boundaries of Babai's cells, k = (m + 1/2) r / 2^s for both roundings
    for s in (64, 66, 127, 128, 130, 190, 250):
        ks += [(R << 1 >> s) % R, ((R >> s) + 1) % R, (R - (R >> s)) % R]
    return ks + [rng.randrange(R) for _ in range(300)]


@pytest.mark.parametrize("group", (1, 2))
def test_recoding_reconstructs_the_scalar(mc, group):
    """sum_j (-1)^neg_j m_j L^j == k (mod r), every m_j < 2^bits, and the signed c-bit digits reconstruct every m_j within their range"""
    lam, bits = (LAMBDA_G1, 128) if group == 1 else (LAMBDA_G2, 66)
    for k in _crafted_scalars():
        for c in (5, 8, 13, 16):
            w, subs, digits = _recode(mc, group, k, c)
            assert w == bits // c + 1
            assert sum(s * m * pow(lam, j, R) for j, (s, m) in enumerate(subs)) % R == k % R, hex(k)
            for (s, m), ds in zip(subs, digits):
                assert 0 <= m < 2**bits
                assert sum(d << (c * i) for i, d in enumerate(ds)) == m
                assert all(-(2 ** (c - 1)) < d <= 2 ** (c - 1) for d in ds)
    assert mc.hc_msm_recode(group, le(R), 8, (ctypes.c_int * 4)(), ctypes.create_string_buffer(96), (ctypes.c_int * 160)()) == -2


def _oracle_msm(oracle, m, group, pts, ks):
    size = 64 if group == 1 else 128
    mul, add, frm = (oracle.g1_mul, m.g1_add, m.g1_from_raw) if group == 1 else (oracle.g2_mul, m.g2_add, m.g2_from_raw)
    acc = None
    for i, k in enumerate(ks):
        acc = add(acc, frm(mul(pts[size * i:size * i + size], le(k))))
    return m.g1_raw(acc) if group == 1 else m.g2_raw(acc)


@pytest.mark.parametrize("group", (1, 2))
def test_host_msm_against_the_oracle(mc, oracle, group):
    """the Straus and Pippenger code of the kernels, run on the host, == sum of oracle scalar multiplications, incl. scalars 0, 1, r - 1,
    a repeated point (doubling inside a bucket), P and -P under the same scalar (identity), identity points"""
    sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
    import sipp_model as m
    size = 64 if group == 1 else 128
    rng = random.Random(11 + group)
    A, B = oracle.seeded_inputs(91, 8)
    pts_all = A if group == 1 else B
    pt = [pts_all[size * i:size * i + size] for i in range(8)]
    neg = (lambda b: m.g1_raw(m.g1_neg(m.g1_from_raw(b)))) if group == 1 else (lambda b: m.g2_raw(m.g2_neg(m.g2_from_raw(b))))
    cases = [
        ([pt[0]], [rng.randrange(R)]),
        ([pt[0], pt[1], pt[2]], [0, 1, R - 1]),
        ([pt[3]] * 4, [5, 5, 5, 5]),                                   # one bucket holds the same point 4 times
        ([pt[4], neg(pt[4])], [12345, 12345]),                          # sum is the identity
        ([bytes(size), pt[5], bytes(size)], [7, rng.randrange(R), R - 1]),
        (pt, [rng.randrange(R) for _ in range(8)]),
        (pt * 3, [rng.randrange(R) for _ in range(24)]),
    ]
    for pts, ks in cases:
        pb, kb = b"".join(pts), b"".join(le(k) for k in ks)
        want = _oracle_msm(oracle, m, group, pb, ks)
        for c, part in ((0, 0), (5, 16), (5, 3), (8, 64), (13, 1000)):
            out = ctypes.create_string_buffer(size)
            assert mc.hc_msm(group, pb, kb, len(ks), c, part, out) == 0
            assert out.raw == want, (group, len(ks), c, part)


def test_forced_path_hook_arguments(lib):
    """sipp_test_msm_batch_device: the device form's checks, then the group and the path (c = 0 or 5 .. 16), all before the device;
    a d_scalars or d_points that is only 4-byte aligned is a valid argument"""
    from sipp_b200 import _lib
    f = lib.sipp_test_msm_batch_device
    offs = _szt(0, 2, 5)
    assert f(2, 0, None, FAKE, 5, offs, 2, FAKE) == _lib.ERR_ARG
    assert f(1, 0, FAKE, FAKE, 5, _szt(1, 2, 5), 2, FAKE) == _lib.ERR_ARG
    for group, c in ((0, 0), (3, 0), (1, 4), (2, 17), (2, -1), (1, 1)):
        assert f(group, c, FAKE, FAKE, 5, offs, 2, FAKE) == _lib.ERR_ARG, (group, c)
    if lib.sipp_device_count() == 0:
        for group, c in ((1, 0), (2, 5), (2, 16)):
            assert f(group, c, FAKE, FAKE, 5, offs, 2, FAKE) == _lib.ERR_CUDA
        for name in ENTRIES[2:]:
            assert call(lib, name, points=FAKE + 4, scalars=FAKE + 4, out=FAKE + 8) == _lib.ERR_CUDA
