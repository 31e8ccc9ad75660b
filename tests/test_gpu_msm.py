"""Batched multi-scalar multiplications on the GPU (sipp_g1_msm_batch, sipp_g2_msm_batch and their _device forms): small segments of
every path against the oracle, large ones against a closed form, segments of one point against the scalar-multiplication producers,
host form against device form, the tie to the protocol (final_A and final_B of a proof are MSMs of its inputs), and the refusals."""
import ctypes
import os
import random
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
import sipp_model as m  # noqa: E402

pytestmark = pytest.mark.gpu
P, R = m.P, m.R
T1, T2 = 13, 8  # the Straus / Pippenger thresholds of G1 and G2


def le(v): return v.to_bytes(32, "little")


@pytest.fixture(scope="module")
def sb():
    import sipp_b200
    from sipp_b200 import _lib
    _lib.require_gpu_once()
    return sipp_b200


@pytest.fixture(scope="module")
def torch():
    import torch
    return torch


def _size(group): return 64 if group == 1 else 128
def _msm(sb, group): return sb.g1_msm_batch if group == 1 else sb.g2_msm_batch


def _oracle_sum(oracle, group, pts, ks):
    size = _size(group)
    mul, add, frm, raw = (oracle.g1_mul, m.g1_add, m.g1_from_raw, m.g1_raw) if group == 1 else (oracle.g2_mul, m.g2_add, m.g2_from_raw, m.g2_raw)
    acc = None
    for i, k in enumerate(ks):
        acc = add(acc, frm(mul(pts[size * i:size * i + size], le(k))))
    return raw(acc)


def _neg(group, b):
    return m.g1_raw(m.g1_neg(m.g1_from_raw(b))) if group == 1 else m.g2_raw(m.g2_neg(m.g2_from_raw(b)))


@pytest.mark.parametrize("group", (1, 2))
def test_small_segments_against_the_oracle(sb, oracle, group):
    """segment lengths 0, 1, 2, 3, T - 1, T, T + 1 and a few hundred in one call, plus the edge segments: scalars 0, 1, r - 1, a repeated
    point (doubling inside a bucket), P and -P under one scalar (identity: all-zero bytes), identity points -- on both paths"""
    size = _size(group)
    rng = random.Random(100 + group)
    A, B = oracle.seeded_inputs(51, 64)
    src = A if group == 1 else B
    pt = [src[size * i:size * i + size] for i in range(64)]
    segs = []
    T = T1 if group == 1 else T2
    for length in (0, 1, 2, 3, T - 1, T, T + 1, 300):
        segs.append(([pt[rng.randrange(64)] for _ in range(length)], [rng.randrange(R) for _ in range(length)]))
    for reps in (1, T + 3):  # Straus and Pippenger forms of each edge segment
        segs.append((pt[:3] * reps, [0, 1, R - 1] * reps))
        segs.append(([pt[7]] * (4 * reps), [5] * (4 * reps)))
        segs.append(([pt[8], _neg(group, pt[8])] * reps, [12345, 12345] * reps))
        segs.append(([bytes(size), pt[9], bytes(size)] * reps, [7, rng.randrange(R), R - 1] * reps))
    pts = b"".join(b"".join(s[0]) for s in segs)
    ks = b"".join(le(k) for s in segs for k in s[1])
    got = _msm(sb, group)(pts, ks, [len(s[0]) for s in segs])
    for j, (p, k) in enumerate(segs):
        assert got[j] == _oracle_sum(oracle, group, b"".join(p), k), (group, j, len(k))
    assert got[0] == bytes(size)
    assert got[10] == bytes(size) and got[14] == bytes(size)  # P - P, both paths


def _device_inputs(sb, torch, seed, n):
    """seeded A_i = [a_i] G1, B_i = [b_i] G2 on the device, and (a_i, b_i)"""
    from oracle import pyoracle
    from sipp_b200 import _lib
    dA = torch.empty(64 * n, dtype=torch.uint8, device="cuda")
    dB = torch.empty(128 * n, dtype=torch.uint8, device="cuda")
    _lib.check(_lib.load().sipp_seeded_inputs_device(seed, n, dA.data_ptr(), dB.data_ptr()))
    raw = pyoracle.seeded_scalars(seed, n)
    ab = [int.from_bytes(raw[32 * i:32 * i + 32], "little") for i in range(2 * n)]
    return dA, dB, ab[0::2], ab[1::2]


def _scalars(seed, n):
    from oracle import pyoracle
    raw = pyoracle.seeded_scalars(seed, (n + 1) // 2)[:32 * n]
    return raw, [int.from_bytes(raw[32 * i:32 * i + 32], "little") for i in range(n)]


@pytest.mark.parametrize("shape", ["one_2p16", "one_2p20", "batch_4096x128", "ragged"])
def test_large_against_the_closed_form(sb, torch, shape):
    """MSM(A, s) over a segment == [sum a_i s_i mod r] G1 and MSM(B, s) == [sum b_i s_i mod r] G2 (generator paths)"""
    lengths = {"one_2p16": [1 << 16], "one_2p20": [1 << 20], "batch_4096x128": [128] * 4096,
               "ragged": [1, 0, 3, T2 - 1, T2, 5000, T1 - 1, 2, 1 << 14, T1, 700, 1, T1 + 1, 40000]}[shape]
    n = sum(lengths)
    dA, dB, a, b = _device_inputs(sb, torch, 61, n)
    kraw, s = _scalars(62, n)
    dk = torch.frombuffer(bytearray(kraw), dtype=torch.uint8).cuda()
    count = len(lengths)
    o1 = torch.empty(64 * count, dtype=torch.uint8, device="cuda")
    o2 = torch.empty(128 * count, dtype=torch.uint8, device="cuda")
    sb.g1_msm_batch_device(dA.data_ptr(), dk.data_ptr(), n, lengths, o1.data_ptr())
    sb.g2_msm_batch_device(dB.data_ptr(), dk.data_ptr(), n, lengths, o2.data_ptr())
    ta, tb, off = [], [], 0
    for length in lengths:
        ta.append(sum(a[i] * s[i] for i in range(off, off + length)) % R)
        tb.append(sum(b[i] * s[i] for i in range(off, off + length)) % R)
        off += length
    idx = list(range(count)) if count <= 64 else random.Random(5).sample(range(count), 64)
    got1, got2 = bytes(o1.cpu().numpy()), bytes(o2.cpu().numpy())
    g2gen = m.g2_raw(m.G2_GEN)
    want1 = sb.g1_generator_mul_batch([le(ta[j]) for j in idx])
    want2 = sb.g2_mul_batch(g2gen, [le(tb[j]) for j in idx])
    for q, j in enumerate(idx):
        w1 = want1[q] if ta[j] else bytes(64)
        w2 = want2[q] if tb[j] else bytes(128)
        assert got1[64 * j:64 * j + 64] == w1, (shape, j, lengths[j])
        assert got2[128 * j:128 * j + 128] == w2, (shape, j, lengths[j])


def test_segments_of_one(sb, oracle, torch):
    """G2: byte for byte sipp_g2_mul_batch; G1: oracle.g1_mul on a sample"""
    n = 4096
    dA, dB, _, _ = _device_inputs(sb, torch, 71, n)
    kraw, s = _scalars(72, n)
    kl = bytearray(kraw)
    kl[0:32], kl[32:64], kl[64:96] = le(0), le(1), le(R - 1)
    A, B = bytes(dA.cpu().numpy()), bytes(dB.cpu().numpy())
    got2 = sb.g2_msm_batch(B, bytes(kl), [1] * n)
    assert got2 == sb.g2_mul_batch(B, bytes(kl))
    got1 = sb.g1_msm_batch(A, bytes(kl), [1] * n)
    for i in [0, 1, 2] + random.Random(3).sample(range(3, n), 40):
        assert got1[i] == oracle.g1_mul(A[64 * i:64 * i + 64], bytes(kl[32 * i:32 * i + 32])), i


@pytest.mark.parametrize("group", (1, 2))
def test_host_form_equals_device_form(sb, torch, group):
    """byte-identical; device inputs written by torch right before the call need no synchronisation"""
    size = _size(group)
    lengths = [3, 0, T1, T2, 1000, 1, 129]
    n = sum(lengths)
    dA, dB, _, _ = _device_inputs(sb, torch, 81, n)
    kraw, _ = _scalars(82, n)
    dp = dA if group == 1 else dB
    host = _msm(sb, group)(bytes(dp.cpu().numpy()), kraw, lengths)
    fn = sb.g1_msm_batch_device if group == 1 else sb.g2_msm_batch_device
    kt = torch.frombuffer(bytearray(kraw), dtype=torch.uint8).cuda()
    torch.cuda.synchronize()
    pts2 = torch.empty_like(dp)
    k2 = torch.empty_like(kt)
    out = torch.full((size * len(lengths),), 0xA5, dtype=torch.uint8, device="cuda")
    big = torch.randn(4096, 4096, device="cuda")
    for _ in range(4):
        big = big @ big                               # keeps the legacy stream busy while the copies below queue behind it
    pts2.copy_(dp)
    k2.copy_(kt)
    fn(pts2.data_ptr(), k2.data_ptr(), n, lengths, out.data_ptr())
    assert [bytes(out[size * j:size * j + size].cpu().numpy()) for j in range(len(lengths))] == host


def _challenges(sb, A, B, proof):
    """x_k of sipp_verify_native (tests/golden/sipp_model.py): pairs, Z, then (Z_L, Z_R) per round"""
    n = len(A) // 64
    tr = sb.Transcript()
    for i in range(n):
        tr.append_g1(A[64 * i:64 * i + 64])
        tr.append_g2(B[128 * i:128 * i + 128])
    pf = list(proof)
    tr.append_fq12(pf.pop())
    xs = []
    while n > 1:
        tr.append_fq12(pf.pop())
        tr.append_fq12(pf.pop())
        xs.append(int.from_bytes(tr.get_challenge(), "little"))
        n //= 2
    return xs


def _fold_scalars(xs, n):
    """c_i = prod_k x_k^(bit (log2 n - 1 - k) of i)"""
    L = len(xs)
    out = []
    for i in range(n):
        c = 1
        for k, x in enumerate(xs):
            if (i >> (L - 1 - k)) & 1:
                c = c * x % R
        out.append(c)
    return out


def test_protocol_finals_are_msms(sb, oracle):
    """final_A = MSM(A, c), final_B = MSM(B, d) for the challenges of a seeded n = 2^12 proof, and for a 64-instance sample of a
    4,096 x 128 batch with one segment per instance"""
    n = 1 << 12
    A, B = oracle.seeded_inputs(91, n, threads=8)
    proof, st = sb.sipp_prove_native_statement(A, B)
    xs = _challenges(sb, A, B, proof)
    c = _fold_scalars(xs, n)
    d = _fold_scalars([pow(x, R - 2, R) for x in xs], n)
    assert sb.g1_msm_batch(A, b"".join(map(le, c)), [n]) == [st.final_A]
    assert sb.g2_msm_batch(B, b"".join(map(le, d)), [n]) == [st.final_B]
    cnt, m_ = 4096, 128
    A2, B2 = sb.seeded_inputs(92, cnt * m_)
    res = sb.sipp_prove_native_batch_statement(A2, B2, m_)
    sample = random.Random(9).sample(range(cnt), 64)
    cs, ds, pa, pb = [], [], [], []
    for j in sample:
        a, b = A2[64 * m_ * j:64 * m_ * (j + 1)], B2[128 * m_ * j:128 * m_ * (j + 1)]
        xs = _challenges(sb, a, b, res[j][0])
        cs += _fold_scalars(xs, m_)
        ds += _fold_scalars([pow(x, R - 2, R) for x in xs], m_)
        pa.append(a)
        pb.append(b)
    got1 = sb.g1_msm_batch(b"".join(pa), b"".join(map(le, cs)), [m_] * 64)
    got2 = sb.g2_msm_batch(b"".join(pb), b"".join(map(le, ds)), [m_] * 64)
    assert got1 == [res[j][1].final_A for j in sample]
    assert got2 == [res[j][1].final_B for j in sample]


def test_refusals(sb, oracle, torch):
    """a scalar >= r in the device form fails with SIPP_ERR_ENCODING and leaves d_out untouched; an off-curve G1 point and a G2 point
    outside the subgroup are refused with validation on; with SIPP_OPT_VALIDATE_POINTS = 0 valid inputs give the same bytes"""
    from sipp_b200 import _lib
    n = 40
    A, B = oracle.seeded_inputs(93, n)
    kraw, _ = _scalars(94, n)
    lengths = [1, 39]
    for group, pts in ((1, A), (2, B)):
        size = _size(group)
        fn = sb.g1_msm_batch_device if group == 1 else sb.g2_msm_batch_device
        bad = bytearray(kraw)
        bad[32 * 17:32 * 18] = le(R)
        dp = torch.frombuffer(bytearray(pts), dtype=torch.uint8).cuda()
        dk = torch.frombuffer(bad, dtype=torch.uint8).cuda()
        out = torch.full((size * 2,), 0x5A, dtype=torch.uint8, device="cuda")
        with pytest.raises(sb.SippError) as ei:
            fn(dp.data_ptr(), dk.data_ptr(), n, lengths, out.data_ptr())
        assert ei.value.code == _lib.ERR_ENCODING
        assert bytes(out.cpu().numpy()) == b"\x5a" * (size * 2)
        want = _msm(sb, group)(pts, kraw, lengths)
        try:
            sb.set_option(_lib.OPT_VALIDATE_POINTS, 0)
            assert _msm(sb, group)(pts, kraw, lengths) == want
        finally:
            sb.set_option(_lib.OPT_VALIDATE_POINTS, 1)
    off = bytearray(A)
    off[64 * 5 + 32:64 * 5 + 64] = le((int.from_bytes(off[64 * 5 + 32:64 * 5 + 64], "little") + 1) % P)  # y + 1: off the curve
    with pytest.raises(sb.SippError) as ei:
        sb.g1_msm_batch(bytes(off), kraw, lengths)
    assert ei.value.code == _lib.ERR_ENCODING and "curve" in str(ei.value)
    # a point of the twist outside G2: find x with x^3 + b' a square in Fq2, not multiplied by the cofactor
    x = 1
    while True:
        rhs = m.f2_add(m.f2_mul(m.f2_sqr((x, 1)), (x, 1)), m.B_TWIST)
        y = _fq2_sqrt(rhs)
        if y is not None:
            break
        x += 1
    q = m.g2_raw(((x, 1), y))
    with pytest.raises(sb.SippError) as ei:
        sb.g2_msm_batch(B[:128 * 39] + q, kraw, lengths)
    assert ei.value.code == _lib.ERR_ENCODING and "subgroup" in str(ei.value)


def _fq2_sqrt(a):
    """a square root in Fq2 = Fq[u]/(u^2 + 1), or None (p = 3 mod 4: the complex method)"""
    a0, a1 = a
    norm = (a0 * a0 + a1 * a1) % P
    s = pow(norm, (P + 1) // 4, P)
    if s * s % P != norm:
        return None
    for t in (s, P - s):
        x2 = (a0 + t) * pow(2, P - 2, P) % P
        x0 = pow(x2, (P + 1) // 4, P)
        if x0 * x0 % P == x2 and x0:
            x1 = a1 * pow(2 * x0, P - 2, P) % P
            if m.f2_sqr((x0, x1)) == (a0 % P, a1 % P):
                return (x0, x1)
    return None


@pytest.mark.parametrize("group", (1, 2))
def test_scalars_and_points_only_word_aligned(sb, torch, group):
    """device pointers that are 4- or 8-byte aligned but not 16-byte aligned are valid: same bytes as aligned buffers"""
    size = _size(group)
    lengths = [1, 5, T1 + 1, 300]
    n = sum(lengths)
    dA, dB, _, _ = _device_inputs(sb, torch, 83, n)
    kraw, _ = _scalars(84, n)
    dp = dA if group == 1 else dB
    fn = sb.g1_msm_batch_device if group == 1 else sb.g2_msm_batch_device
    want = _msm(sb, group)(bytes(dp.cpu().numpy()), kraw, lengths)
    for shift in (4, 8, 12):
        kbuf = torch.zeros(32 * n + 16, dtype=torch.uint8, device="cuda")
        pbuf = torch.zeros(size * n + 16, dtype=torch.uint8, device="cuda")
        kbuf[shift:shift + 32 * n] = torch.frombuffer(bytearray(kraw), dtype=torch.uint8).cuda()
        pbuf[shift:shift + size * n] = dp
        out = torch.zeros(size * len(lengths) + 16, dtype=torch.uint8, device="cuda")
        fn(pbuf.data_ptr() + shift, kbuf.data_ptr() + shift, n, lengths, out.data_ptr() + shift)
        got = bytes(out[shift:shift + size * len(lengths)].cpu().numpy())
        assert [got[size * j:size * j + size] for j in range(len(lengths))] == want, shift


def test_forced_paths_agree(sb, torch):
    """sipp_test_msm_batch_device: Straus and Pippenger (several c) give the plan's bytes on the same segments"""
    from sipp_b200 import _lib
    lib = _lib.load()
    lengths = [1, 3, 8, 15, 16, 40, 0, 200]
    n = sum(lengths)
    dA, dB, _, _ = _device_inputs(sb, torch, 85, n)
    kraw, _ = _scalars(86, n)
    dk = torch.frombuffer(bytearray(kraw), dtype=torch.uint8).cuda()
    offs = [0]
    for length in lengths:
        offs.append(offs[-1] + length)
    co = (ctypes.c_size_t * len(offs))(*offs)
    for group, dp in ((1, dA), (2, dB)):
        size = _size(group)
        want = _msm(sb, group)(bytes(dp.cpu().numpy()), kraw, lengths)
        for c in (0, 5, 9, 16):
            out = torch.empty(size * len(lengths), dtype=torch.uint8, device="cuda")
            _lib.check(lib.sipp_test_msm_batch_device(group, c, dp.data_ptr(), dk.data_ptr(), n, co, len(lengths), out.data_ptr()))
            got = bytes(out.cpu().numpy())
            assert [got[size * j:size * j + size] for j in range(len(lengths))] == want, (group, c)


def test_unweighted_and_repeated_scalars(sb, torch):
    """k_i = 1 for every point (one bucket holds every term: the block-summed long buckets) equals sipp_g2_sum / the closed form; so does
    one repeated random scalar"""
    n = 1 << 16
    dA, dB, a, b = _device_inputs(sb, torch, 87, n)
    A, B = bytes(dA.cpu().numpy()), bytes(dB.cpu().numpy())
    k = 0x1234567890ABCDEF1234567890ABCDEF % R
    for s in (1, k):
        ks = le(s) * n
        g1 = sb.g1_msm_batch(A, ks, [n])[0]
        g2 = sb.g2_msm_batch(B, ks, [n])[0]
        ta, tb = sum(a) * s % R, sum(b) * s % R
        assert g1 == sb.g1_generator_mul_batch([le(ta)])[0]
        assert g2 == sb.g2_mul_batch(m.g2_raw(m.G2_GEN), [le(tb)])[0]
        if s == 1:
            assert g2 == sb.g2_sum(B)


def test_device_refusal_precedence(sb, oracle, torch):
    """with a scalar >= r and a coordinate >= p in one call, both forms name the scalar (the host form's order)"""
    from sipp_b200 import _lib
    n = 20
    A, _ = oracle.seeded_inputs(95, n)
    kraw, _ = _scalars(96, n)
    k = bytearray(kraw)
    k[32 * 3:32 * 4] = le(R + 5)
    pts = bytearray(A)
    pts[64 * 11:64 * 11 + 32] = le(P)
    with pytest.raises(sb.SippError) as ei:
        sb.g1_msm_batch(bytes(pts), bytes(k), [n])
    assert ei.value.code == _lib.ERR_ENCODING and "scalar" in str(ei.value)
    out = torch.full((64,), 0x33, dtype=torch.uint8, device="cuda")
    dp = torch.frombuffer(pts, dtype=torch.uint8).cuda()
    dk = torch.frombuffer(k, dtype=torch.uint8).cuda()
    with pytest.raises(sb.SippError) as ei:
        sb.g1_msm_batch_device(dp.data_ptr(), dk.data_ptr(), n, [n], out.data_ptr())
    assert ei.value.code == _lib.ERR_ENCODING and "scalar" in str(ei.value)
    assert bytes(out.cpu().numpy()) == b"\x33" * 64
    k[32 * 3:32 * 4] = le(5)
    dk = torch.frombuffer(k, dtype=torch.uint8).cuda()
    with pytest.raises(sb.SippError) as ei:
        sb.g1_msm_batch_device(dp.data_ptr(), dk.data_ptr(), n, [n], out.data_ptr())
    assert ei.value.code == _lib.ERR_ENCODING and "coordinate" in str(ei.value)

