"""Batched multi-exponentiations in GT on the GPU (sipp_gt_msm_batch and its _device form): small segments of every path against
square-and-multiply on the oracle's Fq12 arithmetic, large ones against a closed form, forced paths against each other, host form
against device form, the refusals, and the tie to the protocol (final_Z of a proof is one multi-exponentiation of its proof elements,
for proof elements outside GT too)."""
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
T = 512  # the short / Pippenger threshold
ONE12 = (1).to_bytes(32, "little") + bytes(352)


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


def _rand_fq12(rng):
    return b"".join(le(rng.randrange(P)) for _ in range(12))


def _oracle_msm(oracle, elems, ks):
    """prod g_i^k_i by square-and-multiply on the oracle's Fq12 arithmetic (as tests/test_gpu_challenges.py oracle_pow), then products"""
    if not ks:
        return ONE12
    acc = ONE12 * len(ks)
    for bit in range(255, -1, -1):
        acc = oracle.field_op("FQ12_SQR", acc)
        sel = b"".join(g if (k >> bit) & 1 else ONE12 for g, k in zip(elems, ks))
        acc = oracle.field_op("FQ12_MUL", acc, sel)
    out = acc[:384]
    for i in range(1, len(ks)):
        out = oracle.field_op("FQ12_MUL", out, acc[384 * i:384 * i + 384])
    return out


def _edge_segments(oracle, rng, gt):
    """(elements, scalars) segments of lengths 0, 1, 2, T - 1, T, T + 1 and a few hundred, plus the edge cases on both sides of T"""
    ones = (1 << 5) - 1  # all-ones digits for c = 5 (and for every c dividing it): 0b11111...
    allones = sum(ones << (5 * w) for w in range(50)) % R
    pool = [gt[i] for i in range(len(gt))] + [_rand_fq12(rng) for _ in range(8)]
    segs = []
    for length in (0, 1, 2, T - 1, T, T + 1, 300):
        segs.append(([pool[rng.randrange(len(pool))] for _ in range(length)], [rng.randrange(R) for _ in range(length)]))
    g, h = gt[0], _rand_fq12(rng)
    ginv = oracle.field_op("FQ12_INV", g)
    maxfq = le(P - 1) * 12
    for reps in (1, T // 2 + 1):  # short and Pippenger forms of each edge segment
        segs.append(([g, h, pool[3]] * reps, [0, 1, R - 1] * reps))
        segs.append(([h, g] * reps, [(1 << 253) - 1, allones] * reps))
        segs.append(([g] * (3 * reps), [5, 5, 77] * reps))                      # a repeated element
        segs.append(([g, ginv] * reps, [12345, 12345] * reps))                  # an element next to its inverse: 1
        segs.append(([ONE12, h] * reps, [rng.randrange(R), 3] * reps))
        segs.append(([bytes(384), h] * reps, [0, 9] * reps))                    # 0^0 = 1
        segs.append(([bytes(384), h] * reps, [7, 9] * reps))                    # 0^7 = 0
        segs.append(([maxfq, h] * reps, [rng.randrange(R), 2] * reps))          # coordinates p - 1
    return segs


def _flatten(segs):
    return b"".join(b"".join(s[0]) for s in segs), b"".join(le(k) for s in segs for k in s[1]), [len(s[0]) for s in segs]


def test_small_segments_against_the_oracle(sb, oracle):
    """every length class and edge case against square-and-multiply; the empty segment gives one, g g^-1 gives one, 0^k gives 0"""
    rng = random.Random(7)
    A, B = oracle.seeded_inputs(31, 4)
    gt = [sb.pairing(A[64 * i:64 * i + 64], B[128 * i:128 * i + 128]) for i in range(4)]
    segs = _edge_segments(oracle, rng, gt)
    el, ks, lengths = _flatten(segs)
    got = sb.gt_msm_batch(el, ks, lengths)
    for j, (g, k) in enumerate(segs):
        assert got[j] == _oracle_msm(oracle, g, k), (j, len(k))
    assert got[0] == ONE12
    inv = [j for j, (g, k) in enumerate(segs) if len(g) == 2 and g[1] == oracle.field_op("FQ12_INV", g[0]) and k[0] == k[1]]
    assert inv and all(got[j] == ONE12 for j in inv)


def _forced(sb, torch, c, el, ks, lengths):
    from sipp_b200 import _lib
    n, count = len(ks) // 32, len(lengths)
    de = torch.frombuffer(bytearray(el), dtype=torch.uint8).cuda()
    dk = torch.frombuffer(bytearray(ks), dtype=torch.uint8).cuda()
    out = torch.empty(384 * count, dtype=torch.uint8, device="cuda")
    offs = [0]
    for length in lengths:
        offs.append(offs[-1] + length)
    _lib.check(_lib.load().sipp_test_gt_msm_batch_device(c, de.data_ptr(), dk.data_ptr(), n, (ctypes.c_size_t * len(offs))(*offs), count,
                                                         out.data_ptr()))
    b = bytes(out.cpu().numpy())
    return [b[384 * j:384 * j + 384] for j in range(count)]


def test_forced_paths_agree(sb, oracle, torch):
    """the short path and Pippenger with c = 2, 3, 5, 8, 13, 16 give the same bytes on the same segments, non-GT elements included"""
    rng = random.Random(8)
    A, B = oracle.seeded_inputs(32, 4)
    gt = [sb.pairing(A[64 * i:64 * i + 64], B[128 * i:128 * i + 128]) for i in range(4)]
    el, ks, lengths = _flatten(_edge_segments(oracle, rng, gt))
    want = sb.gt_msm_batch(el, ks, lengths)
    for c in (0, 2, 3, 5, 8, 13, 16):
        assert _forced(sb, torch, c, el, ks, lengths) == want, c


def _pair_elements(sb, torch, seed, n):
    """g_i = e(A_i, B_i) = e(G1, G2)^(a_i b_i) of seeded points, on the device, and the a_i b_i"""
    from oracle import pyoracle
    from sipp_b200 import _lib
    dA = torch.empty(64 * n, dtype=torch.uint8, device="cuda")
    dB = torch.empty(128 * n, dtype=torch.uint8, device="cuda")
    _lib.check(_lib.load().sipp_seeded_inputs_device(seed, n, dA.data_ptr(), dB.data_ptr()))
    raw = pyoracle.seeded_scalars(seed, n)
    ab = [int.from_bytes(raw[32 * i:32 * i + 32], "little") for i in range(2 * n)]
    de = torch.empty(384 * n, dtype=torch.uint8, device="cuda")
    sb.inner_product_batch_device(dA.data_ptr(), dB.data_ptr(), n, [1] * n, de.data_ptr())
    return de, [a * b % R for a, b in zip(ab[0::2], ab[1::2])]


def _scalars(seed, n):
    from oracle import pyoracle
    raw = pyoracle.seeded_scalars(seed, (n + 1) // 2)[:32 * n]
    return raw, [int.from_bytes(raw[32 * i:32 * i + 32], "little") for i in range(n)]


def _closed_form(sb, ts):
    g2 = m.g2_raw(m.G2_GEN)
    pts = sb.g1_generator_mul_batch([le(t) for t in ts])
    return sb.pairing_batch(pts, [g2] * len(ts))


@pytest.mark.parametrize("shape", ["one_2p16", "one_2p20", "batch_4096x128", "unweighted_2p16"])
def test_large_against_the_closed_form(sb, torch, shape):
    """prod e(A_i, B_i)^(k_i) over a segment == e([sum a_i b_i k_i mod r] G1, G2)"""
    lengths = {"one_2p16": [1 << 16], "one_2p20": [1 << 20], "batch_4096x128": [128] * 4096, "unweighted_2p16": [1 << 16]}[shape]
    n = sum(lengths)
    de, ab = _pair_elements(sb, torch, 41, n)
    if shape.startswith("unweighted"):
        kraw, s = le(1) * n, [1] * n
    else:
        kraw, s = _scalars(42, n)
    dk = torch.frombuffer(bytearray(kraw), dtype=torch.uint8).cuda()
    count = len(lengths)
    out = torch.empty(384 * count, dtype=torch.uint8, device="cuda")
    sb.gt_msm_batch_device(de.data_ptr(), dk.data_ptr(), n, lengths, out.data_ptr())
    idx = list(range(count)) if count <= 64 else random.Random(5).sample(range(count), 64)
    ts, off = [], [0]
    for length in lengths:
        off.append(off[-1] + length)
    for j in idx:
        ts.append(sum(ab[i] * s[i] for i in range(off[j], off[j + 1])) % R)
    want = _closed_form(sb, ts)
    got = bytes(out.cpu().numpy())
    for q, j in enumerate(idx):
        assert got[384 * j:384 * j + 384] == want[q], (shape, j)


def test_host_form_equals_device_form(sb, oracle, torch):
    """byte-identical; device inputs only 4-byte aligned and written by torch right before the call need no synchronisation"""
    rng = random.Random(9)
    lengths = [3, 0, T - 1, T, 1000, 1, 129]
    n = sum(lengths)
    el = b"".join(_rand_fq12(rng) for _ in range(n))
    kraw = b"".join(le(rng.randrange(R)) for _ in range(n))
    host = sb.gt_msm_batch(el, kraw, lengths)
    e_src = torch.frombuffer(bytearray(el), dtype=torch.uint8).cuda()
    k_src = torch.frombuffer(bytearray(kraw), dtype=torch.uint8).cuda()
    torch.cuda.synchronize()
    e2 = torch.empty(384 * n + 4, dtype=torch.uint8, device="cuda")
    k2 = torch.empty(32 * n + 4, dtype=torch.uint8, device="cuda")
    out = torch.full((384 * len(lengths) + 4,), 0xA5, dtype=torch.uint8, device="cuda")
    big = torch.randn(4096, 4096, device="cuda")
    for _ in range(4):
        big = big @ big                               # keeps the legacy stream busy while the copies below queue behind it
    e2[4:].copy_(e_src)
    k2[4:].copy_(k_src)
    sb.gt_msm_batch_device(e2.data_ptr() + 4, k2.data_ptr() + 4, n, lengths, out.data_ptr() + 4)
    got = bytes(out.cpu().numpy())
    assert [got[4 + 384 * j:4 + 384 * j + 384] for j in range(len(lengths))] == host
    assert got[:4] == b"\xa5" * 4


def test_refusals(sb, torch):
    """scalar >= r and coordinate >= p give SIPP_ERR_ENCODING on the device, scalar first, and leave d_out untouched"""
    from sipp_b200 import _lib
    rng = random.Random(10)
    lengths = [2, T + 3]
    n = sum(lengths)
    el = bytearray(b"".join(_rand_fq12(rng) for _ in range(n)))
    ks = bytearray(b"".join(le(rng.randrange(R)) for _ in range(n)))
    bad_el = bytearray(el)
    bad_el[384 * 6 + 32 * 11:384 * 6 + 32 * 12] = le(P)
    for seg_elem in (1, n - 1):  # one refusal on each path
        bad_k = bytearray(ks)
        bad_k[32 * seg_elem:32 * seg_elem + 32] = le(R)
        for e_, k_, what in ((el, bad_k, "scalar"), (bad_el, ks, "p"), (bad_el, bad_k, "scalar")):
            de = torch.frombuffer(bytearray(e_), dtype=torch.uint8).cuda()
            dk = torch.frombuffer(bytearray(k_), dtype=torch.uint8).cuda()
            out = torch.full((384 * 2,), 0x5A, dtype=torch.uint8, device="cuda")
            with pytest.raises(sb.SippError) as ei:
                sb.gt_msm_batch_device(de.data_ptr(), dk.data_ptr(), n, lengths, out.data_ptr())
            assert ei.value.code == _lib.ERR_ENCODING
            assert what in _lib.load().sipp_last_error().decode()
            assert bytes(out.cpu().numpy()) == b"\x5a" * 768
    # the library still works after a refusal
    assert sb.gt_msm_batch(bytes(el), bytes(ks), lengths) == sb.gt_msm_batch(bytes(el), bytes(ks), lengths)


# ---- the protocol tie: final_Z = Z prod_k Z_L(k)^x_k Z_R(k)^(1/x_k) -----------------------------------------------------------------
def _challenges_and_factors(sb, A, B, proof):
    n = len(A) // 64
    tr = sb.Transcript()
    for i in range(n):
        tr.append_g1(A[64 * i:64 * i + 64])
        tr.append_g2(B[128 * i:128 * i + 128])
    pf = list(proof)
    z = pf.pop()
    tr.append_fq12(z)
    elems, ks = [z], [1]
    while n > 1:
        zl, zr = pf.pop(), pf.pop()
        tr.append_fq12(zl)
        tr.append_fq12(zr)
        x = int.from_bytes(tr.get_challenge(), "little")
        elems += [zl, zr]
        ks += [x, pow(x, R - 2, R)]
        n //= 2
    return elems, ks


def _verify_final_z(sb, A, B, proof):
    """sipp_verify_native's status and final_Z (written on SIPP_ERR_VERIFY too)"""
    from sipp_b200 import _lib
    p = b"".join(proof)
    fa, fb, fz = (ctypes.create_string_buffer(s) for s in (64, 128, 384))
    rc = _lib.load().sipp_verify_native(A, len(A) // 64, B, len(B) // 128, p, len(p) // 384, fa, fb, fz)
    return rc, fz.raw


@pytest.mark.parametrize("fe_norm", [0, 1])
def test_protocol_tie(sb, oracle, fe_norm):
    """for seeded proofs of n = 2, 2^7, 2^12 and a 64-proof sample of a 4,096 x 128 batch, gt_msm_batch over [Z, Z_L(k), Z_R(k)] with
    [1, x_k, 1/x_k] from the replayed transcript equals sipp_verify_native's final_Z byte for byte -- also for a proof whose Z_L(1) is a
    random Fq12 outside GT, which the verifier rejects while still writing final_Z"""
    from sipp_b200 import _lib
    old = _lib.load().sipp_get_option(_lib.OPT_FE_NORMALISATION)
    _lib.check(_lib.load().sipp_set_option(_lib.OPT_FE_NORMALISATION, fe_norm))
    try:
        segs, want = [], []
        for seed, n in ((121, 2), (122, 1 << 7), (123, 1 << 12)):
            A, B = oracle.seeded_inputs(seed, n, threads=8)
            proof = sb.sipp_prove_native(A, B)
            st = sb.sipp_verify_native(A, B, proof)
            segs.append(_challenges_and_factors(sb, A, B, proof))
            want.append(st.final_Z)
        # a proof element outside GT: the verifier fails, its final_Z is still the product of powers
        A, B = oracle.seeded_inputs(124, 16)
        proof = list(sb.sipp_prove_native(A, B))
        proof[-2] = _rand_fq12(random.Random(11))
        rc, fz = _verify_final_z(sb, A, B, proof)
        assert rc == _lib.ERR_VERIFY
        segs.append(_challenges_and_factors(sb, A, B, proof))
        want.append(fz)
        # a 64-proof sample of a 4,096 x 128 batch
        cnt, m_ = 4096, 128
        A2, B2 = sb.seeded_inputs(125, cnt * m_)
        res = sb.sipp_prove_native_batch_statement(A2, B2, m_)
        for j in random.Random(12).sample(range(cnt), 64):
            a, b = A2[64 * m_ * j:64 * m_ * (j + 1)], B2[128 * m_ * j:128 * m_ * (j + 1)]
            segs.append(_challenges_and_factors(sb, a, b, res[j][0]))
            want.append(res[j][1].final_Z)
        el, ks, lengths = _flatten(segs)
        assert sb.gt_msm_batch(el, ks, lengths) == want
    finally:
        _lib.check(_lib.load().sipp_set_option(_lib.OPT_FE_NORMALISATION, old))
