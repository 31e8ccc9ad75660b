"""The fold and GT-exponentiation kernels under chosen challenges (tests/challenge_catalogue.py): zero, negative and one-digit
sub-scalars, a zero first component, the longest digit schedules and the Babai rounding edges, which the transcript's random
challenges practically never produce.  Every expected value comes from the CPU oracle, except where a docstring says otherwise:
the device recoding against the host recoding, the single-proof and batched point folds, the pairing-matrix stages, sipp_gt_fold,
and the refusal of bad fold scalars on every route."""
import ctypes
import os
import random
from concurrent.futures import ThreadPoolExecutor

import pytest

import challenge_catalogue as cc

pytestmark = pytest.mark.gpu
R = cc.R
P = 0x30644E72E131A029B85045B68181585D97816A916871CA8D3C208C16D87CFD47
ONE12 = (1).to_bytes(32, "little") + bytes(352)
THREADS = os.cpu_count() or 1
# every option of include/sipp_b200.h with its default
DEFAULTS = {1: 0, 2: 0, 3: 0, 4: 1, 5: 8192, 6: 1, 7: 256, 8: 1536, 9: 32, 10: 1, 11: 0, 12: 1, 13: 1, 14: 32, 15: 256, 16: 8, 17: 1, 18: 0}
le = cc.le


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


@pytest.fixture(scope="module")
def plist(lib):
    return cc.pairs(cc.catalogue(lib))


@pytest.fixture(scope="module")
def base(oracle):
    return oracle.seeded_inputs(61, 2000, threads=THREADS)


def pmap(fn, items):
    with ThreadPoolExecutor(max_workers=THREADS) as ex:  # the oracle's ctypes calls release the GIL
        return list(ex.map(fn, items))


def g1(A, i): return A[64 * i:64 * i + 64]
def g2(B, i): return B[128 * i:128 * i + 128]


def plant(oracle, A, B, h, x, xi, kinds=(0, 1, 2, 3), at=0):
    """exceptional points of the fold A_i + x A_{i+h}, B_i + x^-1 B_{i+h}: kind 0 an identity partner, 1 an identity base, 2 a doubling
    (A_i = x A_{i+h}, B_i = x^-1 B_{i+h}), 3 a sum equal to O (A_i = -x A_{i+h}, B_i = -x^-1 B_{i+h}); element at + t for the t-th kind"""
    A, B = bytearray(A), bytearray(B)
    for t, kind in enumerate(kinds):
        i = (at + t) % h
        if kind == 0:
            A[64 * (i + h):64 * (i + h + 1)] = bytes(64)
            B[128 * (i + h):128 * (i + h + 1)] = bytes(128)
        elif kind == 1:
            A[64 * i:64 * (i + 1)] = bytes(64)
            B[128 * i:128 * (i + 1)] = bytes(128)
        else:
            sx, sxi = (x, xi) if kind == 2 else (R - x, R - xi)
            A[64 * i:64 * (i + 1)] = oracle.g1_mul(g1(A, i + h), le(sx))
            B[128 * i:128 * (i + 1)] = oracle.g2_mul(g2(B, i + h), le(sxi))
    return bytes(A), bytes(B)


def oracle_fold(oracle, A, B, x, xi, idx=None):
    """A_i + x A_{i+h}, B_i + x^-1 B_{i+h} for i in idx (all i < h by default)"""
    h = len(A) // 128
    if idx is not None:
        A = b"".join(g1(A, i) for i in idx) + b"".join(g1(A, i + h) for i in idx)
        B = b"".join(g2(B, i) for i in idx) + b"".join(g2(B, i + h) for i in idx)
    return oracle.fold_g1(A, le(x)), oracle.fold_g2(B, le(xi))


def ctx_fold(sipp, A, B, x, xi):
    ctx = sipp.ProverContext(A, B)
    try:
        ctx.fold(le(x), le(xi))
        assert len(ctx) == len(A) // 128
        return ctx.read()
    finally:
        ctx.close()


# ------------------------------------------------------------------------------------------------ 1. device recoding
def test_device_recoding_matches_host(lib, plist):
    """glv::plan_build on the device (the tables of k_tr_round) gives the host plan word for word: the catalogue in both
    orientations, the Babai edges of every row and 10^5 random pairs"""
    rng = random.Random(21)
    prs = [(x, xi) for _, x, xi in plist]
    for k in cc.boundary_scalars(seed=9, per_row=8).values():
        prs += [(k, cc.inv(k)), (cc.inv(k), k)]
    prs += [(x, cc.inv(x)) for x in (rng.randrange(1, R) for _ in range(100000))]
    count = len(prs)
    xs = b"".join(le(x) for x, _ in prs)
    xis = b"".join(le(xi) for _, xi in prs)
    dev = (ctypes.c_uint32 * (cc.PLAN_WORDS * count))()
    assert lib.sipp_test_fold_plan_device(xs, xis, count, dev) == 0, lib.sipp_last_error()
    host = (ctypes.c_uint32 * (cc.PLAN_WORDS * count))()
    for j in range(count):
        out = ctypes.cast(ctypes.addressof(host) + 4 * cc.PLAN_WORDS * j, ctypes.POINTER(ctypes.c_uint32))
        assert lib.sipp_test_fold_plan(xs[32 * j:32 * j + 32], xis[32 * j:32 * j + 32], out, cc.PLAN_WORDS) == cc.PLAN_WORDS
    if bytes(dev) != bytes(host):
        bad = next(j for j in range(count) if dev[cc.PLAN_WORDS * j:cc.PLAN_WORDS * (j + 1)] != host[cc.PLAN_WORDS * j:cc.PLAN_WORDS * (j + 1)])
        pytest.fail("device plan differs for pair %d: x = %#x" % (bad, prs[bad][0]))


# ------------------------------------------------------------------------------------------------ 2. single-proof point folds
@pytest.mark.parametrize("h", [1, 7, 16, 17, 33, 257, 1000])
def test_point_fold_catalogue(sipp, lib, oracle, plist, base, h):
    """every catalogue pair on k_fold_wide (SIPP_OPT_WIDE_FOLD_MAX above h) and on k_fold_split (0), with the exceptional points
    planted under that scalar.  Up to h = 257 every point is compared with the oracle; at h = 1000 the two kernels must agree byte for
    byte and the planted points plus 24 random ones are compared with the oracle."""
    from sipp_b200 import _lib
    A0, B0 = base[0][:64 * 2 * h], base[1][:128 * 2 * h]
    rng = random.Random(h)
    cases = []
    for k, (label, x, xi) in enumerate(plist):
        if h >= 4:
            A, B = plant(oracle, A0, B0, h, x, xi, at=k % h)
            planted = [(k % h + t) % h for t in range(4)]
        else:
            A, B = plant(oracle, A0, B0, h, x, xi, kinds=(k % 4,))
            planted = [0]
        idx = None if h <= 257 else sorted(set(planted + rng.sample(range(h), 24)))
        cases.append((label, x, xi, A, B, idx))
    want = pmap(lambda c: oracle_fold(oracle, c[3], c[4], c[1], c[2], c[5]), cases)
    got = {}
    for kernel, wide in (("k_fold_wide", 1 << 20), ("k_fold_split", 0)):
        _lib.check(lib.sipp_set_option(_lib.OPT_WIDE_FOLD_MAX, wide))
        for (label, x, xi, A, B, idx), (wa, wb) in zip(cases, want):
            a, b = ctx_fold(sipp, A, B, x, xi)
            got[kernel, label] = (a, b)
            if idx is not None:
                a = b"".join(g1(a, i) for i in idx)
                b = b"".join(g2(b, i) for i in idx)
            assert a == wa, (kernel, label, "G1")
            assert b == wb, (kernel, label, "G2")
    for label, *_ in cases:
        assert got["k_fold_wide", label] == got["k_fold_split", label], label


def test_point_fold_straus(sipp, lib, oracle):
    """k_fold_straus (a single proof with h >= 16384) for r - L1, L2^2, 2^64, 1 and r - 1 in both orientations: bytes equal to
    k_fold_split (GPU against GPU over all 2 x 16384 points), and the planted exceptional points and a random sample against the
    oracle"""
    from sipp_b200 import _lib
    h = 16384
    A0, B0 = sipp.seeded_inputs(62, 2 * h)
    rng = random.Random(5)
    for name in ("r-L1", "L2^2", "2^64", "1", "r-1"):
        c = cc.STRUCTURED[name][0]
        for x, xi in ((c, cc.inv(c)), (cc.inv(c), c)):
            at = rng.randrange(h - 4)
            A, B = plant(oracle, A0, B0, h, x, xi, at=at)
            _lib.check(lib.sipp_set_option(_lib.OPT_FOLD_STRAUS, 1))
            got = ctx_fold(sipp, A, B, x, xi)
            _lib.check(lib.sipp_set_option(_lib.OPT_FOLD_STRAUS, 0))
            _lib.check(lib.sipp_set_option(_lib.OPT_WIDE_FOLD_MAX, 0))
            split = ctx_fold(sipp, A, B, x, xi)
            _lib.check(lib.sipp_set_option(_lib.OPT_WIDE_FOLD_MAX, DEFAULTS[_lib.OPT_WIDE_FOLD_MAX]))
            assert got == split, (name, x == c)
            idx = sorted(set([at, at + 1, at + 2, at + 3, 0, h - 1] + rng.sample(range(h), 10)))
            wa, wb = oracle_fold(oracle, A, B, x, xi, idx)
            assert b"".join(g1(got[0], i) for i in idx) == wa and b"".join(g2(got[1], i) for i in idx) == wb, (name, x == c)


# ------------------------------------------------------------------------------------------------ 3. batched folds, mixed plans
def fold_batch(lib, A, B, n, count, xs, xis, kernel):
    h = n // 2
    oa, ob = ctypes.create_string_buffer(64 * h * count), ctypes.create_string_buffer(128 * h * count)
    rc = lib.sipp_test_fold_batch(A, B, n, count, b"".join(le(x) for x in xs), b"".join(le(x) for x in xis), kernel, oa, ob)
    assert rc == 0, lib.sipp_last_error()
    return oa.raw, ob.raw


@pytest.mark.parametrize("h", [1, 2, 3, 8, 16, 17, 31, 32, 33])
def test_batched_fold_mixed_plans(lib, oracle, plist, base, h):
    """24 instances whose scalars cycle through the catalogue (so one warp holds plans of 1 and of 66 / 128 digits, zero and
    non-zero components) on k_fold_batch, k_fold_wide_batch and k_fold_straus, exceptional points planted in every third instance:
    every folded point against the oracle"""
    count, n = 24, 2 * h
    A, B = bytearray(), bytearray()
    xs, xis, want_jobs = [], [], []
    for j in range(count):
        _, x, xi = plist[(j * 7 + h) % len(plist)]
        a, b = base[0][64 * n * j:64 * n * (j + 1)], base[1][128 * n * j:128 * n * (j + 1)]
        if j % 3 == 0:
            a, b = plant(oracle, a, b, h, x, xi, kinds=(0, 1, 2, 3) if h >= 4 else ((j // 3) % 4,), at=j % h)
        A += a
        B += b
        xs.append(x)
        xis.append(xi)
        want_jobs.append((a, b, x, xi))
    want = pmap(lambda w: oracle_fold(oracle, *w), want_jobs)
    wa, wb = b"".join(w[0] for w in want), b"".join(w[1] for w in want)
    for kernel in (0, 1, 2):
        a, b = fold_batch(lib, bytes(A), bytes(B), n, count, xs, xis, kernel)
        for j in range(count):
            assert a[64 * h * j:64 * h * (j + 1)] == wa[64 * h * j:64 * h * (j + 1)], (kernel, j, "G1")
            assert b[128 * h * j:128 * h * (j + 1)] == wb[128 * h * j:128 * h * (j + 1)], (kernel, j, "G2")


def test_batched_fold_single_scalar_equals_single_proof_fold(sipp, lib, plist, base):
    """one scalar for every instance: each kernel's batch equals the single-proof fold of each instance (GPU against GPU)"""
    count, n = 8, 32
    A, B = base[0][:64 * n * count], base[1][:128 * n * count]
    for label in ("2^64", "L2^2^-1", "r-1"):
        x, xi = next((x, xi) for lab, x, xi in plist if lab == label)
        single = [ctx_fold(sipp, A[64 * n * j:64 * n * (j + 1)], B[128 * n * j:128 * n * (j + 1)], x, xi) for j in range(count)]
        for kernel in (0, 1, 2):
            a, b = fold_batch(lib, A, B, n, count, [x] * count, [xi] * count, kernel)
            assert a == b"".join(s[0] for s in single) and b == b"".join(s[1] for s in single), (label, kernel)


# ------------------------------------------------------------------------------------------------ 4. stages with chosen challenges
# the challenge of round k: SEQ[k % len(SEQ)] (catalogue labels; "^-1" = the orientation (c^-1, c))
SEQ = ["2^64", "2^64^-1", "L2^2", "1", "L2^3^-1", "r-L2", "r-1^-1", "2^66", "u^-1", "r-L1^-1", "naf66-g2^-1", "naf128-g1", "r-2^128"]


def schedule(lib, n):
    """per round of a proof of n points with stages on, under the current options: 'mat' (k_mat_fold runs with the round's GT plan),
    'last' (the last round of a stage: no matrix fold) or 'point' (the points are folded, no stage)"""
    kinds, m, mt = [], n, lib.sipp_test_stage_blocks(0, n)
    while m > 1:
        if not mt:
            mt = lib.sipp_test_stage_blocks(1, m)
        if mt:
            kinds.append("mat" if mt > 2 else "last")
            mt = mt // 2 if mt > 2 else 0
        else:
            kinds.append("point")
        m //= 2
    return kinds


def gt_zero(lib, k):
    """the GT recoding of k (the G2 tables, as gt_plan_build) has a zero sub-scalar"""
    _, comps, _, _ = cc.components(cc.host_plan(1, k, lib))
    return any(v == 0 for v, _ in comps)


def oracle_rounds(oracle, A, B, chal):
    """Z, then Z_L, Z_R of every round on the point route, and the points after every fold"""
    out, pts = [oracle.inner_product(A, B, threads=THREADS)], []
    for x, xi in chal:
        h = len(A) // 128
        out += [oracle.inner_product(A[64 * h:], B[:128 * h], threads=THREADS), oracle.inner_product(A[:64 * h], B[128 * h:], threads=THREADS)]
        A, B = oracle_fold(oracle, A, B, x, xi)
        pts.append((A, B))
    return out, pts


def run_rounds(sipp, A, B, chal, stages, bad=None):
    """the round loop of a host with its own transcript, with the given challenges; returns Z, Z_L, Z_R of every round and, per round,
    the points read after the fold (None once they are refused).  bad(ctx, round) runs before every fold."""
    ctx = sipp.ProverContext(A, B)
    try:
        ctx.set_stages(stages)
        out, pts = [ctx.inner_product()], []
        for k, (x, xi) in enumerate(chal):
            out += list(ctx.cross_products())
            if bad:
                bad(ctx, k)
            ctx.fold(le(x), le(xi))
            try:
                pts.append(ctx.read())
            except sipp.SippError as e:
                assert e.code == -2
                pts.append(None)
        assert len(ctx) == 1
        return out, pts
    finally:
        ctx.close()


def challenges(plist, rounds, offset=0):
    by = {label: (x, xi) for label, x, xi in plist}
    return [by[SEQ[(k + offset) % len(SEQ)]] for k in range(rounds)]


@pytest.mark.parametrize("n, first", [(16, 1), (128, 0), (1024, 1)], ids=["tail", "lookahead-tail", "first-lookahead-tail"])
def test_stage_route_chosen_challenges(sipp, lib, oracle, plist, n, first):
    """the pairing-matrix stages (k_mat_fold on GT, the look-ahead point folds) with challenges from the catalogue: every Z, Z_L,
    Z_R equals the oracle's on the point route, the points read during a look-ahead stage are the oracle's folded points, and reads
    are refused once the tail has begun"""
    from sipp_b200 import _lib
    _lib.check(lib.sipp_set_option(_lib.OPT_MATRIX_FIRST, first))
    kinds = schedule(lib, n)
    want_kinds = {16: ["mat"] * 3 + ["last"], 128: ["mat", "mat", "last"] + ["mat"] * 3 + ["last"],
                  1024: ["mat", "mat", "last"] * 2 + ["mat"] * 3 + ["last"]}[n]
    assert kinds == want_kinds, kinds
    A, B = oracle.seeded_inputs(70 + n, n, threads=THREADS)
    chal = challenges(plist, len(kinds))
    mat = [c for c, k in zip(chal, kinds) if k == "mat"]
    assert any(gt_zero(lib, x) for x, _ in mat) and any(gt_zero(lib, xi) for _, xi in mat)   # the zero-sub-scalar branch, both exponents
    want, want_pts = oracle_rounds(oracle, A, B, chal)
    got, pts = run_rounds(sipp, A, B, chal, True)
    assert len(got) == len(want)
    for k, (g, w) in enumerate(zip(got, want)):
        assert g == w, "element %d of %d" % (k, len(want))
    # the points stay readable until the first fold of the tail (the stage of single points), refused from there on
    tail = max(k for k in range(len(kinds)) if k == 0 or kinds[k - 1] == "last")
    for k, p in enumerate(pts):
        if k < tail:
            assert p == want_pts[k], k
        else:
            assert p is None, k


def test_stage_route_n4096_against_point_route(sipp, lib, plist):
    """n = 4096 (first stage of 32 blocks, a look-ahead stage, the tail) with catalogue challenges, against the same loop with stages
    off (GPU against GPU: the oracle is slow at this size)"""
    n = 4096
    kinds = schedule(lib, n)
    assert kinds == ["mat"] * 4 + ["last"] + ["mat", "mat", "last"] + ["mat"] * 3 + ["last"], kinds
    A, B = sipp.seeded_inputs(71, n)
    chal = challenges(plist, len(kinds), offset=3)
    mat = [c for c, k in zip(chal, kinds) if k == "mat"]
    assert any(gt_zero(lib, x) for x, _ in mat) and any(gt_zero(lib, xi) for _, xi in mat)
    on, _ = run_rounds(sipp, A, B, chal, True)
    off, _ = run_rounds(sipp, A, B, chal, False)
    assert on == off


# ------------------------------------------------------------------------------------------------ 5. sipp_gt_fold
def oracle_pow(oracle, bases, exps):
    """bases[i]^exps[i] by square-and-multiply on the oracle's Fq12 arithmetic, all at once"""
    acc = ONE12 * len(bases)
    for bit in range(255, -1, -1):
        acc = oracle.field_op("FQ12_SQR", acc)
        sel = b"".join(b if (e >> bit) & 1 else ONE12 for b, e in zip(bases, exps))
        acc = oracle.field_op("FQ12_MUL", acc, sel)
    return [acc[384 * i:384 * (i + 1)] for i in range(len(bases))]


@pytest.mark.parametrize("engine", [1, 0], ids=["engine", "per-thread"])
def test_gt_fold_exponents(sipp, lib, oracle, plist, engine):
    """Z_L^x Z Z_R^(1/x) (sipp_gt_fold) for the catalogue pairs and the edges of the 2-bit windows (3, 4, 2^253 - 1, 2^128 +- 1,
    r - 2, with their inverses, both orientations), on GT elements and on arbitrary Fq12 elements"""
    from sipp_b200 import _lib
    _lib.check(lib.sipp_set_option(_lib.OPT_FE_ENGINE, engine))
    prs = [(x, xi) for _, x, xi in plist]
    for e in (3, 4, 2**253 - 1, 2**128 - 1, 2**128 + 1, R - 2):
        prs += [(e, cc.inv(e)), (cc.inv(e), e)]
    A, B = oracle.seeded_inputs(73, 6, threads=THREADS)
    gt = [oracle.pairing(g1(A, i), g2(B, i)) for i in range(6)]
    rng = random.Random(74)
    triples = []
    for k in range(len(prs)):
        if k % 2:
            triples.append(tuple(b"".join(rng.randrange(P).to_bytes(32, "little") for _ in range(12)) for _ in range(3)))
        else:
            triples.append((gt[k % 6], gt[(k + 1) % 6], gt[(k + 2) % 6]))
    zl = oracle_pow(oracle, [t[0] for t in triples], [x for x, _ in prs])
    zr = oracle_pow(oracle, [t[2] for t in triples], [xi for _, xi in prs])
    want = oracle.field_op("FQ12_MUL", oracle.field_op("FQ12_MUL", b"".join(zl), b"".join(t[1] for t in triples)), b"".join(zr))
    for k, ((x, xi), (a, z, b)) in enumerate(zip(prs, triples)):
        out = ctypes.create_string_buffer(384)
        assert lib.sipp_gt_fold(a, z, b, le(x), le(xi), out) == 0, lib.sipp_last_error()
        assert out.raw == want[384 * k:384 * (k + 1)], (k, hex(x))


# ------------------------------------------------------------------------------------------------ 6. refusals
BAD = [("x=r", lambda x, xi: (R, xi), -6), ("x=2^256-1", lambda x, xi: (2**256 - 1, xi), -6), ("x_inv=r", lambda x, xi: (x, R), -6),
       ("x=0", lambda x, xi: (0, xi), -4), ("mismatched", lambda x, xi: (x, (xi + 1) % R), -6)]


@pytest.mark.parametrize("n, first, stages", [(16, 1, False), (128, 1, True), (128, 0, True)],
                         ids=["point-route", "first-stage-tail", "lookahead-tail"])
def test_fold_refuses_bad_scalars(sipp, lib, oracle, plist, n, first, stages):
    """x = r, x = 2^256 - 1, x_inv = r, x = 0 and a wrong inverse are refused before every fold -- on the point route and, with
    stages on, during the first stage, a look-ahead stage, the tail and the tail's last round -- with the context unchanged: the
    valid folds that follow give the oracle's Z_L, Z_R and points"""
    from sipp_b200 import _lib
    _lib.check(lib.sipp_set_option(_lib.OPT_MATRIX_FIRST, first))
    kinds = schedule(lib, n) if stages else ["point"] * 4
    if stages:
        assert kinds[-1] == "last" and "mat" in kinds
    A, B = oracle.seeded_inputs(80 + n, n, threads=THREADS)
    chal = challenges(plist, len(kinds), offset=5)
    seen = set()

    def bad(ctx, k):
        before = len(ctx)
        for name, make, code in BAD:
            x, xi = make(*chal[k])
            with pytest.raises(sipp.SippError) as ei:
                ctx.fold(le(x), le(xi))
            assert ei.value.code == code, (name, k)
            assert len(ctx) == before, (name, k)
        seen.add(kinds[k])

    want, want_pts = oracle_rounds(oracle, A, B, chal)
    got, pts = run_rounds(sipp, A, B, chal, stages, bad)
    assert got == want
    assert seen == ({"mat", "last"} if stages else {"point"})
    for p, w in zip(pts, want_pts):
        assert p is None or p == w
    if not stages:
        assert all(p is not None for p in pts)
