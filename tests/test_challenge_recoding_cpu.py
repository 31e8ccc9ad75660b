"""CPU checks of the fold-challenge catalogue (tests/challenge_catalogue.py) and of the fold-scalar contract: the host recoding of every
catalogue pair is a valid plan, the catalogue reaches the branches of the fold kernels that random challenges do not, and
sipp_gt_fold refuses out-of-range, zero and mismatched scalars before it needs a device."""
import ctypes
import random

import pytest

import challenge_catalogue as cc

R = cc.R


@pytest.fixture(scope="module")
def lib():
    from sipp_b200 import _lib
    return _lib.load()


@pytest.fixture(scope="module")
def plist(lib):
    return cc.pairs(cc.catalogue(lib))


def test_constants():
    assert (cc.L1 * cc.L1 + cc.L1 + 1) % R == 0            # phi^2 + phi + 1 = 0 on G1
    assert (cc.L2**4 - cc.L2**2 + 1) % R == 0              # the 12th cyclotomic polynomial at p = L2 (mod r)
    assert cc.L2 < R and cc.L2 == 0x6f4d8248eeb859fbf83e9682e87cfd46  # the eigenvalue glv_consts.h was generated for


def test_catalogue_plans_recombine(lib, plist):
    """every pair: sum_j v_j L1^j == x, sum_j v_j L2^j == x^-1 (mod r), G1 sub-scalars < 2^128 (NAF <= 129 digits), G2 < 2^66
    (NAF <= 67), non-adjacent digits, and g1_bits / g2_bits the longest component"""
    for label, x, xi in plist:
        g1, g2, b1, b2 = cc.components(cc.host_plan(x, xi, lib))
        assert sum(v * pow(cc.L1, j, R) for j, (v, _) in enumerate(g1)) % R == x, label
        assert sum(v * pow(cc.L2, j, R) for j, (v, _) in enumerate(g2)) % R == xi, label
        assert all(abs(v) < 2**128 for v, _ in g1) and all(abs(v) < 2**66 for v, _ in g2), label
        assert b1 == max(d for _, d in g1) <= 129 and b2 == max(d for _, d in g2) <= 67, label


def test_structured_decompositions(lib):
    """the sign and NAF length of every component of the structured scalars, as measured on this recoding"""
    for name, (c, want_g1, want_g2) in cc.STRUCTURED.items():
        g1, _, _, _ = cc.components(cc.host_plan(c, cc.inv(c), lib))
        _, g2, _, _ = cc.components(cc.host_plan(cc.inv(c), c, lib))
        assert cc.profile(g1) == want_g1, (name, cc.profile(g1))
        assert cc.profile(g2) == want_g2, (name, cc.profile(g2))


def test_catalogue_reaches_the_kernel_branches(lib, plist):
    f = cc.classify(plist, lib)
    zero_at = [j for j in range(4) if f["g2_zero_at"][j]]
    assert len(zero_at) >= 3, f["g2_zero_at"]               # a zero G2 / GT component at three different indices
    assert f["g1_zero_first"]                               # the G1 component sum starts from the identity
    assert f["g1_negative"] and f["g2_negative"]
    assert f["g1_one_digit"] and f["g2_one_digit"]
    assert f["g2_66"] and f["g1_128"]                       # the longest schedules random scalars give


def test_random_scalars_miss_those_branches(lib):
    """why the catalogue exists: random scalars reach none of the zero or one-digit components"""
    rng = random.Random(1)
    f = cc.classify([("r%d" % i, x, cc.inv(x)) for i, x in enumerate(rng.randrange(1, R) for _ in range(300))], lib)
    assert not any(f["g2_zero_at"].values()) and not f["g1_zero_first"]
    assert not f["g1_one_digit"] and not f["g2_one_digit"]


def test_longest_naf_search_is_seeded(lib):
    a, b = cc.longest_naf_scalars(lib), cc.longest_naf_scalars(lib)
    assert a == b
    _, _, b1, _ = cc.components(cc.host_plan(a["naf128-g1"], 1, lib))
    _, _, _, b2 = cc.components(cc.host_plan(1, a["naf66-g2"], lib))
    assert (b1, b2) == (128, 66)


def test_boundary_scalars_straddle_a_rounding_step():
    tables = cc.babai_tables()
    assert [s for _, s in tables["g1"]] == [-1, -1] and [s for _, s in tables["g2"]] == [1, 1, 1, 1]
    edges = cc.boundary_scalars(per_row=3)
    assert len(edges) == 2 * 3 * 6
    for name, k in edges.items():
        if name.endswith("minus1"):
            continue
        key, i = name.split("-")[1], int(name.split("-")[2])
        g, sign = tables[key][i]
        assert cc.babai_coefficient(k, g, sign) != cc.babai_coefficient(k - 1, g, sign), name
        assert k - 1 == edges[name + "-minus1"]


def test_boundary_scalars_recode(lib):
    for k in cc.boundary_scalars(seed=7, per_row=4).values():
        for x, xi in ((k, cc.inv(k)), (cc.inv(k), k)):
            g1, g2, _, _ = cc.components(cc.host_plan(x, xi, lib))
            assert sum(v * pow(cc.L1, j, R) for j, (v, _) in enumerate(g1)) % R == x
            assert sum(v * pow(cc.L2, j, R) for j, (v, _) in enumerate(g2)) % R == xi


@pytest.mark.parametrize("x, xi, code", [
    (R, 1, -6),                       # x = r: would be reduced mod r
    (2**256 - 1, 1, -6),
    (1, R, -6),                       # x_inv = r
    (0, 0, -4),                       # zero challenge: the reference panics on x.inverse().unwrap()
    (0, 1, -4),
    (2, 2, -6),                       # not inverse to each other
    (3, pow(2, -1, R), -6),
], ids=["x=r", "x=2^256-1", "x_inv=r", "zero", "zero-x_inv=1", "2,2", "3,1/2"])
def test_gt_fold_refuses_bad_scalars_without_a_device(lib, x, xi, code):
    """sipp_gt_fold checks its scalars before it touches the device: the refusal is the same with or without a GPU"""
    out = ctypes.create_string_buffer(384)
    one = (1).to_bytes(32, "little") + bytes(352)
    rc = lib.sipp_gt_fold(one, one, one, cc.le(x), cc.le(xi), out)
    assert rc == code, lib.sipp_last_error()
    if code == -6 and x < R and xi < R:
        assert b"not the inverse" in lib.sipp_last_error()
    assert out.raw == bytes(384)


def test_fold_batch_hook_checks_arguments_without_a_device(lib):
    """sipp_test_fold_batch checks its scalar pairs (as sipp_ctx_fold) before it needs a device"""
    A, B = bytes(64 * 4), bytes(128 * 4)
    out_a, out_b = ctypes.create_string_buffer(64 * 4), ctypes.create_string_buffer(128 * 4)
    xs = cc.le(5) + cc.le(7)
    good = cc.le(cc.inv(5)) + cc.le(cc.inv(7))
    bad = cc.le(cc.inv(5)) + cc.le(cc.inv(5))
    assert lib.sipp_test_fold_batch(A, B, 2, 2, xs, bad, 0, out_a, out_b) == -6
    assert lib.sipp_test_fold_batch(A, B, 2, 2, cc.le(5) + cc.le(0), good, 0, out_a, out_b) == -4
    assert lib.sipp_test_fold_batch(A, B, 3, 1, xs, good, 0, out_a, out_b) == -2   # n odd
    assert lib.sipp_test_fold_batch(A, B, 2, 2, xs, good, 3, out_a, out_b) == -2   # no such kernel
    if lib.sipp_device_count() == 0:
        assert lib.sipp_test_fold_batch(A, B, 2, 2, xs, good, 0, out_a, out_b) == -1
