"""Chosen fold challenges for the tests of the fold and GT-exponentiation kernels.  TEST ONLY.

Every fold round multiplies G1 by the challenge x and G2 by x^-1.  The host (glv.cc) and the device transcript (k_transcript.cu)
recode both into short sub-scalars -- GLV with 2 components for G1 (x = k0 + k1 L1), GLS with 4 for G2 and GT
(k = k0 + k1 L2 + k2 L2^2 + k3 L2^3) -- written in non-adjacent form.  The kernels that consume these plans have branches that
random challenges (what Poseidon hands them) almost never reach: zero, negative and one-digit sub-scalars, a zero first component,
the longest digit schedules.  The scalars here reach them on purpose; each is used as (c, c^-1) and as (c^-1, c), so that G1, G2
and GT each get the structured side.
"""
import ctypes
import os
import random
import re

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
R = 0x30644E72E131A029B85045B68181585D2833E84879B9709143E1F593F0000001
U = 4965661367192848881                                 # the BN parameter
L2 = 6 * U * U                                          # psi acts on G2 as [L2], the p-power Frobenius on GT as well
L1 = 0xb3c4d79d41a917585bfc41088d8daaa78b17ea66b99c90dd  # phi acts on G1 as [L1]
PLAN_WORDS = 68                                         # 6 x {plus[5], minus[5], neg}, g1_bits, g2_bits

# name -> scalar, with its host recoding: (sign, NAF digits) per component, 0 for a zero component; G1 from x = c, G2 / GT from
# x^-1 = c (the orientation (c^-1, c))
STRUCTURED = {
    "1": (1, [(1, 1), 0], [(1, 1), 0, 0, 0]),
    "u": (U, [(1, 63), 0], [(1, 63), 0, 0, 0]),
    "2^64": (2**64, [(1, 65), 0], [(1, 65), 0, 0, 0]),
    "2^66": (2**66, [(1, 67), 0], [(1, 65), (-1, 2), (1, 2), (-1, 2)]),
    "r-1": (R - 1, [(-1, 1), 0], [(1, 66), (1, 1), (-1, 1), (1, 1)]),
    "L2^2": (L2**2 % R, [0, (-1, 1)], [(1, 65), (1, 1), (-1, 64), 0]),
    "L2^3": (L2**3 % R, [(1, 128), (-1, 128)], [(1, 65), 0, (-1, 1), (-1, 65)]),
    "r-L2": (R - L2, [(1, 66), (-1, 128)], [(1, 65), (1, 64), 0, (-1, 63)]),
    "r-L1": (R - L1, [0, (-1, 1)], [(1, 65), (1, 1), (-1, 64), 0]),
    "r-2^128": (R - 2**128, [(1, 127), (-1, 128)], [(1, 66), (1, 64), (1, 63), (-1, 64)]),
}
SEARCH_SEED = 20261021


def le(v):
    return v.to_bytes(32, "little")


def inv(v):
    return pow(v, -1, R)


def _lib():
    from sipp_b200 import _lib as L
    return L.load()


def host_plan(x, x_inv, lib=None):
    """the 68 plan words of sipp_test_fold_plan (glv.cc) for the pair"""
    lib = lib or _lib()
    buf = (ctypes.c_uint32 * PLAN_WORDS)()
    nw = lib.sipp_test_fold_plan(le(x), le(x_inv), buf, PLAN_WORDS)
    assert nw == PLAN_WORDS, nw
    return list(buf)


def components(words):
    """plan words -> ([(value, digits) for the 2 G1 components], [... the 4 G2 components], g1_bits, g2_bits); value is the signed
    sub-scalar the kernel applies to endo^j(P), digits its NAF length.  Asserts the masks are disjoint and non-adjacent."""
    out = []
    for j in range(6):
        w = words[11 * j:11 * j + 11]
        plus = sum(w[i] << (32 * i) for i in range(5))
        minus = sum(w[5 + i] << (32 * i) for i in range(5))
        assert plus & minus == 0, "a digit is both +1 and -1"
        nz = plus | minus
        assert nz & (nz >> 1) == 0, "adjacent non-zero digits"
        v = plus - minus
        out.append((-v if w[10] else v, nz.bit_length()))
    return out[:2], out[2:], words[66], words[67]


def profile(comps):
    """[(sign, digits) or 0] per component, as in STRUCTURED"""
    return [0 if v == 0 else (1 if v > 0 else -1, d) for v, d in comps]


def _splitmix(state):
    state = (state + 0x9E3779B97F4A7C15) & (2**64 - 1)
    z = state
    z = ((z ^ (z >> 30)) * 0xBF58476D1CE4E5B9) & (2**64 - 1)
    z = ((z ^ (z >> 27)) * 0x94D049BB133111EB) & (2**64 - 1)
    return state, z ^ (z >> 31)


def seeded_scalars(seed=SEARCH_SEED):
    """SplitMix64 limbs, least significant first, top limb masked to 62 bits, values >= r rejected"""
    s = seed
    while True:
        limbs = []
        for _ in range(4):
            s, z = _splitmix(s)
            limbs.append(z)
        limbs[3] &= 2**62 - 1
        k = sum(limbs[i] << (64 * i) for i in range(4))
        if k < R:
            yield k


def longest_naf_scalars(lib=None, limit=20000):
    """the first scalars of the seeded stream whose host recoding reaches the longest NAF seen over 3 x 10^6 random scalars: 66
    digits for a G2 component, 128 for a G1 component (scalar c: G1 from x = c, G2 from x^-1 = c)"""
    lib = lib or _lib()
    g1 = g2 = None
    for i, k in enumerate(seeded_scalars()):
        if i >= limit:
            break
        _, _, b1, b2 = components(host_plan(k, k, lib))
        if g1 is None and b1 == 128:
            g1 = k
        if g2 is None and b2 == 66:
            g2 = k
        if g1 is not None and g2 is not None:
            return {"naf128-g1": g1, "naf66-g2": g2}
    raise AssertionError("the seeded search found no 128-digit G1 / 66-digit G2 recoding")


def babai_tables():
    """the rounding constants of glv_consts.h: {'g1': [(g_i, sign_i)] * 2, 'g2': [(g_i, sign_i)] * 4}"""
    src = open(os.path.join(ROOT, "sipp_b200", "csrc", "glv_consts.h")).read()
    out = {}
    for key, name in (("g1", "SIPP_GLV_G1_RECIP"), ("g2", "SIPP_GLS_G2_RECIP")):
        body = re.search(name + r"\[\d\]\[5\] = \{(.*?)\};", src, re.S).group(1)
        rows = re.findall(r"\{([^{}]*)\}", body)
        gs = [sum(int(x, 16) << (64 * i) for i, x in enumerate(re.findall(r"0x([0-9a-f]+)ull", row))) for row in rows]
        signs = [int(x) for x in re.search(name + r"_SIGN\[\d\] = \{([^}]*)\}", src).group(1).split(",")]
        assert len(gs) == len(signs) == (2 if key == "g1" else 4)
        out[key] = list(zip(gs, signs))
    return out


def babai_coefficient(k, g, sign):
    return sign * (k * g >> 320)


def boundary_scalars(seed=5, per_row=1):
    """k = ceil(m 2^320 / g_i) and k - 1 for random m: the smallest scalars whose Babai coefficient c_i = sign_i floor(k g_i / 2^320)
    steps, i.e. the edges of the rounding domain of every row of both bases (all below r)"""
    rng = random.Random(seed)
    out = {}
    for key, rows in babai_tables().items():
        for i, (g, sign) in enumerate(rows):
            mmax = R * g >> 320
            for t in range(per_row):
                m = rng.randrange(1, mmax)
                k = -(-(m << 320) // g)
                assert 1 < k < R
                out["edge-%s-%d-%d" % (key, i, t)] = k
                out["edge-%s-%d-%d-minus1" % (key, i, t)] = k - 1
    return out


def catalogue(lib=None, n_random=4, seed=11):
    """name -> scalar: the structured scalars, the longest-NAF scalars, the Babai edges and a few random ones"""
    cat = {name: v for name, (v, _, _) in STRUCTURED.items()}
    cat.update(longest_naf_scalars(lib))
    cat.update(boundary_scalars())
    rng = random.Random(seed)
    for i in range(n_random):
        cat["random-%d" % i] = rng.randrange(2, R)
    assert all(0 < v < R for v in cat.values())
    return cat


def pairs(cat):
    """[(label, x, x^-1)]: every scalar in both orientations"""
    out = []
    for name, c in cat.items():
        out.append((name, c, inv(c)))
        out.append((name + "^-1", inv(c), c))
    return out


def classify(plist, lib=None):
    """what the host plans of the pairs reach: sets of labels per property"""
    lib = lib or _lib()
    found = {"g2_zero_at": {0: set(), 1: set(), 2: set(), 3: set()}, "g1_zero_first": set(), "g1_negative": set(), "g2_negative": set(),
             "g1_one_digit": set(), "g2_one_digit": set(), "g2_66": set(), "g1_128": set()}
    for label, x, xi in plist:
        g1, g2, b1, b2 = components(host_plan(x, xi, lib))
        for j, (v, _) in enumerate(g2):
            if v == 0:
                found["g2_zero_at"][j].add(label)
        if g1[0][0] == 0:
            found["g1_zero_first"].add(label)
        if any(v < 0 for v, _ in g1):
            found["g1_negative"].add(label)
        if any(v < 0 for v, _ in g2):
            found["g2_negative"].add(label)
        if any(d == 1 for _, d in g1):
            found["g1_one_digit"].add(label)
        if any(d == 1 for _, d in g2):
            found["g2_one_digit"].add(label)
        if b2 == 66:
            found["g2_66"].add(label)
        if b1 == 128:
            found["g1_128"].add(label)
    return found
