"""Batched multi-scalar multiplications (sipp_g1_msm_batch_device, sipp_g2_msm_batch_device) against what the library offered before,
on device-resident inputs.  python tools/msm_time.py [--out profiles/msm_time.json] [--reps 5]

  M1  G1, one segment of 2^16 and one of 2^20                      no earlier G1 path: points / s
  M2  G2, one segment of 2^16 and one of 2^20                      sipp_g2_mul_batch_device + sipp_g2_sum_device
  M3  4,096 segments of 128, G1 and G2                             G2: sipp_g2_mul_batch_device alone (a lower bound of the naive cost)
  M4  2^16 segments of 1, G2                                       sipp_g2_mul_batch_device (point_count = count)
  M5  verifier-shaped: n = 2^12, c_i / d_i products of 12 challenges, G1 + G2
  T*  both sides of the Straus / Pippenger thresholds (G1 13 points, G2 8): 4,096 segments of 4, 7, 8, 15, 16 and 32, G1 and G2
  M4 also times the C entry point with offsets built once, with and without the point validation (SIPP_OPT_VALIDATE_POINTS)
  X*  both paths forced at the same length (sipp_test_msm_batch_device): 4,096 segments of 8 .. 16 points (G1), 4 .. 12 (G2)
  U   unweighted sums, every k_i = 1 (one bucket holds every term), 2^20 points, G1 and G2   G2: sipp_g2_sum_device

Inputs are seeded points A_i = [a_i] G1, B_i = [b_i] G2 (sipp_seeded_inputs_device) and seeded scalars s_i.  Every timed output is
checked: against the comparison arm byte for byte, or against the closed form [sum a_i s_i] G1 / [sum b_i s_i] G2 (on a sample of
segments).  Warm wall times (a host clock around each call, which returns when its outputs are complete), the median of `reps` passes
with the arms alternated inside each pass.  The card's name and power limit are read in the same run."""
import argparse
import ctypes
import json
import os
import random
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
import torch  # noqa: E402

import sipp_b200  # noqa: E402
import sipp_model as m  # noqa: E402
from oracle import pyoracle  # noqa: E402
from sipp_b200 import _lib  # noqa: E402

R = m.R


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True, timeout=30)
        name, power = [x.strip() for x in q.stdout.strip().splitlines()[0].split(",")]
        return name, power
    except Exception as e:  # the numbers stay meaningful only with the card beside them: say so
        return "unknown (%s)" % e, "unknown"


def alternated(arms, reps):
    for fn in arms.values():
        fn()
    ts = {k: [] for k in arms}
    for _ in range(reps):
        for k, fn in arms.items():
            t0 = time.perf_counter()
            fn()
            ts[k].append((time.perf_counter() - t0) * 1e3)
    return {k: {"median_ms": round(statistics.median(v), 3), "min_ms": round(min(v), 3), "reps": reps} for k, v in ts.items()}


def le(v): return v.to_bytes(32, "little")


def dev(b): return torch.frombuffer(bytearray(b), dtype=torch.uint8).cuda()
def host(t): return bytes(t.cpu().numpy())


class Inputs:
    def __init__(self, n, seed=7):
        self.n = n
        self.dA = torch.empty(64 * n, dtype=torch.uint8, device="cuda")
        self.dB = torch.empty(128 * n, dtype=torch.uint8, device="cuda")
        _lib.check(_lib.load().sipp_seeded_inputs_device(seed, n, self.dA.data_ptr(), self.dB.data_ptr()))
        raw = pyoracle.seeded_scalars(seed, n)
        self.ab = [int.from_bytes(raw[32 * i:32 * i + 32], "little") for i in range(2 * n)]
        kraw = pyoracle.seeded_scalars(seed + 1, (n + 1) // 2)[:32 * n]
        self.s = [int.from_bytes(kraw[32 * i:32 * i + 32], "little") for i in range(n)]
        self.dk = dev(kraw)


def check_closed_form(inp, lengths, o1, o2, sample=16):
    """sampled segments of the G1 / G2 outputs against [sum a_i s_i] G1, [sum b_i s_i] G2"""
    offs = [0]
    for length in lengths:
        offs.append(offs[-1] + length)
    idx = list(range(len(lengths))) if len(lengths) <= sample else random.Random(1).sample(range(len(lengths)), sample)
    ok = True
    for j in idx:
        s, e = offs[j], offs[j + 1]
        if o1 is not None:
            t = sum(inp.ab[2 * i] * inp.s[i] for i in range(s, e)) % R
            want = sipp_b200.g1_generator_mul_batch([le(t)])[0] if t else bytes(64)
            ok &= host(o1[64 * j:64 * j + 64]) == want
        if o2 is not None:
            t = sum(inp.ab[2 * i + 1] * inp.s[i] for i in range(s, e)) % R
            want = sipp_b200.g2_mul_batch(m.g2_raw(m.G2_GEN), [le(t)])[0] if t else bytes(128)
            ok &= host(o2[128 * j:128 * j + 128]) == want
    return bool(ok)


def szt(v):
    return (ctypes.c_size_t * len(v))(*v)


def window_bits(group, length):
    """the window size msm.cu plans for a Pippenger segment of `length` points (its cost model)"""
    nc, bits = (2, 128) if group == 1 else (4, 66)
    return min(((bits // c + 1) * (nc * length + 3 * 2 ** (c - 1)), c) for c in range(5, 17))[1]


def msm_arm(group, inp, lengths, out):
    fn = sipp_b200.g1_msm_batch_device if group == 1 else sipp_b200.g2_msm_batch_device
    pts = inp.dA if group == 1 else inp.dB
    return lambda: fn(pts.data_ptr(), inp.dk.data_ptr(), inp.n, lengths, out.data_ptr())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--quick", action="store_true", help="skip the 2^20 segments")
    args = ap.parse_args()
    lib = _lib.load()
    _lib.require_gpu_once()
    name, power = card()
    res = {"card": name, "power_limit": power, "reps": args.reps, "workloads": {}}
    W = res["workloads"]

    def record(key, d):
        W[key] = d
        print(key, json.dumps(d), flush=True)

    # M1 / M2: one segment
    for n in ([1 << 16] if args.quick else [1 << 16, 1 << 20]):
        inp = Inputs(n)
        o1 = torch.empty(64, dtype=torch.uint8, device="cuda")
        o2 = torch.empty(128, dtype=torch.uint8, device="cuda")
        mul = torch.empty(128 * n, dtype=torch.uint8, device="cuda")
        naive = torch.empty(128, dtype=torch.uint8, device="cuda")

        def naive_g2():
            _lib.check(lib.sipp_g2_mul_batch_device(inp.dB.data_ptr(), n, inp.dk.data_ptr(), n, mul.data_ptr()))
            _lib.check(lib.sipp_g2_sum_device(mul.data_ptr(), n, naive.data_ptr()))
        t = alternated({"g1_msm": msm_arm(1, inp, [n], o1), "g2_msm": msm_arm(2, inp, [n], o2), "g2_mul_batch+g2_sum": naive_g2}, args.reps)
        ok = check_closed_form(inp, [n], o1, o2) and host(o2) == host(naive)
        record("M1_M2_n%d" % n, {"n": n, "times": t, "g1_points_per_s": round(n / (t["g1_msm"]["median_ms"] / 1e3)),
                                 "g2_points_per_s": round(n / (t["g2_msm"]["median_ms"] / 1e3)),
                                 "g2_speedup": round(t["g2_mul_batch+g2_sum"]["median_ms"] / t["g2_msm"]["median_ms"], 2), "outputs_ok": ok})
        del inp, mul

    # M3 and the threshold workloads: 4,096 segments of L
    for L in (128, 4, 7, 8, 15, 16, 32):
        count = 4096
        n = count * L
        inp = Inputs(n, seed=11)
        lengths = [L] * count
        o1 = torch.empty(64 * count, dtype=torch.uint8, device="cuda")
        o2 = torch.empty(128 * count, dtype=torch.uint8, device="cuda")
        mul = torch.empty(128 * n, dtype=torch.uint8, device="cuda")
        arms = {"g1_msm": msm_arm(1, inp, lengths, o1), "g2_msm": msm_arm(2, inp, lengths, o2)}
        if L == 128:
            arms["g2_mul_batch_alone"] = lambda: _lib.check(lib.sipp_g2_mul_batch_device(inp.dB.data_ptr(), n, inp.dk.data_ptr(), n, mul.data_ptr()))
        t = alternated(arms, args.reps)
        d = {"count": count, "length": L, "times": t, "outputs_ok": check_closed_form(inp, lengths, o1, o2),
             "g1_ns_per_point": round(t["g1_msm"]["median_ms"] * 1e6 / n, 1), "g2_ns_per_point": round(t["g2_msm"]["median_ms"] * 1e6 / n, 1)}
        if L == 128:
            d["g2_speedup_vs_mul_alone"] = round(t["g2_mul_batch_alone"]["median_ms"] / t["g2_msm"]["median_ms"], 2)
        record("M3_4096x128" if L == 128 else "T_4096x%d" % L, d)
        del inp, mul

    # M4: 2^16 segments of one point, G2
    n = 1 << 16
    inp = Inputs(n, seed=13)
    o2 = torch.empty(128 * n, dtype=torch.uint8, device="cuda")
    mul = torch.empty(128 * n, dtype=torch.uint8, device="cuda")
    o3 = torch.empty(128 * n, dtype=torch.uint8, device="cuda")
    o4 = torch.empty(128 * n, dtype=torch.uint8, device="cuda")
    offs = szt(list(range(n + 1)))  # built once: the C entry point without the Python wrapper's per-call offsets

    def c_entry(out):
        return lambda: _lib.check(lib.sipp_g2_msm_batch_device(inp.dB.data_ptr(), inp.dk.data_ptr(), n, offs, n, out.data_ptr()))

    def c_entry_unvalidated():
        sipp_b200.set_option(_lib.OPT_VALIDATE_POINTS, 0)
        try:
            c_entry(o4)()
        finally:
            sipp_b200.set_option(_lib.OPT_VALIDATE_POINTS, 1)
    t = alternated({"g2_msm": msm_arm(2, inp, [1] * n, o2), "g2_msm_c_entry": c_entry(o3), "g2_msm_c_entry_no_validation": c_entry_unvalidated,
                    "g2_mul_batch": lambda: _lib.check(lib.sipp_g2_mul_batch_device(inp.dB.data_ptr(), n, inp.dk.data_ptr(), n, mul.data_ptr()))},
                   args.reps)
    record("M4_2p16x1", {"count": n, "times": t, "g2_speedup": round(t["g2_mul_batch"]["median_ms"] / t["g2_msm"]["median_ms"], 2),
                         "g2_speedup_c_entry": round(t["g2_mul_batch"]["median_ms"] / t["g2_msm_c_entry"]["median_ms"], 2),
                         "g2_speedup_c_entry_no_validation": round(t["g2_mul_batch"]["median_ms"] / t["g2_msm_c_entry_no_validation"]["median_ms"], 2),
                         "outputs_ok": host(o2) == host(mul) and host(o3) == host(mul) and host(o4) == host(mul)})
    del inp, mul

    # X: both paths forced at the same lengths around the thresholds (sipp_test_msm_batch_device), 4,096 segments
    for group, lens in ((1, range(8, 17)), (2, range(4, 13))):
        for L in lens:
            count = 4096
            n = count * L
            inp = Inputs(n, seed=23)
            lengths = [L] * count
            co = szt([L * j for j in range(count + 1)])
            size = 64 if group == 1 else 128
            pts = inp.dA if group == 1 else inp.dB
            outs = {c: torch.empty(size * count, dtype=torch.uint8, device="cuda") for c in (0, window_bits(group, L))}
            arms = {("straus" if c == 0 else "pippenger_c%d" % c): (lambda c=c: _lib.check(lib.sipp_test_msm_batch_device(
                group, c, pts.data_ptr(), inp.dk.data_ptr(), n, co, count, outs[c].data_ptr()))) for c in outs}
            t = alternated(arms, args.reps)
            o = list(outs.values())
            ok = host(o[0]) == host(o[1]) and check_closed_form(inp, lengths, o[0] if group == 1 else None, o[0] if group == 2 else None, sample=8)
            record("X_g%d_4096x%d" % (group, L), {"group": group, "count": count, "length": L, "times": t, "outputs_ok": ok,
                                                 "planned": "straus" if L < (13 if group == 1 else 8) else "pippenger"})
            del inp

    # U: unweighted sums (every k_i = 1: one bucket holds every term), 2^20 points
    n = 1 << 20
    inp = Inputs(n, seed=29)
    ones = dev((1).to_bytes(32, "little") * n)
    o1 = torch.empty(64, dtype=torch.uint8, device="cuda")
    o2 = torch.empty(128, dtype=torch.uint8, device="cuda")
    sm = torch.empty(128, dtype=torch.uint8, device="cuda")
    t = alternated({"g1_msm": lambda: sipp_b200.g1_msm_batch_device(inp.dA.data_ptr(), ones.data_ptr(), n, [n], o1.data_ptr()),
                    "g2_msm": lambda: sipp_b200.g2_msm_batch_device(inp.dB.data_ptr(), ones.data_ptr(), n, [n], o2.data_ptr()),
                    "g2_sum": lambda: _lib.check(lib.sipp_g2_sum_device(inp.dB.data_ptr(), n, sm.data_ptr()))}, args.reps)
    inp.s = [1] * n
    record("U_unweighted_2p20", {"n": n, "times": t, "outputs_ok": check_closed_form(inp, [n], o1, o2) and host(o2) == host(sm)})
    del inp

    # M5: verifier-shaped, n = 2^12, scalars are products of 12 challenges (and of their inverses)
    n, L = 1 << 12, 12
    rng = random.Random(17)
    xs = [rng.randrange(1, R) for _ in range(L)]
    c, d = [], []
    for i in range(n):
        ci, di = 1, 1
        for k, x in enumerate(xs):
            if (i >> (L - 1 - k)) & 1:
                ci, di = ci * x % R, di * pow(x, R - 2, R) % R
        c.append(ci)
        d.append(di)
    inp = Inputs(n, seed=19)
    dc, dd = dev(b"".join(map(le, c))), dev(b"".join(map(le, d)))
    o1 = torch.empty(64, dtype=torch.uint8, device="cuda")
    o2 = torch.empty(128, dtype=torch.uint8, device="cuda")

    def both():
        sipp_b200.g1_msm_batch_device(inp.dA.data_ptr(), dc.data_ptr(), n, [n], o1.data_ptr())
        sipp_b200.g2_msm_batch_device(inp.dB.data_ptr(), dd.data_ptr(), n, [n], o2.data_ptr())
    t = alternated({"g1+g2_msm": both}, args.reps)
    inp.s = c
    ok1 = check_closed_form(inp, [n], o1, None)
    inp.s = d
    ok2 = check_closed_form(inp, [n], None, o2)
    record("M5_verifier_2p12", {"n": n, "times": t, "design_estimate_ms": 8.0, "outputs_ok": ok1 and ok2})

    res["all_outputs_ok"] = all(v["outputs_ok"] for v in W.values())
    print(json.dumps({"card": name, "power_limit": power, "all_outputs_ok": res["all_outputs_ok"]}))
    if args.out:
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)
    return 0 if res["all_outputs_ok"] else 1


if __name__ == "__main__":
    sys.exit(main())
