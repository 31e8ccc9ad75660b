"""Batched multi-exponentiations in GT (sipp_gt_msm_batch_device) on device-resident inputs.
python tools/gt_msm_time.py [--out profiles/gt_msm_time.json] [--reps 5]

  G1  one segment of 2^16 and one of 2^20 elements
  V*  verifier-shaped batches, 4,096 segments of 1 + 2 log2 n elements ([Z, Z_L(k), Z_R(k)] with [1, x_k, 1/x_k]): n = 2^12 (25 elements)
      and n = 128 (15).  Comparison: the per-round sipp_gt_fold route (log2 n dependent calls per proof), timed on a 64-proof sample and
      scaled by 4,096 / 64
  U   unweighted product, every k_i = 1 (one bucket holds every element), 2^20 elements
  X*  both paths forced at the same length (sipp_test_gt_msm_batch_device): 4,096 segments of 2 .. 256 elements (fewer segments of 512
      and 1,024, 2^20 elements in all), the short path against Pippenger with the window size of the cost model
  S*  the same for one segment of 2^12 .. 2^18 elements.  The X and S rows set the threshold.

Elements are e(A_i, B_i) of seeded points (sipp_seeded_inputs_device, sipp_inner_product_batch_device with segments of one), scalars
seeded.  Every timed output is checked: against the closed form e([sum a_i b_i k_i] G1, G2) on a sample of segments, or against the
comparison arm byte for byte.  Warm wall times (a host clock around each call, which returns when its outputs are complete), the median
of `reps` passes with the arms alternated inside each pass.  The card's name and power limit are read in the same run."""
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
def szt(v): return (ctypes.c_size_t * len(v))(*v)


class Elements:
    """g_i = e(A_i, B_i) = e(G1, G2)^(a_i b_i) on the device"""
    def __init__(self, n, seed):
        self.n = n
        dA = torch.empty(64 * n, dtype=torch.uint8, device="cuda")
        dB = torch.empty(128 * n, dtype=torch.uint8, device="cuda")
        _lib.check(_lib.load().sipp_seeded_inputs_device(seed, n, dA.data_ptr(), dB.data_ptr()))
        raw = pyoracle.seeded_scalars(seed, n)
        ab = [int.from_bytes(raw[32 * i:32 * i + 32], "little") for i in range(2 * n)]
        self.e = [a * b % R for a, b in zip(ab[0::2], ab[1::2])]
        self.d = torch.empty(384 * n, dtype=torch.uint8, device="cuda")
        sipp_b200.inner_product_batch_device(dA.data_ptr(), dB.data_ptr(), n, [1] * n, self.d.data_ptr())


def closed_form_ok(el, ks, lengths, out, sample=8):
    offs = [0]
    for length in lengths:
        offs.append(offs[-1] + length)
    idx = list(range(len(lengths))) if len(lengths) <= sample else random.Random(1).sample(range(len(lengths)), sample)
    ts = [sum(el.e[i] * ks[i] for i in range(offs[j], offs[j + 1])) % R for j in idx]
    want = sipp_b200.pairing_batch(sipp_b200.g1_generator_mul_batch([le(t) for t in ts]), [m.g2_raw(m.G2_GEN)] * len(ts))
    got = host(out)
    return all(got[384 * j:384 * j + 384] == want[q] for q, j in enumerate(idx))


def gt_call(c, d_el, d_k, n, lengths, out):
    offs = [0]
    for length in lengths:
        offs.append(offs[-1] + length)
    o = szt(offs)
    lib = _lib.load()
    if c is None:
        return lambda: _lib.check(lib.sipp_gt_msm_batch_device(d_el.data_ptr(), d_k.data_ptr(), n, o, len(lengths), out.data_ptr()))
    return lambda: _lib.check(lib.sipp_test_gt_msm_batch_device(c, d_el.data_ptr(), d_k.data_ptr(), n, o, len(lengths), out.data_ptr()))


def plan_c(length):
    out = (ctypes.c_int * 2)()
    _lib.load().sipp_test_gt_msm_plan(szt([0, length]), 1, out, 2)
    return out[1]


def pippenger_c(length):
    """the window size the cost model gives a Pippenger segment of this length (the plan's, when it plans Pippenger)"""
    return min((-(-254 // c) * (length + 2 * 2 ** c) + c * -(-254 // c), c) for c in range(2, 17))[1]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "gt_msm_time.json"))
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--quick", action="store_true", help="only the threshold rows")
    a = ap.parse_args()
    _lib.require_gpu(0)
    name, power = card()
    res = {"card": name, "power_limit": power, "reps": a.reps, "rows": {}}
    rows = res["rows"]
    big = Elements(1 << 20, 5)
    rng = random.Random(3)
    ks_all = [rng.randrange(R) for _ in range(1 << 20)]
    dk_all = dev(b"".join(le(k) for k in ks_all))

    def row(key, lengths, arms, check):
        t = alternated(arms, a.reps)
        rows[key] = {"lengths": lengths if len(lengths) <= 4 else "%d x %d" % (len(lengths), lengths[0]), "times": t, "checked": bool(check())}
        print(key, json.dumps(rows[key]), flush=True)

    # X: both paths forced, 4,096 segments of each length (fewer beyond 256, so that they fit the 2^20 elements); S: one segment
    for length in (2, 4, 7, 8, 9, 16, 32, 64, 128, 256, 512, 1024, 1 << 12, 1 << 14, 1 << 16, 1 << 18):
        cnt = 1 if length >= 1 << 12 else min(4096, (1 << 20) // length)
        n = cnt * length
        lengths = [length] * cnt
        o0 = torch.empty(384 * cnt, dtype=torch.uint8, device="cuda")
        o1 = torch.empty_like(o0)
        cp = pippenger_c(length)
        key = ("S_len%d" if cnt == 1 else "X_len%d") % length
        row(key, lengths, {"short": gt_call(0, big.d, dk_all, n, lengths, o0), "pippenger_c%d" % cp: gt_call(cp, big.d, dk_all, n, lengths, o1)},
            lambda: host(o0) == host(o1) and closed_form_ok(big, ks_all, lengths, o0))
        rows[key]["plan_c"] = plan_c(length)
    if not a.quick:
        # G1: one segment
        for lg in (16, 20):
            n = 1 << lg
            o = torch.empty(384, dtype=torch.uint8, device="cuda")
            row("G1_2p%d" % lg, [n], {"gt_msm": gt_call(None, big.d, dk_all, n, [n], o)}, lambda: closed_form_ok(big, ks_all, [n], o))
        # U: unweighted
        n = 1 << 20
        ones = [1] * n
        d1 = dev(le(1) * n)
        o = torch.empty(384, dtype=torch.uint8, device="cuda")
        row("U_2p20", [n], {"gt_msm": gt_call(None, big.d, d1, n, [n], o)}, lambda: closed_form_ok(big, ones, [n], o))
        # V: verifier-shaped, against the per-round sipp_gt_fold route on 64 proofs (scaled)
        lib = _lib.load()
        for logn in (12, 7):
            seg = 1 + 2 * logn
            n = 4096 * seg
            xs = [rng.randrange(1, R) for _ in range(4096 * logn)]
            ks = []
            for j in range(4096):
                ks.append(1)
                for k in range(logn):
                    x = xs[j * logn + k]
                    ks += [x, pow(x, R - 2, R)]
            dk = dev(b"".join(le(k) for k in ks))
            lengths = [seg] * 4096
            o = torch.empty(384 * 4096, dtype=torch.uint8, device="cuda")
            el_host = host(big.d[:384 * 64 * seg])
            fold_out = [None] * 64

            def fold_route():
                for j in range(64):
                    base = 384 * seg * j
                    z = el_host[base:base + 384]
                    buf = ctypes.create_string_buffer(384)
                    for k in range(logn):
                        zl = el_host[base + 384 * (1 + 2 * k):base + 384 * (2 + 2 * k)]
                        zr = el_host[base + 384 * (2 + 2 * k):base + 384 * (3 + 2 * k)]
                        _lib.check(lib.sipp_gt_fold(zl, z, zr, le(ks[seg * j + 1 + 2 * k]), le(ks[seg * j + 2 + 2 * k]), buf))
                        z = buf.raw
                    fold_out[j] = z
            arms = {"gt_msm_4096": gt_call(None, big.d, dk, n, lengths, o), "gt_fold_route_64": fold_route}
            key = "V_n2p%d" % logn
            row(key, lengths, arms, lambda: host(o)[:384 * 64] == b"".join(fold_out) and closed_form_ok(big, ks, lengths, o))
            t = rows[key]["times"]["gt_fold_route_64"]["median_ms"]
            rows[key]["gt_fold_route_4096_scaled_ms"] = round(t * 4096 / 64, 1)
            rows[key]["gt_fold_calls_per_proof"] = logn
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({"card": name, "power_limit": power}))


if __name__ == "__main__":
    main()
