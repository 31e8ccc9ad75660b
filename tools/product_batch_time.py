"""Batched independent products (sipp_inner_product_batch, sipp_pairing_batch) against loops of the one-product calls, on seeded
inputs, in one process.  python tools/product_batch_time.py [--out profiles/product_batch_time.json] [--reps 5]

  W1  4,096 segments of 128 pairs (checking 4,096 BLS aggregates)    vs a loop of sipp_inner_product over the first 256, extrapolated
  W2  pairing_batch of 2^16 pairs                                    vs a loop of 256 sipp_pairing calls, extrapolated
  W3  one 2^16 segment plus 4,095 seeded lengths in 0..64 (skewed)
  W4  one 2^16 segment                                               vs sipp_inner_product on the same pairs

Per workload: warm wall time (host clock around calls that end in a device synchronise, after one warm-up call; W1's 15 GB line
table is far beyond the 126 MB of L2, so every pass reads HBM), Miller loops/s from miller_ms of a separate SIPP_OPT_PROFILE = 1
pass, and a seeded sample of 64 outputs compared with sipp_inner_product.  The card's name and power limit are recorded beside the
numbers."""
import argparse
import json
import os
import random
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import sipp_b200  # noqa: E402
from sipp_b200 import _lib  # noqa: E402


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True, timeout=30)
        name, power = [x.strip() for x in q.stdout.strip().splitlines()[0].split(",")]
        return name, power
    except Exception as e:  # the numbers stay meaningful only with the card beside them: say so
        return "unknown (%s)" % e, "unknown"


def timed(fn, reps):
    fn()  # warm-up: module load, pool blocks, line table
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        ts.append((time.perf_counter() - t0) * 1e3)
    return {"median_ms": statistics.median(ts), "min_ms": min(ts), "reps": reps}


def profiled(fn):
    sipp_b200.set_option(_lib.OPT_PROFILE, 1)
    try:
        sipp_b200.stats(reset=True)
        fn()
        st = sipp_b200.stats(reset=True)
    finally:
        sipp_b200.set_option(_lib.OPT_PROFILE, 0)
    return {"miller_pairs": st["miller_pairs"], "miller_ms": st["miller_ms"], "reduce_fe_ms": st["reduce_fe_ms"],
            "miller_loops_per_s": st["miller_pairs"] / (st["miller_ms"] * 1e-3) if st["miller_ms"] > 0 else None}


def segments(A, B, lengths):
    out, pos = [], 0
    for length in lengths:
        out.append((A[64 * pos:64 * (pos + length)], B[128 * pos:128 * (pos + length)]))
        pos += length
    return out


def check_sample(A, B, lengths, out, seed):
    segs = segments(A, B, lengths)
    idx = sorted(random.Random(seed).sample(range(len(lengths)), min(64, len(lengths))))
    bad = [j for j in idx if out[j] != sipp_b200.inner_product(*segs[j])]
    return {"checked": len(idx), "mismatches": bad}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "product_batch_time.json"))
    ap.add_argument("--reps", type=int, default=5)
    args = ap.parse_args()
    _lib.require_gpu(0)
    name, power = card()
    print("card: %s, power limit %s" % (name, power), flush=True)
    res = {"card": name, "power_limit": power, "workloads": {}}
    rng = random.Random(2026)
    N = 1 << 16

    def report(key, r):
        res["workloads"][key] = r
        print(key, json.dumps(r), flush=True)

    # W1: 4,096 x 128
    lengths = [128] * 4096
    A, B = sipp_b200.seeded_inputs(101, 128 * 4096)
    r = {"pairs": len(A) // 64, "products": len(lengths)}
    r["batch"] = timed(lambda: sipp_b200.inner_product_batch(A, B, lengths), args.reps)
    r["batch"].update(profiled(lambda: sipp_b200.inner_product_batch(A, B, lengths)))
    segs = segments(A, B, lengths)[:256]
    sipp_b200.inner_product(*segs[0])
    t0 = time.perf_counter()
    for a, b in segs:
        sipp_b200.inner_product(a, b)
    loop_ms = (time.perf_counter() - t0) * 1e3
    r["loop_of_inner_product"] = {"timed_calls": 256, "timed_ms": loop_ms, "per_call_ms": loop_ms / 256,
                                  "extrapolated_ms_for_4096": loop_ms * 16, "note": "extrapolated from 256 calls"}
    r["speedup_vs_extrapolated_loop"] = loop_ms * 16 / r["batch"]["median_ms"]
    r["check"] = check_sample(A, B, lengths, sipp_b200.inner_product_batch(A, B, lengths), 1)
    report("W1_4096x128", r)

    # W2: 2^16 pairings
    A, B = sipp_b200.seeded_inputs(102, N)
    r = {"pairs": N, "products": N}
    r["batch"] = timed(lambda: sipp_b200.pairing_batch(A, B), args.reps)
    r["batch"].update(profiled(lambda: sipp_b200.pairing_batch(A, B)))
    sipp_b200.pairing(A[:64], B[:128])
    t0 = time.perf_counter()
    for j in range(256):
        sipp_b200.pairing(A[64 * j:64 * (j + 1)], B[128 * j:128 * (j + 1)])
    loop_ms = (time.perf_counter() - t0) * 1e3
    r["loop_of_pairing"] = {"timed_calls": 256, "timed_ms": loop_ms, "per_call_ms": loop_ms / 256,
                            "extrapolated_ms_for_65536": loop_ms * 256, "note": "extrapolated from 256 calls"}
    r["speedup_vs_extrapolated_loop"] = loop_ms * 256 / r["batch"]["median_ms"]
    r["check"] = check_sample(A, B, [1] * N, sipp_b200.pairing_batch(A, B), 2)
    report("W2_pairing_2p16", r)

    # W3: skewed
    lengths = [N] + [rng.randrange(0, 65) for _ in range(4095)]
    A, B = sipp_b200.seeded_inputs(103, sum(lengths))
    r = {"pairs": sum(lengths), "products": len(lengths), "longest": N}
    r["batch"] = timed(lambda: sipp_b200.inner_product_batch(A, B, lengths), args.reps)
    r["batch"].update(profiled(lambda: sipp_b200.inner_product_batch(A, B, lengths)))
    out = sipp_b200.inner_product_batch(A, B, lengths)
    r["check"] = check_sample(A, B, lengths, out, 3)
    r["check"]["long_segment_equal"] = out[0] == sipp_b200.inner_product(*segments(A, B, lengths)[0])
    report("W3_skewed", r)

    # W4: one 2^16 segment
    A, B = sipp_b200.seeded_inputs(104, N)
    r = {"pairs": N, "products": 1}
    r["batch"] = timed(lambda: sipp_b200.inner_product_batch(A, B, [N]), args.reps)
    r["batch"].update(profiled(lambda: sipp_b200.inner_product_batch(A, B, [N])))
    r["inner_product"] = timed(lambda: sipp_b200.inner_product(A, B), args.reps)
    r["inner_product"].update(profiled(lambda: sipp_b200.inner_product(A, B)))
    r["check"] = {"equal": sipp_b200.inner_product_batch(A, B, [N])[0] == sipp_b200.inner_product(A, B)}
    a, b = r["batch"]["miller_loops_per_s"], r["inner_product"]["miller_loops_per_s"]
    r["miller_rate_batch_over_single"] = a / b if a and b else None
    report("W4_one_2p16", r)

    w1, w3 = res["workloads"]["W1_4096x128"], res["workloads"]["W3_skewed"]
    res["ns_per_pair"] = {k: v["batch"]["median_ms"] * 1e6 / v["pairs"] for k, v in res["workloads"].items()}
    res["W3_over_W1_time_per_pair"] = (w3["batch"]["median_ms"] / w3["pairs"]) / (w1["batch"]["median_ms"] / w1["pairs"])
    ok = all(not v["check"].get("mismatches") and v["check"].get("equal", True) and v["check"].get("long_segment_equal", True)
             for v in res["workloads"].values())
    res["outputs_ok"] = ok
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print("summary: ns/pair %s, W3/W1 per pair %.2f, outputs_ok %s -> %s" % (
        {k: round(v, 1) for k, v in res["ns_per_pair"].items()}, res["W3_over_W1_time_per_pair"], ok, args.out), flush=True)
    return 0 if ok else 1


if __name__ == "__main__":
    sys.exit(main())
