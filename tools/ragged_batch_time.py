"""Ragged batched proving (sipp_prove_native_batch_ragged) against the ways a caller proves mixed sizes without it, on seeded inputs,
in one process.  python tools/ragged_batch_time.py [--out profiles/ragged_batch_time.json] [--reps 5]

  W1  4,096 instances of n = 128 through the ragged call              vs sipp_prove_native_batch (the uniform call)
  W2  4,096 instances, n cycling through 2^2 .. 2^9 in a seeded shuffle vs one sipp_prove_native_batch call per size (summed)
      (522,240 pairs, about the pairs of W1)                              and vs sipp_prove_native in a loop (64 calls, extrapolated)
  W3  one 2^12 instance plus 4,095 instances of n = 16                   vs one sipp_prove_native_batch call per size (summed)
      (the device absorb chain of the 2^12 instance, 32,768 permutations, bounds the call)

Warm wall times through host buffers (a host clock around calls that end in a device synchronise, after one warm-up of each arm),
the median of `reps` passes with the arms alternated inside each pass.  Every workload checks a seeded sample of 64 instances against
the comparison arm.  The card's name and power limit are read in the same run and recorded beside the numbers."""
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


def alternated(arms, reps):
    """arms: {name: fn}; one warm-up call of each, then `reps` passes calling every arm once, in turn"""
    for fn in arms.values():
        fn()
    ts = {k: [] for k in arms}
    for _ in range(reps):
        for k, fn in arms.items():
            t0 = time.perf_counter()
            fn()
            ts[k].append((time.perf_counter() - t0) * 1e3)
    return {k: {"median_ms": statistics.median(v), "min_ms": min(v), "reps": reps} for k, v in ts.items()}


def split(A, B, lengths):
    out, pos = [], 0
    for n in lengths:
        out.append((A[64 * pos:64 * (pos + n)], B[128 * pos:128 * (pos + n)]))
        pos += n
    return out


def per_size(A, B, lengths):
    """one uniform batched call per distinct size; proofs back in the instances' order"""
    inst = split(A, B, lengths)
    out = [None] * len(lengths)
    for n in sorted(set(lengths)):
        js = [j for j in range(len(lengths)) if lengths[j] == n]
        for j, p in zip(js, sipp_b200.sipp_prove_native_batch(b"".join(inst[j][0] for j in js), b"".join(inst[j][1] for j in js), n)):
            out[j] = p
    return out


def check_sample(got, want, seed):
    idx = sorted(random.Random(seed).sample(range(len(got)), min(64, len(got))))
    return {"checked": len(idx), "mismatches": [j for j in idx if got[j] != want[j]]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "ragged_batch_time.json"))
    ap.add_argument("--reps", type=int, default=5)
    args = ap.parse_args()
    _lib.require_gpu(0)
    name, power = card()
    res = {"gpu": name, "power_limit": power, "method": __doc__.strip().splitlines()[-4:], "workloads": {}}
    prove = sipp_b200.sipp_prove_native_batch_ragged

    # W1
    A, B = sipp_b200.seeded_inputs(1, 128 * 4096)
    lengths = [128] * 4096
    t = alternated({"ragged": lambda: prove(A, B, lengths), "uniform": lambda: sipp_b200.sipp_prove_native_batch(A, B, 128)}, args.reps)
    w = {"instances": 4096, "pairs": 128 * 4096, "ragged_ms": t["ragged"], "uniform_ms": t["uniform"],
         "ratio_ragged_over_uniform": t["ragged"]["median_ms"] / t["uniform"]["median_ms"],
         "sample": check_sample(prove(A, B, lengths), sipp_b200.sipp_prove_native_batch(A, B, 128), 11)}
    res["workloads"]["W1_4096x128"] = w
    print("W1", json.dumps(w), flush=True)

    # W2
    lengths = [1 << (2 + (j % 8)) for j in range(4096)]
    random.Random(2).shuffle(lengths)
    A, B = sipp_b200.seeded_inputs(2, sum(lengths))
    t = alternated({"ragged": lambda: prove(A, B, lengths), "per_size": lambda: per_size(A, B, lengths)}, args.reps)
    inst = split(A, B, lengths)
    loop_idx = random.Random(3).sample(range(len(lengths)), 64)
    sipp_b200.sipp_prove_native(*inst[loop_idx[0]])
    t0 = time.perf_counter()
    for j in loop_idx:
        sipp_b200.sipp_prove_native(*inst[j])
    loop_ms = (time.perf_counter() - t0) * 1e3
    loop_pairs = sum(lengths[j] for j in loop_idx)
    got = prove(A, B, lengths)
    w = {"instances": 4096, "pairs": sum(lengths), "sizes": "2^2 .. 2^9, 512 instances each, seeded shuffle",
         "ragged_ms": t["ragged"], "per_size_calls_summed_ms": t["per_size"],
         "speedup_over_per_size": t["per_size"]["median_ms"] / t["ragged"]["median_ms"],
         "single_loop": {"calls": 64, "ms": loop_ms, "ms_per_call": loop_ms / 64,
                         "extrapolated_ms": loop_ms / 64 * len(lengths), "pairs_of_the_64": loop_pairs},
         "sample": check_sample(got, per_size(A, B, lengths), 12)}
    w["sample_vs_single"] = {"checked": 8, "mismatches": [j for j in loop_idx[:8] if got[j] != sipp_b200.sipp_prove_native(*inst[j])]}
    res["workloads"]["W2_mixed_2to9"] = w
    print("W2", json.dumps(w), flush=True)

    # W3
    lengths = [16] * 2000 + [4096] + [16] * 2095
    A, B = sipp_b200.seeded_inputs(4, sum(lengths))
    t = alternated({"ragged": lambda: prove(A, B, lengths), "per_size": lambda: per_size(A, B, lengths)}, args.reps)
    inst = split(A, B, lengths)
    t0 = time.perf_counter()
    single = sipp_b200.sipp_prove_native(*inst[2000])
    single_ms = (time.perf_counter() - t0) * 1e3
    got = prove(A, B, lengths)
    w = {"instances": 4096, "pairs": sum(lengths), "ragged_ms": t["ragged"], "per_size_calls_summed_ms": t["per_size"],
         "ratio_ragged_over_per_size": t["ragged"]["median_ms"] / t["per_size"]["median_ms"],
         "sipp_prove_native_2p12_ms": single_ms, "absorb_chain_permutations": 8 * 4096,
         "sample": check_sample(got, per_size(A, B, lengths), 13), "big_instance_equal": got[2000] == single}
    res["workloads"]["W3_2p12_plus_4095x16"] = w
    print("W3", json.dumps(w), flush=True)

    os.makedirs(os.path.dirname(args.out), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print("wrote", args.out)


if __name__ == "__main__":
    main()
