"""Ragged batched verification (sipp_verify_native_batch_ragged) against the ways a caller verifies mixed sizes without it, on seeded
inputs proved by sipp_prove_native_batch_ragged, in one process.  python tools/ragged_verify_time.py [--out profiles/ragged_verify_time.json] [--reps 5]

  V1  4,096 instances of n = 128 through the ragged call              vs sipp_verify_native_batch (the uniform call)
  V2  4,096 instances, n cycling through 2^2 .. 2^9 in a seeded shuffle vs one sipp_verify_native_batch call per size (summed)
      (the instances of the ragged prover's W2)                           and vs sipp_verify_native in a loop (64 calls, extrapolated)
  V3  one 2^12 instance plus 4,095 instances of n = 16                   vs one sipp_verify_native_batch call per size (summed)

Every arm calls the C ABI with its buffers laid out before the clock starts (the per-size arm gets its instances already grouped by
size, which favours it).  Warm wall times through host buffers (a host clock around calls that end in a device synchronise, after
one warm-up of each arm), the median of `reps` passes with the arms alternated inside each pass.  Every workload checks that every
instance verifies and that the finals of a seeded sample of 64 instances equal the comparison arm's.  The card's name and power
limit are read in the same run and recorded beside the numbers."""
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


class Ragged:
    """one sipp_verify_native_batch_ragged call over prepared buffers; results and finals per instance afterwards"""

    def __init__(self, A, B, lengths, proofs):
        self.count, self.n = len(lengths), sum(lengths)
        offs, po = [0], [0]
        for length, p in zip(lengths, proofs):
            offs.append(offs[-1] + length)
            po.append(po[-1] + len(p))
        self.A, self.B, self.P = A, B, b"".join(b"".join(p) for p in proofs)
        self.offs = (ctypes.c_size_t * len(offs))(*offs)
        self.po = (ctypes.c_size_t * len(po))(*po)
        self.res = (ctypes.c_int * self.count)()
        self.fa, self.fb, self.fz = (ctypes.create_string_buffer(k * self.count) for k in (64, 128, 384))

    def __call__(self):
        _lib.check(_lib.load().sipp_verify_native_batch_ragged(self.A, self.n, self.B, self.n, self.offs, self.count, self.P, self.po, self.res,
                                                                self.fa, self.fb, self.fz))

    def result(self, j):
        return self.res[j], (self.fa.raw[64 * j:64 * j + 64], self.fb.raw[128 * j:128 * j + 128], self.fz.raw[384 * j:384 * j + 384])


class Uniform(Ragged):
    """one sipp_verify_native_batch call over prepared buffers"""

    def __init__(self, A, B, n, proofs):
        super().__init__(A, B, [n] * len(proofs), proofs)
        self.size, self.plen = n, len(proofs[0])

    def __call__(self):
        _lib.check(_lib.load().sipp_verify_native_batch(self.A, self.B, self.size, self.count, self.P, self.plen, self.res, self.fa, self.fb, self.fz))


class PerSize:
    """one Uniform call per distinct size, the instances grouped by size beforehand"""

    def __init__(self, A, B, lengths, proofs):
        inst = split(A, B, lengths)
        self.calls, self.where = [], {}
        for n in sorted(set(lengths)):
            js = [j for j in range(len(lengths)) if lengths[j] == n]
            for k, j in enumerate(js):
                self.where[j] = (len(self.calls), k)
            self.calls.append(Uniform(b"".join(inst[j][0] for j in js), b"".join(inst[j][1] for j in js), n, [proofs[j] for j in js]))

    def __call__(self):
        for c in self.calls:
            c()

    def result(self, j):
        c, k = self.where[j]
        return self.calls[c].result(k)


def check(ragged, other, count, seed):
    ragged()
    other()
    idx = sorted(random.Random(seed).sample(range(count), min(64, count)))
    return {"all_ok": all(ragged.result(j)[0] == _lib.OK for j in range(count)), "checked": len(idx),
            "mismatches": [j for j in idx if ragged.result(j) != other.result(j)]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "ragged_verify_time.json"))
    ap.add_argument("--reps", type=int, default=5)
    args = ap.parse_args()
    _lib.require_gpu(0)
    name, power = card()
    res = {"gpu": name, "power_limit": power, "method": __doc__.strip().splitlines()[-6:], "workloads": {}}
    prove = sipp_b200.sipp_prove_native_batch_ragged

    # V1
    lengths = [128] * 4096
    A, B = sipp_b200.seeded_inputs(1, sum(lengths))
    proofs = prove(A, B, lengths)
    rg, un = Ragged(A, B, lengths, proofs), Uniform(A, B, 128, proofs)
    t = alternated({"ragged": rg, "uniform": un}, args.reps)
    w = {"instances": 4096, "pairs": sum(lengths), "ragged_ms": t["ragged"], "uniform_ms": t["uniform"],
         "ratio_ragged_over_uniform": t["ragged"]["median_ms"] / t["uniform"]["median_ms"], "sample": check(rg, un, len(lengths), 21)}
    res["workloads"]["V1_4096x128"] = w
    print("V1", json.dumps(w), flush=True)

    # V2
    lengths = [1 << (2 + (j % 8)) for j in range(4096)]
    random.Random(2).shuffle(lengths)
    A, B = sipp_b200.seeded_inputs(2, sum(lengths))
    proofs = prove(A, B, lengths)
    rg, ps = Ragged(A, B, lengths, proofs), PerSize(A, B, lengths, proofs)
    t = alternated({"ragged": rg, "per_size": ps}, args.reps)
    inst = split(A, B, lengths)
    loop_idx = random.Random(3).sample(range(len(lengths)), 64)
    sipp_b200.sipp_verify_native(*inst[loop_idx[0]], proofs[loop_idx[0]])
    t0 = time.perf_counter()
    for j in loop_idx:
        sipp_b200.sipp_verify_native(*inst[j], proofs[j])
    loop_ms = (time.perf_counter() - t0) * 1e3
    w = {"instances": 4096, "pairs": sum(lengths), "sizes": "2^2 .. 2^9, 512 instances each, seeded shuffle",
         "ragged_ms": t["ragged"], "per_size_calls_summed_ms": t["per_size"],
         "speedup_over_per_size": t["per_size"]["median_ms"] / t["ragged"]["median_ms"],
         "single_loop": {"calls": 64, "ms": loop_ms, "ms_per_call": loop_ms / 64, "extrapolated_ms": loop_ms / 64 * len(lengths),
                         "pairs_of_the_64": sum(lengths[j] for j in loop_idx)},
         "speedup_over_single_loop": loop_ms / 64 * len(lengths) / t["ragged"]["median_ms"],
         "sample": check(rg, ps, len(lengths), 22)}
    singles = [sipp_b200.sipp_verify_native(*inst[j], proofs[j]) for j in loop_idx[:8]]
    w["sample_vs_single"] = {"checked": 8, "mismatches": [j for j, st in zip(loop_idx[:8], singles)
                                                          if rg.result(j) != (_lib.OK, (st.final_A, st.final_B, st.final_Z))]}
    res["workloads"]["V2_mixed_2to9"] = w
    print("V2", json.dumps(w), flush=True)

    # V3
    lengths = [16] * 2000 + [4096] + [16] * 2095
    A, B = sipp_b200.seeded_inputs(4, sum(lengths))
    proofs = prove(A, B, lengths)
    rg, ps = Ragged(A, B, lengths, proofs), PerSize(A, B, lengths, proofs)
    t = alternated({"ragged": rg, "per_size": ps}, args.reps)
    inst = split(A, B, lengths)
    t0 = time.perf_counter()
    single = sipp_b200.sipp_verify_native(*inst[2000], proofs[2000])
    single_ms = (time.perf_counter() - t0) * 1e3
    w = {"instances": 4096, "pairs": sum(lengths), "ragged_ms": t["ragged"], "per_size_calls_summed_ms": t["per_size"],
         "ratio_ragged_over_per_size": t["ragged"]["median_ms"] / t["per_size"]["median_ms"],
         "sipp_verify_native_2p12_ms": single_ms, "absorb_chain_permutations": 8 * 4096, "sample": check(rg, ps, len(lengths), 23),
         "big_instance_equal": rg.result(2000) == (_lib.OK, (single.final_A, single.final_B, single.final_Z))}
    res["workloads"]["V3_2p12_plus_4095x16"] = w
    print("V3", json.dumps(w), flush=True)

    os.makedirs(os.path.dirname(args.out), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print("wrote", args.out)


if __name__ == "__main__":
    main()
