"""Proof and statement in one call (sipp_prove_native_statement and its batched and ragged forms) against the way a caller gets the
statement without it: the prover, then the matching verifier.  python tools/statement_time.py [--out profiles/statement_time.json] [--reps 5]

  S1  n = 128                 sipp_prove_native            | + sipp_verify_native               | sipp_prove_native_statement
  S2  n = 2^12                (same arms)
  S3  n = 2^16                (same arms)
  B1  4,096 x n = 128         sipp_prove_native_batch      | + sipp_verify_native_batch         | sipp_prove_native_batch_statement
  R1  the ragged W2 mix       sipp_prove_native_batch_ragged | + sipp_verify_native_batch_ragged | sipp_prove_native_batch_ragged_statement
      (4,096 instances, n cycling through 2^2 .. 2^9, seeded shuffle)

Every arm calls the C ABI with its buffers laid out before the clock starts.  Warm wall times through host buffers (a host clock
around calls that end in a device synchronise, after one warm-up of each arm), the median of `reps` passes with the arms alternated
inside each pass.  The bar: the statement call's time minus the plain prover's is at most 20 % of the verifier's time, taken as the
prove + verify arm minus the plain prover.  Every workload checks that the statement call's proofs equal the plain prover's and that
a seeded sample of its statements equals the verifier arm's.  The card's name and power limit are read in the same run."""
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


def proof_len(n):
    return 2 * (n.bit_length() - 1) + 1


class Work:
    """prepared buffers of one workload: instance j = pairs [offs[j], offs[j + 1]); proofs and finals of each arm"""

    def __init__(self, A, B, lengths):
        self.A, self.B, self.lengths, self.count, self.n = A, B, lengths, len(lengths), sum(lengths)
        offs, po = [0], [0]
        for length in lengths:
            offs.append(offs[-1] + length)
            po.append(po[-1] + proof_len(length))
        self.po = po
        self.offs = (ctypes.c_size_t * len(offs))(*offs)
        self.poffs = (ctypes.c_size_t * len(po))(*po)
        self.proofs, self.sproofs = (ctypes.create_string_buffer(384 * po[-1]) for _ in range(2))
        self.res = (ctypes.c_int * self.count)()
        self.vfin = [ctypes.create_string_buffer(k * self.count) for k in (64, 128, 384)]
        self.sfin = [ctypes.create_string_buffer(k * self.count) for k in (64, 128, 384)]

    def finals(self, fin, j):
        return tuple(f.raw[k * j:k * (j + 1)] for f, k in zip(fin, (64, 128, 384)))


def single_arms(w):
    lib = _lib.load()
    n, np = w.n, proof_len(w.n)

    def plain():
        _lib.check(lib.sipp_prove_native(w.A, n, w.B, n, w.proofs))

    def prove_verify():
        plain()
        _lib.check(lib.sipp_verify_native(w.A, n, w.B, n, w.proofs, np, *w.vfin))

    def statement():
        _lib.check(lib.sipp_prove_native_statement(w.A, n, w.B, n, w.sproofs, *w.sfin))
    return {"plain": plain, "prove_verify": prove_verify, "statement": statement}


def batch_arms(w):
    lib = _lib.load()
    size, count = w.lengths[0], w.count

    def plain():
        _lib.check(lib.sipp_prove_native_batch(w.A, w.B, size, count, w.proofs))

    def prove_verify():
        plain()
        _lib.check(lib.sipp_verify_native_batch(w.A, w.B, size, count, w.proofs, proof_len(size), w.res, *w.vfin))
        assert all(r == _lib.OK for r in w.res)

    def statement():
        _lib.check(lib.sipp_prove_native_batch_statement(w.A, w.B, size, count, w.sproofs, *w.sfin))
    return {"plain": plain, "prove_verify": prove_verify, "statement": statement}


def ragged_arms(w):
    lib = _lib.load()

    def plain():
        _lib.check(lib.sipp_prove_native_batch_ragged(w.A, w.n, w.B, w.n, w.offs, w.count, w.proofs))

    def prove_verify():
        plain()
        _lib.check(lib.sipp_verify_native_batch_ragged(w.A, w.n, w.B, w.n, w.offs, w.count, w.proofs, w.poffs, w.res, *w.vfin))
        assert all(r == _lib.OK for r in w.res)

    def statement():
        _lib.check(lib.sipp_prove_native_batch_ragged_statement(w.A, w.n, w.B, w.n, w.offs, w.count, w.sproofs, *w.sfin))
    return {"plain": plain, "prove_verify": prove_verify, "statement": statement}


def measure(name, w, arms, reps, seed):
    t = alternated(arms, reps)
    plain, pv, st = (t[k]["median_ms"] for k in ("plain", "prove_verify", "statement"))
    verify = pv - plain
    idx = sorted(random.Random(seed).sample(range(w.count), min(64, w.count)))
    out = {"instances": w.count, "pairs": w.n, "plain_ms": t["plain"], "prove_verify_ms": t["prove_verify"], "statement_ms": t["statement"],
           "verify_ms_derived": verify, "statement_minus_plain_ms": st - plain, "overhead_over_verify": (st - plain) / verify,
           "bar_met": st - plain <= 0.2 * verify, "speedup_over_prove_verify": pv / st,
           "proofs_equal": w.proofs.raw == w.sproofs.raw, "sample_checked": len(idx),
           "sample_mismatches": [j for j in idx if w.finals(w.vfin, j) != w.finals(w.sfin, j)]}
    print(name, json.dumps(out), flush=True)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "statement_time.json"))
    ap.add_argument("--reps", type=int, default=5)
    args = ap.parse_args()
    _lib.require_gpu(0)
    name, power = card()
    res = {"gpu": name, "power_limit": power, "method": __doc__.strip().splitlines()[-8:], "workloads": {}}
    for key, n, seed in (("S1_n128", 128, 11), ("S2_n4096", 4096, 12), ("S3_n65536", 1 << 16, 13)):
        A, B = sipp_b200.seeded_inputs(seed, n)
        w = Work(A, B, [n])
        res["workloads"][key] = measure(key, w, single_arms(w), args.reps, seed)
    lengths = [128] * 4096
    A, B = sipp_b200.seeded_inputs(14, sum(lengths))
    w = Work(A, B, lengths)
    res["workloads"]["B1_4096x128"] = measure("B1_4096x128", w, batch_arms(w), args.reps, 14)
    lengths = [1 << (2 + (j % 8)) for j in range(4096)]
    random.Random(2).shuffle(lengths)
    A, B = sipp_b200.seeded_inputs(2, sum(lengths))
    w = Work(A, B, lengths)
    res["workloads"]["R1_mixed_2to9"] = measure("R1_mixed_2to9", w, ragged_arms(w), args.reps, 15)
    res["workloads"]["R1_mixed_2to9"]["sizes"] = "2^2 .. 2^9, 512 instances each, seeded shuffle"
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print("wrote", args.out)


if __name__ == "__main__":
    main()
