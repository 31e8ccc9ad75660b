"""Batched verification from device memory (sipp_verify_native_batch_device, sipp_verify_native_batch_ragged_device) against the host
forms on the same bytes, in one process.  python tools/verify_device_time.py [--out profiles/verify_device_time.json] [--reps 5]

  B1  4,096 instances of n = 128                                      sipp_verify_native_batch         | _device
  R1  4,096 instances, n cycling through 2^2 .. 2^9, seeded shuffle   sipp_verify_native_batch_ragged  | _device
      (the R1 mix of tools/statement_time.py)
  S1  64 instances of n = 16, where launch latency dominates          sipp_verify_native_batch         | _device

The host arm calls the C ABI on host buffers laid out before the clock starts (it uploads A, B and the proofs and downloads the
outcome); the device arm calls it on torch CUDA buffers already resident, results and finals staying in HBM.  Both calls return when
their outputs are complete.  Warm wall times (a host clock around each call, after one warm-up of each arm), the median of `reps`
passes with the arms alternated inside each pass.  Every workload checks that every instance verifies and that the device arm's
results and finals equal the host arm's byte for byte.  The card's name and power limit are read in the same run."""
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
import torch  # noqa: E402

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


def plen(n):
    return 2 * (n.bit_length() - 1) + 1


def szt(v):
    return (ctypes.c_size_t * len(v))(*v)


def running(v):
    o = [0]
    for x in v:
        o.append(o[-1] + x)
    return o


class Workload:
    """one batch (lengths all equal: the uniform calls) proved on the device, with both arms' buffers laid out"""

    def __init__(self, lengths, seed):
        self.lengths, self.count, self.n = lengths, len(lengths), sum(lengths)
        self.uniform = len(set(lengths)) == 1
        lib = _lib.load()
        self.dA = torch.empty(64 * self.n, dtype=torch.uint8, device="cuda")
        self.dB = torch.empty(128 * self.n, dtype=torch.uint8, device="cuda")
        self.plens = [plen(x) for x in lengths]
        self.dP = torch.zeros(384 * sum(self.plens), dtype=torch.uint8, device="cuda")
        torch.cuda.synchronize()
        _lib.check(lib.sipp_seeded_inputs_device(seed, self.n, self.dA.data_ptr(), self.dB.data_ptr()))
        self.offs, self.poffs = szt(running(lengths)), szt(running(self.plens))
        if self.uniform:
            _lib.check(lib.sipp_prove_native_batch_device(self.dA.data_ptr(), self.dB.data_ptr(), lengths[0], self.count, self.dP.data_ptr()))
        else:
            _lib.check(lib.sipp_prove_native_batch_ragged_device(self.dA.data_ptr(), self.dB.data_ptr(), self.n, self.offs, self.count, self.dP.data_ptr()))
        self.A, self.B, self.P = (t.cpu().numpy().tobytes() for t in (self.dA, self.dB, self.dP))
        self.res = (ctypes.c_int * self.count)()
        self.fa, self.fb, self.fz = (ctypes.create_string_buffer(k * self.count) for k in (64, 128, 384))
        self.dres = torch.zeros(self.count, dtype=torch.int32, device="cuda")
        self.dfins = [torch.zeros(k * self.count, dtype=torch.uint8, device="cuda") for k in (64, 128, 384)]
        torch.cuda.synchronize()

    def host(self):
        lib = _lib.load()
        if self.uniform:
            _lib.check(lib.sipp_verify_native_batch(self.A, self.B, self.lengths[0], self.count, self.P, self.plens[0], self.res, self.fa, self.fb, self.fz))
        else:
            _lib.check(lib.sipp_verify_native_batch_ragged(self.A, self.n, self.B, self.n, self.offs, self.count, self.P, self.poffs, self.res,
                                                            self.fa, self.fb, self.fz))

    def device(self):
        lib = _lib.load()
        f = [t.data_ptr() for t in self.dfins]
        if self.uniform:
            _lib.check(lib.sipp_verify_native_batch_device(self.dA.data_ptr(), self.dB.data_ptr(), self.lengths[0], self.count, self.dP.data_ptr(),
                                                           self.plens[0], self.dres.data_ptr(), *f))
        else:
            _lib.check(lib.sipp_verify_native_batch_ragged_device(self.dA.data_ptr(), self.dB.data_ptr(), self.n, self.offs, self.count, self.dP.data_ptr(),
                                                                  self.poffs, self.dres.data_ptr(), *f))

    def check(self):
        self.host()
        self.device()
        dev = (self.dres.cpu().tolist(), *(t.cpu().numpy().tobytes() for t in self.dfins))
        return {"all_ok": list(self.res) == [0] * self.count, "device_equals_host": dev == (list(self.res), self.fa.raw, self.fb.raw, self.fz.raw)}

    def run(self, reps):
        t = alternated({"host": self.host, "device": self.device}, reps)
        return {"instances": self.count, "pairs": self.n, "input_bytes": len(self.A) + len(self.B) + len(self.P),
                "host_form_ms": t["host"], "device_form_ms": t["device"],
                "saving_ms": t["host"]["median_ms"] - t["device"]["median_ms"],
                "ratio_device_over_host": t["device"]["median_ms"] / t["host"]["median_ms"], **self.check()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "verify_device_time.json"))
    ap.add_argument("--reps", type=int, default=5)
    args = ap.parse_args()
    _lib.require_gpu(0)
    name, power = card()
    res = {"gpu": name, "power_limit": power, "method": __doc__.strip().splitlines()[-6:], "workloads": {}}
    mix = [1 << (2 + (j % 8)) for j in range(4096)]
    random.Random(2).shuffle(mix)
    for key, lengths, seed in (("B1_4096x128", [128] * 4096, 1), ("R1_mixed_2to9", mix, 2), ("S1_64x16", [16] * 64, 3)):
        w = Workload(lengths, seed).run(args.reps)
        res["workloads"][key] = w
        print(key, json.dumps(w), flush=True)
    os.makedirs(os.path.dirname(args.out), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print("wrote", args.out)


if __name__ == "__main__":
    main()
